"""U-Net discriminator (SURVEY 8f rank 2): drop-in DiscriminatorUNet (BSRGAN/model.py:91-167 = Real_ESRGAN/model.py:29-105).

CPU: the oracle restatement (oracle/disc_oracle.py) is pinned against the reference class (bit-equal: logits, power-iteration
buffers, every parameter gradient, input gradient) and against the committed golden fixture; the drop-in's own CPU path and its
construction (state_dict keys, shapes, seeded initial values) equal the reference class bit for bit.
GPU: the native path (tcgen05 convs in bf16 with fp32 accumulation) against the fp32 oracle on the CPU.  BASELINE.json states no
tolerance for the discriminator.  The bar: per tensor, not further from fp32 than 1.3 x what torch's own autocast of the same
module IN THE SAME 16-BIT FORMAT loses (+ 2e-3) -- fp16, the format the reference scripts run it in and the native default, or
bf16 -- inside absolute caps of 5e-3 / 0.1 (fp16: logits / gradients) and 2e-2 / 0.2 (bf16) relative L2; measured values are
appended to gpurun_out/disc_parity.jsonl and the worst tensor is printed."""
import copy
import glob
import io
import os
import pickle

import pytest
import torch

from oracle import disc_oracle as do
from oracle import make_golden
from oracle import reference_loader as rl

GOLDEN = sorted(glob.glob(os.path.join(os.path.dirname(__file__), "golden", "disc", "*.pt")))


@pytest.fixture
def golden_threads():
    """the thread count the fixture was computed with (bit equality depends on it), whatever the host or an earlier test set"""
    n = torch.get_num_threads()
    torch.set_num_threads(make_golden.THREADS)
    yield
    torch.set_num_threads(n)


def rel_l2(a, b):
    a, b = a.double().flatten().cpu(), b.double().flatten().cpu()
    return float((a - b).norm() / b.norm().clamp_min(1e-30))


def _drop_in(seed=0, **kw):
    from sr_gan_fd_b200.discriminator import DiscriminatorUNet
    torch.manual_seed(seed)
    args = dict(in_channels=3, out_channels=1, channels=64)
    args.update(kw)
    return DiscriminatorUNet(**args)


def _inputs(n, h, w, seed=1):
    g = torch.Generator().manual_seed(seed)
    return torch.rand(n, 3, h, w, generator=g), torch.randn(n, 1, h, w, generator=g)


# ------------------------------------------------------------------------------------------------------------ CPU
@pytest.mark.skipif(not rl.available(), reason="reference tree not present (GPU box)")
@pytest.mark.parametrize("flavour", ["bsrgan", "real"])
def test_disc_oracle_bit_equal_to_reference(flavour):
    m = rl.load_module(flavour)
    torch.manual_seed(0)
    ref = m.DiscriminatorUNet(3, 1, 64)
    assert [n for n, _ in ref.named_parameters()] == do.param_names()
    assert [tuple(p.shape) for n, p in ref.named_parameters() if n.endswith(("weight", "weight_orig"))] == \
           [(o, i, k, k) for o, i, k in do.layer_shapes()]
    state = {k: v.clone() for k, v in ref.state_dict().items()}
    x, dy = _inputs(2, 32, 24)
    for training in (True, False):
        ref.load_state_dict(state)
        ref.train(training)
        ref.zero_grad(set_to_none=True)
        xr = x.clone().requires_grad_(True)
        y = ref(xr)
        y.backward(dy)
        yo, grads, _, dx, buffers = do.forward_backward(state, x, dy, training, input_grad=True)
        assert torch.equal(y, yo)
        assert torch.equal(dx, xr.grad)
        for n, p in ref.named_parameters():
            assert torch.equal(grads[n], p.grad), n
        after = ref.state_dict()
        for k, v in buffers.items():
            assert torch.equal(v, after[k]), k


@pytest.mark.skipif(not rl.available(), reason="reference tree not present (GPU box)")
def test_drop_in_equals_reference_class_on_cpu():
    m = rl.load_module("bsrgan")
    torch.manual_seed(0)
    ref = m.discriminator_unet(in_channels=3, out_channels=1, channels=64)
    mine = _drop_in(0)
    sa, sb = mine.state_dict(), ref.state_dict()
    assert list(sa.keys()) == list(sb.keys())
    assert all(torch.equal(sa[k], sb[k]) for k in sa)
    assert [n for n, _ in mine.named_parameters()] == [n for n, _ in ref.named_parameters()]
    x, dy = _inputs(2, 24, 40)
    ya, yb = mine(x), ref(x)
    assert torch.equal(ya, yb)
    ya.backward(dy)
    yb.backward(dy)
    for (n, p), (_, q) in zip(mine.named_parameters(), ref.named_parameters()):
        assert torch.equal(p.grad, q.grad), n
    assert all(torch.equal(v, ref.state_dict()[k]) for k, v in mine.state_dict().items())  # power-iteration buffers moved alike


def test_drop_in_cpu_path_equals_oracle_and_module_protocol():
    mine = _drop_in(3)
    assert [n for n, _ in mine.named_parameters()] == do.param_names()
    state = {k: v.clone() for k, v in mine.state_dict().items()}
    x, dy = _inputs(1, 16, 16)
    # deepcopy keeps the parameters and drops the native runtime (before the first forward: torch's spectral_norm hook leaves a
    # non-leaf `weight` on the convs afterwards, which no module -- the reference's included -- can deepcopy)
    mine._runtime()
    twin = copy.deepcopy(mine)
    assert "_b200_disc" not in twin.__dict__
    assert all(torch.equal(a, b) for a, b in zip(twin.state_dict().values(), mine.state_dict().values()))
    y = mine(x)
    yo, buffers = do.forward(state, x, training=True)
    assert torch.equal(y, yo)
    for k, v in buffers.items():
        assert torch.equal(mine.state_dict()[k], v)
    # pickle / torch.save round trips
    with torch.no_grad():
        mine(x)  # leaves detached effective weights on the convs
    blob = pickle.dumps(mine)
    again = pickle.loads(blob)
    assert "_b200_disc" not in again.__dict__
    buf = io.BytesIO()
    torch.save(mine.state_dict(), buf)
    buf.seek(0)
    again.load_state_dict(torch.load(buf))
    mine.eval(); again.eval()
    assert torch.equal(mine(x), again(x))


def test_disc_plan_host_bookkeeping():
    import ctypes as C
    from sr_gan_fd_b200 import lib as b200lib
    from sr_gan_fd_b200.build import build_native
    build_native()
    L = b200lib.load()
    h = C.c_void_p()
    d = b200lib.DiscDesc(3, 1, 64, 16, 256, 256, 1, 1)
    assert L.b200sr_disc_plan_create(C.byref(d), C.byref(h)) == 0
    try:
        shapes = do.layer_shapes()
        numel = sum(o * i * k * k for o, i, k in shapes) + 64 + 1
        assert L.b200sr_num_params(h) == 20
        assert L.b200sr_param_numel(h) == numel
        px = [16 * (256 >> l) * (256 >> l) for l in (0, 1, 2, 3, 2, 1, 0, 0, 0, 0)]
        fl = sum(2.0 * k * k * o * i * p for (o, i, k), p in zip(shapes, px))
        assert L.b200sr_flops(h, 0) == fl
        assert L.b200sr_flops(h, 2) == fl
        assert L.b200sr_workspace_bytes(h) > 0 and L.b200sr_packed_bytes(h) > 2 * numel
    finally:
        L.b200sr_plan_destroy(h)
    for bad in (b200lib.DiscDesc(3, 1, 32, 1, 64, 64, 0, 0), b200lib.DiscDesc(3, 1, 64, 1, 60, 64, 0, 0), b200lib.DiscDesc(17, 1, 64, 1, 64, 64, 0, 0)):
        assert L.b200sr_disc_plan_create(C.byref(bad), C.byref(h)) < 0 and L.b200sr_last_error()


@pytest.mark.usefixtures("golden_threads")
@pytest.mark.parametrize("path", GOLDEN, ids=[os.path.basename(p) for p in GOLDEN])
def test_disc_oracle_matches_golden(path):
    """seed + drop-in constructor reproduces the reference's parameters; the oracle reproduces the reference's logits and gradients"""
    fix = torch.load(path)
    mine = _drop_in(fix["seed"])
    state = {k: v.clone() for k, v in mine.state_dict().items()}
    assert abs(float(sum(v.double().sum() for v in state.values())) - fix["param_checksum"]) < 1e-9
    y, grads, _, dx, buffers = do.forward_backward(state, fix["x"], fix["dy"], training=True, input_grad=True)
    assert torch.equal(y, fix["y"])
    assert torch.allclose(dx, fix["dx"], rtol=1e-5, atol=1e-9)
    for k, g in fix["grads"].items():
        assert torch.allclose(grads[k], g, rtol=1e-5, atol=1e-9), k
    for k, nrm in fix["grad_norms"].items():
        assert abs(float(grads[k].double().norm()) - nrm) <= 1e-5 * max(nrm, 1e-12), k
    for k, v in fix["buffers"].items():
        assert torch.equal(buffers[k], v), k


# ------------------------------------------------------------------------------------------------------------ GPU
EFF_NAMES = [name for name, *_ in do.LAYERS]


def _gpu_step(mine, x, dy, input_grad):
    """forward + backward on the GPU module; returns logits, parameter grads, effective-weight grads, dx"""
    mine.zero_grad(set_to_none=True)
    xg = x.cuda().requires_grad_(input_grad)
    eff = {}
    # capture the gradients of the effective weights: the spectral-norm hook leaves them on the conv modules as non-leaf tensors
    y = mine(xg)
    for name, _, _, sn, _ in do.LAYERS:
        if sn:
            conv = mine.get_submodule(name)
            conv.weight.retain_grad()
            eff[name] = conv.weight
    y.backward(dy.cuda())
    grads = {n: p.grad.detach().cpu() for n, p in mine.named_parameters() if p.grad is not None}
    effg = {k: (v.grad.detach().cpu() if v.grad is not None else None) for k, v in eff.items()}
    return y.detach().cpu(), grads, effg, (xg.grad.detach().cpu() if input_grad else None)


def _autocast_errors(state, x, dy, training, go, yo, dxo, dtype=torch.bfloat16):
    """what stock torch autocast of the SAME module (CPU path = the reference's op sequence) loses against fp32"""
    ref = _drop_in(0)
    ref.load_state_dict(state)
    ref.train(training)
    xr = x.clone().requires_grad_(True)
    with torch.autocast("cpu", dtype=dtype):
        y = ref(xr)
    y.float().backward(dy)
    errs = {"logits": rel_l2(y.float(), yo), "dx": rel_l2(xr.grad, dxo)}
    for n, p in ref.named_parameters():
        errs["grad " + n] = rel_l2(p.grad, go[n])
    return errs


def _settle_power_iteration(module, x, iters=5):
    """eval-mode forwards use the stored weight_u / weight_v as they are: a freshly constructed module holds RANDOM vectors, whose
    sigma = u.(W v) is far from the spectral norm (weights blow up by orders of magnitude and overflow fp16 -- in the reference's
    autocast just the same).  A few training-mode forwards give the buffers the values a trained discriminator has."""
    module.train()
    with torch.no_grad():
        for _ in range(iters):
            module(x)
    return module


def _record(tag, payload, fname="disc_parity.jsonl"):
    out = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "gpurun_out")
    if os.path.isdir(out):
        import json
        with open(os.path.join(out, fname), "a") as fh:
            fh.write(json.dumps({"case": tag, **payload}) + "\n")


CAPS = {"fp16": (5e-3, 0.1), "bf16": (2e-2, 0.2)}  # absolute caps on the relative L2 error: (logits, gradients)


@pytest.mark.gpu
@pytest.mark.parametrize("shape,training,fmt", [((2, 64, 64), True, "fp16"), ((3, 40, 72), True, "fp16"), ((1, 32, 32), False, "fp16"),
                                                ((2, 128, 96), True, "fp16"), ((2, 64, 64), True, "bf16"), ((1, 32, 32), False, "bf16")])
def test_gpu_forward_backward_against_oracle(shape, training, fmt):
    """Native path vs the fp32 oracle, next to what torch's own autocast of the same module IN THE SAME 16-BIT FORMAT loses against
    fp32 (fp16 = the format the reference scripts run the discriminator in, and the native default; bf16 = the optional wide-range
    format): per tensor the native path (16-bit operands, fp32 accumulation) must not be further from fp32 than 1.3 x the stock
    autocast path + 2e-3, and inside the absolute caps -- fp16: logits <= 5e-3, gradients <= 0.1; bf16: 2e-2 / 0.2 relative L2.
    (A plain ten-layer feed-forward net has no fp32 residual carrier to lean on, unlike the generator: the rounding of every
    activation shows in the logits, and LeakyReLU-derivative flips near zero show in the gradients.)"""
    n, h, w = shape
    mine = _drop_in(0)
    mine.operand_dtype = fmt
    x, dy = _inputs(n, h, w)
    if not training:
        _settle_power_iteration(mine, x)
    state = {k: v.clone() for k, v in mine.state_dict().items()}
    yo, go, effo, dxo, buffers = do.forward_backward(state, x, dy, training, input_grad=True)
    stock = _autocast_errors(state, x, dy, training, go, yo, dxo, torch.float16 if fmt == "fp16" else torch.bfloat16)
    mine = mine.cuda().train(training)
    y, grads, effg, dx = _gpu_step(mine, x, dy, True)
    errs = {"logits": rel_l2(y, yo), "dx": rel_l2(dx, dxo)}
    for k in do.param_names():
        errs["grad " + k] = rel_l2(grads[k], go[k])
    worst = max(errs, key=errs.get)
    print(f"disc {shape} training={training} {fmt}: logits {errs['logits']:.2e} (stock {fmt} autocast {stock['logits']:.2e}) dx {errs['dx']:.2e} "
          f"({stock['dx']:.2e}) worst {worst} {errs[worst]:.2e} ({stock[worst]:.2e})")
    _record(f"{shape} training={training} {fmt}", {"native_vs_fp32": errs, f"torch_{fmt}_autocast_vs_fp32": stock})
    cap_logits, cap_grad = CAPS[fmt]
    assert errs["logits"] <= cap_logits, errs
    for k, e in errs.items():
        assert e <= cap_grad, (k, e)
        assert e <= 1.3 * stock[k] + 2e-3, (k, e, stock[k])
    # gradients of the EFFECTIVE weights (what the library itself returns, before torch's W / sigma graph)
    for name, g in effg.items():
        assert g is not None and rel_l2(g, effo[name]) <= cap_grad, name
    # the power-iteration buffers moved exactly as the reference moves them (torch's own hook ran once)
    after = mine.state_dict()
    for k, v in buffers.items():
        assert torch.allclose(after[k].cpu(), v, rtol=1e-4, atol=1e-6), k


@pytest.mark.gpu
def test_gpu_frozen_discriminator_gives_input_gradient_only():
    """generator update (BSRGAN/train_bsrgan.py:441-463): requires_grad=False on every discriminator parameter"""
    mine = _drop_in(0)
    state = {k: v.clone() for k, v in mine.state_dict().items()}
    x, dy = _inputs(2, 64, 64, seed=5)
    _, _, _, dxo, _ = do.forward_backward(state, x, dy, True, input_grad=True)
    mine = mine.cuda().train()
    for p in mine.parameters():
        p.requires_grad = False
    xg = x.cuda().requires_grad_(True)
    y = mine(xg)
    y.backward(dy.cuda())
    assert all(p.grad is None for p in mine.parameters())
    assert rel_l2(xg.grad, dxo) <= 0.1
    # and the discriminator update: input without gradient, parameter gradients only; fp16 autocast + GradScaler scale as the script
    for p in mine.parameters():
        p.requires_grad = True
    mine.load_state_dict(state)
    # (upstream gradient of a mean-reduced loss, as BCEWithLogitsLoss gives it, times the GradScaler's initial scale; an O(1)
    # gradient per logit times 65536 overflows fp16 inside torch's own sigma graph under autocast -- in the reference just the same)
    dys = dy / dy.numel()
    _, go, _, _, _ = do.forward_backward(state, x, dys * 65536.0, True)
    with torch.autocast("cuda", dtype=torch.float16):
        y = mine(x.cuda())
    assert y.dtype == torch.float32
    (y * dys.cuda()).sum().mul(65536.0).backward()
    for n, p in mine.named_parameters():
        assert rel_l2(p.grad, go[n]) <= 0.1, n


@pytest.mark.gpu
def test_gpu_other_channel_counts():
    """in_channels = 1 (generic ingest path), out_channels = 2 (two logit maps)"""
    mine = _drop_in(4, in_channels=1, out_channels=2)
    state = {k: v.clone() for k, v in mine.state_dict().items()}
    g = torch.Generator().manual_seed(11)
    x, dy = torch.rand(2, 1, 48, 40, generator=g), torch.randn(2, 2, 48, 40, generator=g)
    st = {k: v.clone().float() for k, v in state.items()}
    leaves = {k: st[k].requires_grad_(True) for k in do.param_names()}
    st.update(leaves)
    xin = x.clone().requires_grad_(True)
    weights, _ = do.effective_weights(st, True)
    yo = do.forward_from_weights(weights, st, xin)
    yo.backward(dy)
    mine = mine.cuda().train()
    xg = x.cuda().requires_grad_(True)
    y = mine(xg)
    y.backward(dy.cuda())
    assert y.shape == (2, 2, 48, 40)
    assert rel_l2(y, yo.detach()) <= 2e-2
    assert rel_l2(xg.grad, xin.grad) <= 0.2
    for n, p in mine.named_parameters():
        assert rel_l2(p.grad, leaves[n].grad) <= 0.2, n


@pytest.mark.gpu
def test_gpu_eval_no_grad_and_determinism():
    x, _ = _inputs(2, 48, 56, seed=9)
    mine = _settle_power_iteration(_drop_in(2), x).cuda().eval()
    with torch.no_grad():
        a = mine(x.cuda())
        b = mine(x.cuda())
    assert not a.requires_grad and torch.equal(a, b)
    state = {k: v.cpu() for k, v in mine.state_dict().items()}
    yo, _ = do.forward(state, x, training=False)
    assert rel_l2(a, yo) <= 5e-3


@pytest.mark.gpu
@pytest.mark.parametrize("path", GOLDEN, ids=[os.path.basename(p) for p in GOLDEN])
def test_gpu_matches_golden(path):
    """the fixture was produced by the reference class itself (oracle/make_golden.py)"""
    fix = torch.load(path)
    mine = _drop_in(fix["seed"]).cuda().train()
    y, grads, _, dx = _gpu_step(mine, fix["x"], fix["dy"], True)
    assert rel_l2(y, fix["y"]) <= 5e-3
    assert rel_l2(dx, fix["dx"]) <= 0.1
    for k, g in fix["grads"].items():
        assert rel_l2(grads[k], g) <= 0.1, k
    for k, nrm in fix["grad_norms"].items():
        assert abs(float(grads[k].double().norm()) - nrm) <= 0.05 * nrm, k


@pytest.mark.gpu
def test_gpu_guard_bands_and_forward_determinism():
    """compute-sanitizer is closed on the GPU pool (profiles/r2_sanitizer_unavailable.log): the discriminator runs through the C ABI
    on workspace / packed / output / gradient / input-gradient buffers framed by guard bands that must come back untouched, and the
    forward pass (no atomics on its path) must be bit-identical over repeated runs on fresh memory."""
    import ctypes as C
    from sr_gan_fd_b200 import lib as _lib
    from sr_gan_fd_b200.discriminator import _DiscPlan
    L = _lib.load()
    dev = torch.device("cuda", 0)
    mine = _drop_in(0).to(dev).train()
    weights = [mine.conv1.weight, mine.conv1.bias] + [mine._effective_weight(c).detach() for c in mine._sn_convs()] + [mine.conv4.weight, mine.conv4.bias]
    w1, b1, d1, d2, d3, u1, u2, u3, c2, c3, w4, b4 = [t.detach().float().contiguous() for t in weights]
    slots = [w1, b1, d1, None, d2, None, d3, None, u1, None, u2, None, u3, None, c2, None, c3, None, w4, b4]
    G = 1 << 16
    for shape, fp16 in [((2, 3, 40, 24), True), ((3, 3, 16, 72), False)]:
        n, c, h, w = shape
        plan = _DiscPlan(3, 1, 64, n, h, w, True, fp16)
        stream = torch.cuda.current_stream().cuda_stream
        x = torch.rand(*shape, device=dev)
        dy = torch.randn(n, 1, h, w, device=dev)
        outs = []
        for rep in range(3):
            def framed(nbytes, fill):
                buf = torch.full((nbytes + 2 * G,), fill, dtype=torch.uint8, device=dev)
                return buf, buf[G:G + nbytes]
            ws_all, ws = framed((plan.workspace_bytes + 1023) // 1024 * 1024, 0xA5)
            pk_all, pk = framed((plan.packed_bytes + 1023) // 1024 * 1024, 0x77)
            y_all, yb = framed(n * h * w * 4, 0x5A)
            g_all, gb = framed(plan.param_numel * 4, 0x3C)
            dx_all, dxb = framed(n * 3 * h * w * 4, 0x69)
            ptrs = (C.c_void_p * 20)(*[t.data_ptr() if t is not None else None for t in slots])
            _lib.check(L.b200sr_pack_weights(plan.handle, ptrs, C.c_void_p(pk.data_ptr()), C.c_void_p(stream)))
            strides = (C.c_int64 * 4)(*x.stride())
            _lib.check(L.b200sr_disc_forward(plan.handle, C.c_void_p(x.data_ptr()), _lib.F32, strides, C.c_void_p(pk.data_ptr()),
                                             C.c_void_p(ws.data_ptr()), C.c_void_p(yb.data_ptr()), C.c_void_p(stream)))
            _lib.check(L.b200sr_disc_backward(plan.handle, C.c_void_p(dy.data_ptr()), C.c_void_p(pk.data_ptr()), C.c_void_p(ws.data_ptr()),
                                              C.c_void_p(gb.data_ptr()), C.c_void_p(dxb.data_ptr()), C.c_void_p(stream)))
            torch.cuda.synchronize()
            for name, full, fill in (("workspace", ws_all, 0xA5), ("packed", pk_all, 0x77), ("output", y_all, 0x5A), ("gradients", g_all, 0x3C),
                                     ("input gradient", dx_all, 0x69)):
                assert bool((full[:G] == fill).all()) and bool((full[-G:] == fill).all()), f"{name} guard band was written ({shape})"
            outs.append((yb.view(torch.float32).clone(), gb.view(torch.float32).clone(), dxb.view(torch.float32).clone()))
        for yb, gb, dxb in outs[1:]:
            assert torch.equal(yb, outs[0][0]), "forward is not bit-reproducible"
            assert torch.isfinite(gb).all() and torch.isfinite(dxb).all()
            assert rel_l2(gb, outs[0][1]) < 1e-5  # fp32 atomics in the weight-gradient flush: order-dependent rounding only
            assert torch.equal(dxb, outs[0][2])   # the data-gradient path has no atomics
