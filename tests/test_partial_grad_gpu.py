"""GPU: the generator backward with frozen and partially frozen parameters (b200sr_backward_select behind autograd).
Every case runs the FULL backward of the same module on the same seeded input in the same process as its reference: frozen
tensors get None, the input gradient is bit-identical (the data-gradient chain is deterministic), wanted parameter gradients
match to rel-L2 1e-6 (only the order of the red.global.add partial sums differs)."""
import copy

import pytest
import torch
import torch.nn.functional as F
from torch.optim.swa_utils import AveragedModel

from oracle import rrdbnet_oracle as orc
from test_partial_grad_host import flags

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda", 0)
TOL_SAME = 1e-6
TOL_GRAD = 1e-2  # the oracle bar of test_model_gpu.py


def _net(factory, nb, seed=0):
    import sr_gan_fd_b200 as b200
    torch.manual_seed(seed)
    net = getattr(b200, factory)(num_blocks=nb)
    params = orc.in_range_fixture({k: v.detach().clone() for k, v in net.state_dict().items()})
    net.load_state_dict(params)
    return net.to(DEV).train(), params


def _inputs(net, shape, seed=1):
    g = torch.Generator().manual_seed(seed)
    lr = torch.rand(*shape, generator=g)
    s = net.upscale_factor
    gt = torch.rand(shape[0], 3, shape[2] * s, shape[3] * s, generator=g)
    return lr, gt


def _poison_backward_buffers(net, y):
    """Fill every workspace tensor that only the backward writes (the output-gradient buffers of the dense blocks, the fp32
    gradient carriers, the tail's gradients) with a finite non-gradient pattern, between the forward and its backward.  A
    backward that stops its data-gradient walk too early, or skips a chain it needs, then reads this pattern instead of what
    an earlier backward left in the same (recycled) memory -- which for the same input would be the correct values."""
    import ctypes as C
    from sr_gan_fd_b200 import lib as _lib
    ws = y.grad_fn.workspace  # the autograd node of the native forward holds its workspace
    plan = net._runtime().last_plan
    names = ["GR", "GC1", "GC2", "GT", "GTB", "GO1", "G3"] + [f"GU{l}" for l in range(1, net._n_up + 1)] + \
            [f"DYB{r}" for r in range(3 * len(net.trunk))]
    for n in names:
        off, nbytes = C.c_int64(), C.c_int64()
        _lib.check(_lib.load().b200sr_debug_buffer(plan.handle, n.encode(), C.byref(off), C.byref(nbytes)))
        ws[off.value:off.value + nbytes.value].fill_(0x3F)  # bf16 0x3F3F / fp32 0x3F3F3F3F: about 0.75 everywhere


def _backward(net, lr, gt, x_grad):
    x = lr.to(DEV).requires_grad_(x_grad)
    y = net(x)
    _poison_backward_buffers(net, y)
    F.l1_loss(y, gt.to(DEV)).backward()
    torch.cuda.synchronize()
    grads = [p.grad.detach().clone() if p.grad is not None else None for p in net.parameters()]
    net.zero_grad(set_to_none=True)
    return grads, (x.grad.detach().clone() if x_grad else None)


def _set_pattern(net, pattern):
    for p, t in zip(net.parameters(), flags(net, pattern)):
        p.requires_grad_(t)


def _check_pattern(net, lr, gt, pattern, x_grad, exact=False):
    # both backwards start from poisoned backward buffers (_backward): the full one shows the pattern is harmless to a backward
    # that writes before it reads, the partial one that it wrote everything it read.  exact: the gradients must be equal bit for
    # bit (deterministic mode, where no atomic reorders a sum)
    _set_pattern(net, "all")
    full, full_dx = _backward(net, lr, gt, x_grad)
    _set_pattern(net, pattern)
    part, dx = _backward(net, lr, gt, x_grad)
    for (name, p), t, gf, gp in zip(net.named_parameters(), flags(net, pattern), full, part):
        if not t:
            assert gp is None, f"{pattern}: {name} is frozen but got a gradient"
            continue
        assert gp is not None, f"{pattern}: {name} is trainable but got no gradient"
        if exact:
            assert torch.equal(gp.view(torch.int32), gf.view(torch.int32)), f"{pattern}: {name} differs from the full deterministic backward"
            continue
        err = orc.rel_l2(gp.cpu(), gf.cpu())
        assert err <= TOL_SAME, f"{pattern}: {name} rel-L2 {err:.3e} against the full backward"
    if x_grad:
        assert torch.equal(dx, full_dx), f"{pattern}: dL/dx differs from the full backward's"
    return part, dx


PATTERNS = [("frozen", True), ("tail", False), ("conv4", False), ("head+half", False), ("one_conv", False),
            ("no_bias", False), ("head+half", True)]
_IDS = ["a_frozen_dx", "b_tail", "c_conv4", "d_head_half", "e_one_conv", "f_no_bias", "g_head_half_dx"]


@pytest.mark.parametrize("pattern,x_grad", PATTERNS, ids=_IDS)
def test_patterns_two_groups(pattern, x_grad):
    """2-RRDB x4 net at 2 x 24 x 20: re-associated dense blocks, two image groups, tail chain + trunk chain.  (A batch of 2, not 1:
    build_plan gives a one-image batch a single image group.)"""
    net, _ = _net("rrdbnet_x4", 2)
    lr, gt = _inputs(net, (2, 3, 24, 20))
    _check_pattern(net, lr, gt, pattern, x_grad)


@pytest.mark.parametrize("factory,shape", [("rrdbnet_x1", (2, 3, 16, 16)), ("rrdbnet_x8", (1, 3, 16, 12)),
                                           ("rrdbnet_x4", (1, 3, 160, 264))], ids=["x1", "x8", "per_conv_frame"])
@pytest.mark.parametrize("pattern,x_grad", [PATTERNS[i] for i in (0, 1, 2, 3, 4)], ids=[_IDS[i] for i in (0, 1, 2, 3, 4)])
def test_patterns_other_geometries(factory, shape, pattern, x_grad):
    """x1 (no upsampling), x8 (three upsample stages), and the per-conv large-frame schedule (one chain for tail and trunk)."""
    net, _ = _net(factory, 2 if factory == "rrdbnet_x1" else 1)
    lr, gt = _inputs(net, shape)
    _check_pattern(net, lr, gt, pattern, x_grad)


@pytest.mark.parametrize("pattern", ["tail", "head+half"])
def test_patterns_config2_deterministic(pattern):
    """BASELINE config 2: 16 x 64 x 64, 23 RRDBs, in deterministic mode, where the partial backward must give the full backward's
    gradients bit for bit.  In the default mode the red.global.add order alone moves the bias gradients of these long sums (the
    upsample convs' run over 262 144 pixels) by a relative L2 of about 1e-6 (1.06e-6 measured for upsampling1.0.bias), so the
    1e-6 bar of the small geometries above could not tell a reordering from a fault here."""
    net, _ = _net("rrdbnet_x4", 23)
    lr, gt = _inputs(net, (16, 3, 64, 64))
    prev = torch.are_deterministic_algorithms_enabled(), torch.is_deterministic_algorithms_warn_only_enabled()
    torch.use_deterministic_algorithms(True, warn_only=True)
    try:
        _check_pattern(net, lr, gt, pattern, False, exact=True)
        assert net._runtime().last_plan.deterministic
    finally:
        torch.use_deterministic_algorithms(prev[0], warn_only=prev[1])


def test_partial_gradients_against_oracle():
    """Pattern (g) at the fp32 oracle's bar: trainable gradients and dL/dx."""
    net, params = _net("rrdbnet_x4", 2)
    lr, gt = _inputs(net, (2, 3, 24, 20))
    part, dx = _check_pattern(net, lr, gt, "head+half", True)
    p_ref = {k: v.clone().requires_grad_(True) for k, v in params.items()}
    x_ref = lr.clone().requires_grad_(True)
    F.l1_loss(orc.rrdbnet_forward(p_ref, x_ref), gt).backward()
    assert orc.rel_l2(dx.cpu(), x_ref.grad) <= TOL_GRAD
    got = [g.flatten().cpu() for g in part if g is not None]
    ref = [p_ref[n].grad.flatten() for (n, _), g in zip(net.named_parameters(), part) if g is not None]
    assert orc.rel_l2(torch.cat(got), torch.cat(ref)) <= TOL_GRAD


def test_profiler_shows_the_skipped_work():
    """Config 2, conv1 and RRDBs 0-10 frozen: the backward launches exactly what b200sr_backward_launches counts, one
    weight-gradient launch per dense block with a wanted conv (plus the tail's), and ONE trunk chain launch behind the tail's."""
    from torch.profiler import ProfilerActivity, profile
    net, _ = _net("rrdbnet_x4", 23)
    lr, gt = _inputs(net, (16, 3, 64, 64))
    _set_pattern(net, "head+half")
    _backward(net, lr, gt, False)  # warm: plan, descriptors, packed weights
    x = lr.to(DEV)
    loss = F.l1_loss(net(x), gt.to(DEV))
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        loss.backward()
        torch.cuda.synchronize()
    ours = ("conv3x3_chain_kernel", "wgrad3x3_kernel", "bias_grad_vec_kernel", "unpack_wgrad_kernel", "add_carriers_to_bf16_kernel",
            "ingest_grad_kernel")  # every kernel a generator backward launches
    names = [e.name for e in prof.events() if any(k in e.name for k in ours)]
    plan = net._runtime().last_plan
    fl = flags(net, "head+half")
    assert len(names) == plan.backward_launches(fl), sorted(set(names))
    L = net._n_up
    wanted_blocks = 3 * (23 - 23 // 2)
    assert sum("wgrad3x3_kernel" in n for n in names) == wanted_blocks + 3 + 2 * L  # + conv4, conv3, 2 per upsample stage, conv2
    assert sum("conv3x3_chain_kernel" in n for n in names) == 2                      # HR tail chain + ONE trunk chain
    assert plan.launches_bwd > plan.backward_launches(fl) > plan.backward_launches(flags(net, "tail")) > \
        plan.backward_launches(flags(net, "conv4"))


def test_data_parallel_buckets_cover_wanted_convs():
    """make_data_parallel(overlap=True) in one process: every wanted conv's range lies in an announced bucket, no bucket holds
    only frozen convs, and the flat buffer is zero over the frozen convs (also those inside a trainable dense block)."""
    from sr_gan_fd_b200.dist import make_data_parallel
    net, _ = _net("rrdbnet_x4", 8)
    lr, gt = _inputs(net, (2, 3, 24, 20))
    reducer = make_data_parallel(net, overlap=True)
    rt = net._runtime()
    flats = []
    finish = rt.grad_done_hook
    rt.grad_done_hook = lambda flat: (flats.append(flat), finish(flat))
    net.trunk[6].rdb2.conv3.weight.requires_grad_(False)  # one frozen conv inside a trainable dense block
    net.trunk[6].rdb2.conv3.bias.requires_grad_(False)
    for n, p in net.named_parameters():
        if n.startswith("conv1.") or (n.startswith("trunk.") and int(n.split(".")[1]) < 4):
            p.requires_grad_(False)
    F.l1_loss(net(lr.to(DEV)), gt.to(DEV)).backward()
    torch.cuda.synchronize()
    numels = [p.numel() for p in net.parameters()]
    offs = [0]
    for k in numels:
        offs.append(offs[-1] + k)
    want = [p.requires_grad for p in net.parameters()]
    conv_ranges = [(offs[i], offs[i + 2], want[i] or want[i + 1]) for i in range(0, len(numels), 2)]
    buckets = reducer.buckets_seen
    assert buckets
    for lo, hi, w in conv_ranges:
        if w:
            assert any(o <= lo and hi <= o + c for o, c in buckets), (lo, hi, buckets)
    for o, c in buckets:
        assert any(w and o <= lo and hi <= o + c for lo, hi, w in conv_ranges), f"bucket {(o, c)} holds only frozen convs"
    flat = flats[0]
    for lo, hi, w in conv_ranges:
        if not w:
            assert int(torch.count_nonzero(flat[lo:hi])) == 0, (lo, hi)


def _trainable_without_first_blocks(model):
    return [not (n.startswith("conv1.") or (n.startswith("trunk.") and n.split(".")[2] == "rdb1")) for n, _ in model.named_parameters()]


@pytest.mark.parametrize("use_scaler", [False, True], ids=["plain", "gradscaler_inf_step"])
def test_fused_adam_ema_with_frozen_parameters_matches_torch(use_scaler):
    """FusedAdamEMA with parameters whose .grad is None == torch.optim.Adam (which skips them) + AveragedModel(avg_fn) (which
    averages every parameter) + GradScaler, including a step with an injected inf; frozen parameters stay bit-identical."""
    import sr_gan_fd_b200 as b200
    from sr_gan_fd_b200.optim import FusedAdamEMA
    decay = 0.99998
    torch.manual_seed(0)
    ref = b200.rrdbnet_x4(num_blocks=1).to(DEV)
    mine = copy.deepcopy(ref)
    train = _trainable_without_first_blocks(ref)
    for model in (ref, mine):
        for p, t in zip(model.parameters(), train):
            p.requires_grad_(t)
    frozen0 = [p.detach().clone() for p, t in zip(mine.parameters(), train) if not t]
    ema_avg = lambda avg, p, n: (1 - decay) * avg + decay * p
    ref_ema, mine_ema = AveragedModel(ref, avg_fn=ema_avg), AveragedModel(mine, avg_fn=ema_avg)
    opt_ref = torch.optim.Adam(ref.parameters(), 2e-4, (0.9, 0.99), 1e-8, 0.0)
    opt_mine = FusedAdamEMA(mine.parameters(), 2e-4, (0.9, 0.99), 1e-8, 0.0, ema_model=mine_ema, ema_decay=decay)
    scaler_ref = torch.amp.GradScaler("cuda", enabled=use_scaler)
    scaler_mine = torch.amp.GradScaler("cuda", enabled=use_scaler)
    g = torch.Generator().manual_seed(3)
    for it in range(4):
        grads = [torch.randn(p.shape, generator=g).to(DEV) * 1e-3 if t else None for p, t in zip(ref.parameters(), train)]
        if use_scaler and it == 2:
            grads[-1][0] = float("inf")
        scale = 65536.0 if use_scaler else 1.0
        for model in (ref, mine):
            for p, gr in zip(model.parameters(), grads):
                p.grad = (gr * scale).clone() if gr is not None else None
        if use_scaler:
            if it == 0:
                scaler_ref.scale(torch.ones(1, device=DEV)); scaler_mine.scale(torch.ones(1, device=DEV))
            scaler_ref.step(opt_ref); scaler_ref.update()
            scaler_mine.step(opt_mine); scaler_mine.update()
        else:
            opt_ref.step()
            opt_mine.step()
        ref_ema.update_parameters(ref)
    for (n, a), b in zip(ref.named_parameters(), mine.parameters()):
        assert torch.allclose(a, b, rtol=2e-5, atol=1e-8), n
    for a, b in zip(ref_ema.module.parameters(), mine_ema.module.parameters()):
        assert torch.allclose(a, b, rtol=2e-5, atol=1e-8)
    assert all(torch.equal(a, b) for a, b in zip(frozen0, [p for p, t in zip(mine.parameters(), train) if not t]))
    assert int(mine_ema.n_averaged) == int(ref_ema.n_averaged)


def test_tail_only_fine_tuning_loop():
    """Three steps of a tail-only fine-tune through the native generator and FusedAdamEMA: every step re-packs the weights,
    the tail moves, the frozen trunk and head stay bit-identical."""
    from sr_gan_fd_b200.optim import FusedAdamEMA
    net, _ = _net("rrdbnet_x4", 2)
    _set_pattern(net, "tail")
    fl = flags(net, "tail")
    before = [p.detach().clone() for p in net.parameters()]
    ema = AveragedModel(net, avg_fn=lambda avg, p, n: 0.5 * avg + 0.5 * p)
    opt = FusedAdamEMA(net.parameters(), 1e-3, ema_model=ema, ema_decay=0.5)
    rt = net._runtime()
    serials = []
    for step in range(3):
        lr, gt = _inputs(net, (2, 3, 24, 20), seed=10 + step)
        F.l1_loss(net(lr.to(DEV)), gt.to(DEV)).backward()
        serials.append(sum(rt.pack_serial.values()))
        opt.step()
        opt.zero_grad(set_to_none=True)
    torch.cuda.synchronize()
    assert serials[0] < serials[1] < serials[2], serials  # the updated tail was re-packed before each later forward
    for (n, p), b, t in zip(net.named_parameters(), before, fl):
        if t:
            assert not torch.equal(p, b), f"{n} did not move"
        else:
            assert torch.equal(p, b), f"frozen {n} changed"
