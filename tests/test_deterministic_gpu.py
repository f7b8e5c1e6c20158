"""GPU: deterministic mode (torch.use_deterministic_algorithms).  Every native call gives bit-identical outputs for
bit-identical inputs, whatever the stream timing, the bucket callback, dx or the freeze pattern; and it stays within the
rel-L2 1e-6 of the default mode, whose atomics only reorder the same partial sums.  Bits are compared as int32 views."""
import contextlib
import ctypes as C
import os
import subprocess
import sys

import pytest
import torch
import torch.nn.functional as F

from oracle import rrdbnet_oracle as orc
from test_partial_grad_gpu import _inputs, _net
from test_partial_grad_host import flags

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda", 0)
TOL_SAME = 1e-6
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@contextlib.contextmanager
def det_mode(on=True, warn_only=True):
    """warn_only: deterministic mode is on either way; torch's own helpers in these tests (the busy matmul, the spectral norm)
    must not raise for a cuBLAS workspace setting that only the end-to-end subprocess test makes"""
    prev = torch.are_deterministic_algorithms_enabled(), torch.is_deterministic_algorithms_warn_only_enabled()
    torch.use_deterministic_algorithms(on, warn_only=warn_only)
    try:
        yield
    finally:
        torch.use_deterministic_algorithms(prev[0], warn_only=prev[1])


def bits(t):
    return t.detach().contiguous().view(torch.int32).cpu()


def same_bits(a, b):
    return torch.equal(bits(a), bits(b))


def native_backward(net, y, dy, with_dx, mask=None, cb=False, busy=False):
    """One more backward of the native forward that made y (the library allows several), straight through the C ABI."""
    from sr_gan_fd_b200 import lib as _lib
    from sr_gan_fd_b200.function import conv_mask
    fn, lib = y.grad_fn, _lib.load()
    plan = fn.plan
    flat = torch.empty(plan.param_numel, dtype=torch.float32, device=DEV)
    dx = torch.empty(fn.x_meta[0], dtype=torch.float32, device=DEV) if with_dx else None
    seen = []
    cbf = _lib.BUCKET_CB(lambda user, off, cnt: seen.append((int(off), int(cnt)))) if cb else _lib.BUCKET_CB()
    side = torch.cuda.Stream()
    if busy:  # other work on the device while the backward runs
        a = torch.randn(4096, 4096, device=DEV)
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            for _ in range(20):
                a = a @ a
                a /= a.norm()
    stream = torch.cuda.current_stream().cuda_stream
    m = conv_mask(mask) if mask is not None else None
    _lib.check(lib.b200sr_backward_select(plan.handle, C.c_void_p(dy.data_ptr()), C.c_void_p(fn.packed.data_ptr()),
                                          C.c_void_p(fn.workspace.data_ptr()), C.c_void_p(flat.data_ptr()),
                                          C.c_void_p(dx.data_ptr()) if dx is not None else None, m, cbf, None, C.c_void_p(stream)))
    torch.cuda.synchronize()
    assert not cb or seen
    return flat, dx


def forward_dy(net, lr, gt, x_grad=True):
    x = lr.to(DEV).requires_grad_(x_grad)
    y = net(x)
    dy = torch.autograd.grad(F.l1_loss(y, gt.to(DEV)), y, retain_graph=True)[0].contiguous()
    return x, y, dy


GEOMETRIES = [
    ("rrdbnet_x4", 2, (2, 3, 24, 20)),     # two image groups
    ("rrdbnet_x1", 2, (2, 3, 16, 16)),     # no upsampling
    ("rrdbnet_x8", 1, (1, 3, 16, 12)),     # three upsample stages
    ("rrdbnet_x4", 1, (1, 3, 160, 264)),   # per-conv schedule
    ("rrdbnet_x4", 1, (2, 12, 24, 20)),    # in_channels 12 (what a pixel-unshuffle front feeds conv1)
    ("rrdbnet_x4", 23, (16, 3, 64, 64)),   # config 2
]


@pytest.mark.parametrize("factory,nb,shape", GEOMETRIES, ids=["x4_groups", "x1", "x8", "per_conv", "in12", "config2"])
def test_generator_backward_is_bit_repeatable(factory, nb, shape):
    if shape[1] != 3:
        import sr_gan_fd_b200 as b200
        torch.manual_seed(0)
        net = getattr(b200, factory)(num_blocks=nb, in_channels=shape[1])
        net.load_state_dict(orc.in_range_fixture({k: v.detach().clone() for k, v in net.state_dict().items()}))
        net = net.to(DEV).train()
    else:
        net, _ = _net(factory, nb)
    lr, gt = _inputs(net, shape)
    with det_mode():
        x, y, dy = forward_dy(net, lr, gt)
        assert net._runtime().last_plan.deterministic
        flat0, dx0 = native_backward(net, y, dy, True)
        for kw in (dict(), dict(cb=True), dict(busy=True), dict(cb=True, busy=True)):
            flat, dx = native_backward(net, y, dy, True, **kw)
            assert same_bits(flat, flat0) and same_bits(dx, dx0), kw
        flat, dx = native_backward(net, y, dy, False)
        assert dx is None and same_bits(flat, flat0)
        # forward + backward pairs through autograd
        for _ in range(2 if nb == 23 else 4):
            x2, y2, _ = forward_dy(net, lr, gt)
            assert same_bits(y2, y)
            F.l1_loss(y2, gt.to(DEV)).backward()
            g = torch.cat([p.grad.flatten() for p in net.parameters()])
            net.zero_grad(set_to_none=True)
            assert same_bits(g, flat0) and same_bits(x2.grad, dx0)
    # the default mode: the same sums in another order
    x, y, dy = forward_dy(net, lr, gt)
    assert not net._runtime().last_plan.deterministic
    ref, ref_dx = native_backward(net, y, dy, True)
    assert same_bits(ref_dx, dx0)  # the data-gradient chain never used atomics
    rt = net._runtime()
    for (name, _), a, b in zip(net.named_parameters(), ref.split(rt.param_numels), flat0.split(rt.param_numels)):
        assert orc.rel_l2(b.cpu(), a.cpu()) <= TOL_SAME, name


@pytest.mark.parametrize("factory,nb,shape", [GEOMETRIES[0], GEOMETRIES[5]], ids=["x4_groups", "config2"])
def test_generator_freeze_patterns_match_the_full_deterministic_backward(factory, nb, shape):
    net, _ = _net(factory, nb)
    lr, gt = _inputs(net, shape)
    rt = net._runtime()
    with det_mode():
        x, y, dy = forward_dy(net, lr, gt)
        full, full_dx = native_backward(net, y, dy, True)
        for pattern in ("tail", "conv4", "head+half", "one_conv", "no_bias"):
            fl = flags(net, pattern)
            for with_dx in (False, True):
                part, dx = native_backward(net, y, dy, with_dx, mask=fl)
                if with_dx:
                    assert same_bits(dx, full_dx), pattern
                for (name, _), want, a, b in zip(net.named_parameters(), fl, part.split(rt.param_numels), full.split(rt.param_numels)):
                    if want:
                        assert same_bits(a, b), (pattern, name)


def test_generator_fp16_tail_is_bit_repeatable(monkeypatch):
    monkeypatch.setenv("B200SR_TAIL_FP16", "1")
    net, _ = _net("rrdbnet_x4", 2)
    lr, gt = _inputs(net, (2, 3, 24, 20))
    with det_mode(warn_only=True):
        x, y, dy = forward_dy(net, lr, gt)
        a, adx = native_backward(net, y, dy, True)
        b, bdx = native_backward(net, y, dy, True, busy=True)
    assert same_bits(a, b) and same_bits(adx, bdx)


@pytest.mark.parametrize("fp16,shape", [(True, (16, 3, 256, 256)), (False, (2, 3, 64, 64))], ids=["fp16_16x256", "bf16_2x64"])
def test_discriminator_gradients_are_bit_repeatable(fp16, shape):
    from sr_gan_fd_b200.discriminator import discriminator_unet
    torch.manual_seed(0)
    d = discriminator_unet(in_channels=3, out_channels=1, channels=64).to(DEV)
    d.operand_dtype = "fp16" if fp16 else "bf16"
    x0 = torch.rand(*shape, generator=torch.Generator().manual_seed(3)).to(DEV)
    # a fresh module's power-iteration vectors are random (sigma far from the spectral norm, weights that overflow fp16): a few
    # training-mode forwards settle them, then eval keeps them fixed so that every call sees the same effective weights
    with torch.no_grad():
        for _ in range(5):
            d(x0)
    d.eval()

    def run(with_dx):
        x = x0.clone().requires_grad_(with_dx)
        d(x).square().mean().backward()
        g = torch.cat([p.grad.flatten() for p in d.parameters() if p.grad is not None])
        d.zero_grad(set_to_none=True)
        return g, (x.grad if with_dx else None)

    with det_mode():
        g0, dx0 = run(True)
        assert d._runtime().last_plan.deterministic
        for with_dx in (True, False, True):
            g, dx = run(with_dx)
            assert same_bits(g, g0)
            if with_dx:
                assert same_bits(dx, dx0)
    ref, _ = run(True)
    assert not d._runtime().last_plan.deterministic
    assert bool(torch.isfinite(g0).all())
    assert orc.rel_l2(g0.cpu(), ref.cpu()) <= TOL_SAME


def test_vgg_loss_and_iqa_sums_are_bit_repeatable():
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    import gan_step
    from sr_gan_fd_b200.iqa import PSNR, SSIM
    from sr_gan_fd_b200.vgg import ContentLoss, ContentLossMulti
    gan_step.patch_vgg19()  # seeded random weights: no download
    multi = ContentLossMulti(gan_step.NODES, gan_step.MEAN, gan_step.STD).to(DEV)  # the five-node loss value of the GAN step
    single = ContentLoss(gan_step.NODES[-1], gan_step.MEAN, gan_step.STD).to(DEV)  # one node, with the gradient w.r.t. sr
    g = torch.Generator().manual_seed(5)
    sr = torch.rand(4, 3, 96, 96, generator=g).to(DEV).requires_grad_(True)
    gt = torch.rand(4, 3, 96, 96, generator=g).to(DEV)
    psnr, ssim = PSNR(4, True), SSIM(4, True)

    def run():
        v = multi(sr, gt).double()
        (gs,) = torch.autograd.grad(single(sr, gt), sr)
        return v, gs, psnr(sr.detach(), gt).double(), ssim(sr.detach(), gt).double()

    with det_mode():
        outs = [run() for _ in range(5)]
    for o in outs[1:]:
        assert torch.equal(o[0].view(torch.int64), outs[0][0].view(torch.int64))
        assert same_bits(o[1], outs[0][1])
        assert torch.equal(o[2].view(torch.int64), outs[0][2].view(torch.int64))
        assert torch.equal(o[3].view(torch.int64), outs[0][3].view(torch.int64))
    ref = run()  # the default mode: the same sums, atomics in another order
    for a, b in zip(ref, outs[0]):
        assert orc.rel_l2(b.double().cpu(), a.double().cpu()) <= 1e-6


_GAN_SCRIPT = r"""
import hashlib, os, sys
import torch
torch.use_deterministic_algorithms(True)
sys.path.insert(0, os.path.join(sys.argv[1], "tools"))
import gan_step
dev = torch.device("cuda", 0)
d, g, content = gan_step.build("b200", dev, seed=0, content="b200", disc="b200")
d.train(); g.train()
step = gan_step.GanStep(d, g, content, dev, optimizer="fused", ema=True)
gen = torch.Generator().manual_seed(8)
lr = torch.rand(2, 3, 32, 32, generator=gen).to(dev)
gt = torch.rand(2, 3, 128, 128, generator=gen).to(dev)
for _ in range(3):
    step(lr, gt)
torch.cuda.synchronize()
h = hashlib.sha256()
for sd in (g.state_dict(), d.state_dict(), step.ema.state_dict()):
    for k, v in sd.items():
        h.update(k.encode()); h.update(v.detach().contiguous().cpu().numpy().tobytes())
print("HASH", h.hexdigest())
"""


def _gan_hash():
    env = dict(os.environ, CUBLAS_WORKSPACE_CONFIG=":4096:8")
    r = subprocess.run([sys.executable, "-c", _GAN_SCRIPT, ROOT], capture_output=True, text=True, env=env, cwd=ROOT, timeout=900)
    assert r.returncode == 0, r.stderr[-4000:]
    return [l for l in r.stdout.splitlines() if l.startswith("HASH")][-1]


def test_all_native_gan_steps_are_bit_reproducible_across_processes():
    """Three all-native GAN steps (generator, U-Net discriminator, VGG loss, FusedAdamEMA) from seed 0 under
    torch.use_deterministic_algorithms(True): two processes end with the same generator, discriminator and EMA weights."""
    assert _gan_hash() == _gan_hash()
