"""GPU: unclamped generator plans and BasicSR's RRDBNet layout (BasicSRRRDBNet / native_generator).

* Same weights, same input: clamp(y_unclamped, 0, 1) is the clamped plan's y bit for bit (training and inference plans); in
  deterministic mode the unclamped backward of where(0 <= y <= 1, dy, 0) is the clamped backward of dy bit for bit (flat gradients, dx).
* Against the fp32 oracle's pre-clamp output, with at least 20 % of the outputs outside [0, 1]: output rel-L2 <= 5e-3, flat gradients and dx <= 1e-2.
* The module under autocast + GradScaler + FusedAdamEMA, freeze patterns, determinism, input dtypes and layouts, tiled inference, a
  workspace poisoned with 0xFF, and native_generator on an instance of BasicSR's class."""
import ctypes as C

import pytest
import torch
from torch import nn

import sr_gan_fd_b200 as b200
from oracle import rrdbnet_oracle as orc
from sr_gan_fd_b200 import lib as _lib
from sr_gan_fd_b200 import tile
from test_basicsr_host import RRDBNet as BasicSRRef
from test_gen_stages_gpu import make_params

pytestmark = pytest.mark.gpu

TOL_OUT, TOL_GRAD, TOL_SAME = 5e-3, 1e-2, 1e-6
# (num_blocks, batch, height, width, in_channels): config-2 geometry, uneven image groups, the per-conv schedule of a large frame,
# and the 12-channel input of a scale-2 model (pixel-unshuffled by 2)
GEOS = [(2, 16, 64, 64, 3), (2, 3, 40, 72, 3), (1, 1, 256, 256, 3), (2, 4, 32, 48, 12)]
GEO_IDS = [f"{nb}rrdb-{n}x{h}x{w}-in{c}" for nb, n, h, w, c in GEOS]


def _params(in_ch, nb, seed, dev):
    """make_params with conv4's weights scaled down: the outputs straddle [0, 1], so the clamp cuts some and passes others"""
    p = make_params(in_ch, 3, nb, 2, seed, dev)
    p[-2] = (p[-2] * 0.25).contiguous()
    return p


class _Raw:
    """one clamped or unclamped generator plan driven through the C ABI, on buffers filled with 0xFF (NaN in bf16 and fp32)"""

    def __init__(self, nb, n, h, w, training, unclamped, det=False, in_ch=3):
        self.L = _lib.load()
        self.n, self.h, self.w, self.in_ch = n, h, w, in_ch
        nd = _lib.NetDesc(in_ch, 3, 64, 32, nb, 2, n, h, w, int(training), 0, int(det))
        self.handle = C.c_void_p()
        create = self.L.b200sr_unclamped_plan_create if unclamped else self.L.b200sr_plan_create
        _lib.check(create(C.byref(nd), C.byref(self.handle)))
        self.dev = torch.device("cuda", 0)
        self.stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
        self.ws = torch.full((int(self.L.b200sr_workspace_bytes(self.handle)),), 0xFF, dtype=torch.uint8, device=self.dev)
        self.pk = torch.zeros(int(self.L.b200sr_packed_bytes(self.handle)), dtype=torch.uint8, device=self.dev)
        self.numel = int(self.L.b200sr_param_numel(self.handle))

    def __del__(self):
        if getattr(self, "handle", None):
            self.L.b200sr_plan_destroy(self.handle)

    def _nan(self, *shape):
        return torch.full(shape, -1, dtype=torch.int32, device=self.dev).view(torch.float32)

    def pack(self, params):
        self.params = params
        ptrs = (C.c_void_p * len(params))(*[t.data_ptr() for t in params])
        _lib.check(self.L.b200sr_pack_weights(self.handle, ptrs, C.c_void_p(self.pk.data_ptr()), self.stream))

    def forward(self, x):
        y = self._nan(self.n, 3, 4 * self.h, 4 * self.w)
        _lib.check(self.L.b200sr_forward(self.handle, C.c_void_p(x.data_ptr()), _lib.F32, (C.c_int64 * 4)(*x.stride()),
                                         C.c_void_p(self.pk.data_ptr()), C.c_void_p(self.ws.data_ptr()), C.c_void_p(y.data_ptr()),
                                         self.stream))
        torch.cuda.synchronize()
        return y

    def backward(self, dy):
        g = self._nan(self.numel)
        dx = self._nan(self.n, self.in_ch, self.h, self.w)
        _lib.check(self.L.b200sr_backward(self.handle, C.c_void_p(dy.data_ptr()), C.c_void_p(self.pk.data_ptr()),
                                          C.c_void_p(self.ws.data_ptr()), C.c_void_p(g.data_ptr()), C.c_void_p(dx.data_ptr()),
                                          _lib.BUCKET_CB(), None, self.stream))
        torch.cuda.synchronize()
        return g, dx


def _bits(a, b):
    return torch.equal(a.contiguous().view(torch.int32), b.contiguous().view(torch.int32))


@pytest.mark.parametrize("training", [True, False])
@pytest.mark.parametrize("geo", GEOS, ids=GEO_IDS)
def test_clamped_unclamped_output_is_the_clamped_output(geo, training):
    nb, n, h, w, in_ch = geo
    params = _params(in_ch, nb, 7, torch.device("cuda", 0))
    x = torch.rand(n, in_ch, h, w, device="cuda", generator=torch.Generator(device="cuda").manual_seed(8))
    outs = []
    for unclamped in (False, True):
        r = _Raw(nb, n, h, w, training, unclamped, in_ch=in_ch)
        r.pack(params)
        outs.append(r.forward(x))
    yc, yu = outs
    assert bool(torch.isfinite(yu).all())
    outside = float(((yu < 0) | (yu > 1)).float().mean())
    assert 0.05 < outside < 0.95, outside  # both sides of the clamp are exercised
    assert torch.equal(torch.clamp(yu, 0, 1), yc), f"{int((torch.clamp(yu, 0, 1) != yc).sum())} of {yc.numel()} elements differ"


@pytest.mark.parametrize("geo", GEOS, ids=GEO_IDS)
def test_unclamped_backward_of_the_masked_gradient_is_the_clamped_backward(geo):
    """deterministic plans: the clamped backward of dy is the unclamped backward of dy with the clamp's pass-through mask applied"""
    nb, n, h, w, in_ch = geo
    dev = torch.device("cuda", 0)
    params = _params(in_ch, nb, 11, dev)
    g = torch.Generator(device="cuda").manual_seed(12)
    x = torch.rand(n, in_ch, h, w, device=dev, generator=g)
    dy = torch.randn(n, 3, 4 * h, 4 * w, device=dev, generator=g)
    clamped = _Raw(nb, n, h, w, True, False, det=True, in_ch=in_ch)
    clamped.pack(params)
    clamped.forward(x)
    gc, dxc = clamped.backward(dy)
    unclamped = _Raw(nb, n, h, w, True, True, det=True, in_ch=in_ch)
    unclamped.pack(params)
    yu = unclamped.forward(x)
    m = (0 <= yu) & (yu <= 1)
    gu, dxu = unclamped.backward(torch.where(m, dy, 0.0))  # where, not a multiply: -dy * 0 is -0.0
    assert bool(torch.isfinite(gu).all()) and bool(torch.isfinite(dxu).all())
    assert _bits(gu, gc), f"{int((gu != gc).sum())} of {gc.numel()} gradient elements differ"
    assert _bits(dxu, dxc), f"{int((dxu != dxc).sum())} of {dxc.numel()} input-gradient elements differ"
    # and the plain unclamped backward differs: dy outside the clamp's range reaches the weights
    gu_full, _ = unclamped.backward(dy)
    assert not torch.equal(gu_full, gc)


def _module(scale, nb, seed, dev=None):
    torch.manual_seed(seed)
    net = b200.BasicSRRRDBNet(3, 3, scale=scale, num_block=nb)
    in_ch = net.conv_first.in_channels
    with torch.no_grad():
        for p, v in zip(net.parameters(), _params(in_ch, nb, seed, torch.device("cpu"))):
            p.copy_(v)
    return net.to(dev) if dev is not None else net


def _oracle(net, x, dy):
    """fp32 oracle of the unclamped output (its pre-clamp value), dx and the flat gradient in state_dict order"""
    nb = len(net.body)
    names = orc.conv_names(nb, 2)
    vals = [p.detach().cpu().clone().requires_grad_(True) for p in net.parameters()]
    p = {f"{names[i // 2]}.{'weight' if i % 2 == 0 else 'bias'}": v for i, v in enumerate(vals)}
    xr = x.detach().cpu().float().clone().requires_grad_(True)
    _, pre = orc.rrdbnet_forward(p, xr, pixel_unshuffle=net._pixel_unshuffle, return_pre_clamp=True)
    pre.backward(dy.cpu())
    return pre.detach(), xr.grad, torch.cat([v.grad.flatten() for v in vals])


@pytest.mark.parametrize("layout", ["nchw", "channels_last"])
@pytest.mark.parametrize("scale", [4, 2])
def test_against_the_fp32_oracle(scale, layout):
    dev = torch.device("cuda", 0)
    net = _module(scale, 2, seed=21)
    g = torch.Generator().manual_seed(22)
    x = torch.rand(4, 3, 32 * net._pixel_unshuffle, 40 * net._pixel_unshuffle, generator=g)
    dy = torch.randn(4, 3, x.shape[2] * scale, x.shape[3] * scale, generator=g)
    y_ref, dx_ref, g_ref = _oracle(net, x, dy)
    outside = float(((y_ref < 0) | (y_ref > 1)).float().mean())
    assert outside >= 0.2, f"only {outside:.1%} of the outputs lie outside [0, 1]: the fixture would not show a clamp"
    net = net.to(dev)
    xd = x.to(dev)
    if layout == "channels_last":
        xd = xd.to(memory_format=torch.channels_last)
    xd.requires_grad_(True)
    y = net(xd)
    assert y.dtype == torch.float32 and y.shape == y_ref.shape
    y.backward(dy.to(dev))
    flat = torch.cat([p.grad.flatten() for p in net.parameters()]).cpu()
    assert orc.rel_l2(y.detach().cpu(), y_ref) <= TOL_OUT
    assert orc.rel_l2(xd.grad.cpu(), dx_ref) <= TOL_GRAD
    assert orc.rel_l2(flat, g_ref) <= TOL_GRAD
    with torch.no_grad():  # inference plan (fp16 tail): same bar
        assert orc.rel_l2(net.eval()(xd).cpu(), y_ref) <= TOL_OUT


def test_input_dtypes_layouts_and_tiling():
    dev = torch.device("cuda", 0)
    net = _module(4, 2, seed=23, dev=dev)
    x = torch.rand(2, 3, 96, 40, device=dev, generator=torch.Generator(device="cuda").manual_seed(24))
    with torch.no_grad():
        y = net(x)
        assert _bits(net(x.to(memory_format=torch.channels_last)), y)
        for dt in (torch.float16, torch.bfloat16):
            xl = x.to(dt)
            assert _bits(net(xl), net(xl.float()))
        whole = net(x)
        tiled, _ = tile.tiled_forward(net, x, 4, num_bands=2, halo=40)
    assert orc.rel_l2(tiled, whole) <= TOL_OUT


def test_autocast_gradscaler_fused_adam_ema_step():
    from sr_gan_fd_b200.optim import FusedAdamEMA
    dev = torch.device("cuda", 0)
    mine = _module(4, 2, seed=25, dev=dev)
    ref = BasicSRRef(3, 3, scale=4, num_block=2).to(dev)
    ref.load_state_dict(mine.state_dict())
    ema = torch.optim.swa_utils.AveragedModel(mine)
    lr = torch.rand(4, 3, 32, 40, device=dev)
    gt = torch.rand(4, 3, 128, 160, device=dev)
    prev = torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32
    torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = False
    try:
        sr_ref = ref(lr)
        nn.functional.l1_loss(sr_ref, gt).backward()
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = prev
    before = [p.detach().clone() for p in mine.parameters()]
    opt = FusedAdamEMA(mine.parameters(), 1e-4, (0.9, 0.99), 1e-8, 0.0, ema_model=ema, ema_decay=0.999)
    scaler = torch.amp.GradScaler("cuda", init_scale=1024.0)
    with torch.autocast("cuda", dtype=torch.float16):
        sr = mine(lr)
        loss = nn.functional.l1_loss(sr.float(), gt)
    scaler.scale(loss).backward()
    assert orc.rel_l2(sr.float(), sr_ref) <= TOL_OUT
    got = torch.cat([p.grad.flatten() for p in mine.parameters()]) / scaler.get_scale()
    want = torch.cat([p.grad.flatten() for p in ref.parameters()])
    assert orc.rel_l2(got, want) <= TOL_GRAD
    scaler.step(opt)
    scaler.update()
    torch.cuda.synchronize()
    moved = [float((p.detach() - b).abs().max()) for p, b in zip(mine.parameters(), before)]
    assert all(m > 0 for m in moved) and all(bool(torch.isfinite(p).all()) for p in mine.parameters())
    for pe, pm in zip(ema.module.parameters(), mine.parameters()):  # the first EMA update copies
        assert torch.equal(pe, pm)
    with torch.no_grad():
        assert orc.rel_l2(ema(lr), mine(lr)) == 0.0


def _trainable(name, pattern):
    if pattern == "head":
        return not name.startswith("conv_first.")
    if pattern == "first_rrdbs":
        return not (name.startswith("body.0.") or name.startswith("body.1."))
    if pattern == "frozen":
        return False
    raise ValueError(pattern)


@pytest.mark.parametrize("pattern", ["head", "first_rrdbs", "frozen"])
def test_freeze_patterns(pattern):
    dev = torch.device("cuda", 0)
    net = _module(4, 3, seed=27, dev=dev)
    g = torch.Generator(device="cuda").manual_seed(28)
    x = torch.rand(4, 3, 32, 40, device=dev, generator=g)
    dy = torch.randn(4, 3, 128, 160, device=dev, generator=g)

    def run(train):
        for p, t in zip(net.parameters(), train):
            p.requires_grad_(t)
            p.grad = None
        xx = x.clone().requires_grad_(True)
        net(xx).backward(dy)
        return [p.grad for p in net.parameters()], xx.grad

    names = [n for n, _ in net.named_parameters()]
    full, full_dx = run([True] * len(names))
    train = [_trainable(n, pattern) for n in names]
    got, dx = run(train)
    for name, t, gp, gf in zip(names, train, got, full):
        if not t:
            assert gp is None, f"{pattern}: {name} is frozen but got a gradient"
            continue
        assert gp is not None, f"{pattern}: {name} is trainable but got no gradient"
        assert orc.rel_l2(gp, gf) <= TOL_SAME, f"{pattern}: {name}"
    assert orc.rel_l2(dx, full_dx) <= TOL_SAME, f"{pattern}: dL/dx differs from the full backward's"


def test_deterministic_repeats_are_bit_identical():
    dev = torch.device("cuda", 0)
    net = _module(4, 2, seed=29, dev=dev)
    g = torch.Generator(device="cuda").manual_seed(30)
    x = torch.rand(16, 3, 64, 64, device=dev, generator=g)
    dy = torch.randn(16, 3, 256, 256, device=dev, generator=g)
    outs = []
    torch.use_deterministic_algorithms(True)
    try:
        for _ in range(3):
            net.zero_grad(set_to_none=True)
            xx = x.clone().requires_grad_(True)
            y = net(xx)
            y.backward(dy)
            outs.append([y.detach().clone(), xx.grad.clone()] + [p.grad.clone() for p in net.parameters()])
    finally:
        torch.use_deterministic_algorithms(False)
    for other in outs[1:]:
        assert all(_bits(a, b) for a, b in zip(outs[0], other))


@pytest.mark.parametrize("geo", GEOS[:2], ids=GEO_IDS[:2])
def test_poisoned_workspace_gives_the_module_results(geo):
    """the C ABI on 0xFF-filled workspace and outputs gives what the module gives on fresh allocations"""
    nb, n, h, w, _ = geo
    dev = torch.device("cuda", 0)
    net = _module(4, nb, seed=31, dev=dev)
    g = torch.Generator(device="cuda").manual_seed(32)
    x = torch.rand(n, 3, h, w, device=dev, generator=g)
    dy = torch.randn(n, 3, 4 * h, 4 * w, device=dev, generator=g)
    raw = _Raw(nb, n, h, w, True, True, det=True)
    raw.pack([p.detach() for p in net.parameters()])
    y = raw.forward(x)
    grads, dx = raw.backward(dy)
    assert bool(torch.isfinite(y).all()) and bool(torch.isfinite(grads).all()) and bool(torch.isfinite(dx).all())
    torch.use_deterministic_algorithms(True)
    try:
        xx = x.clone().requires_grad_(True)
        ym = net(xx)
        ym.backward(dy)
    finally:
        torch.use_deterministic_algorithms(False)
    assert _bits(y, ym.detach())
    assert _bits(grads, torch.cat([p.grad.flatten() for p in net.parameters()]))
    assert _bits(dx, xx.grad)


@pytest.mark.parametrize("scale", [4, 1])
def test_native_generator_on_basicsr_instance(scale):
    dev = torch.device("cuda", 0)
    torch.manual_seed(33)
    ref = BasicSRRef(3, 3, scale=scale, num_block=2).to(dev)
    loaded = b200.BasicSRRRDBNet(3, 3, scale=scale, num_block=2).to(dev)
    loaded.load_state_dict(ref.state_dict())
    adopted = b200.native_generator(ref)
    assert isinstance(adopted, b200.BasicSRRRDBNet)
    x = torch.rand(2, 3, 32, 40, device=dev)
    with torch.no_grad():
        assert _bits(adopted(x), loaded(x))
