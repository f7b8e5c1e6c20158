"""GPU: the RRDB trunk as a module of its own (trunk plans, RRDBTrunk / native_trunk).

* A trunk plan runs the generator's own trunk kernels: fed the generator's conv1 output (T0) it returns the generator's trunk
  output (TR) bit for bit; fed the gradient a tail-only generator backward leaves in GR, a deterministic trunk backward returns the
  full generator backward's trunk weight gradients and its final GR (the gradient w.r.t. conv1's output through the trunk) bit for bit.
* Against the fp32 oracle: output rel-L2 <= 5e-3; the increment y - x, dx and the flat gradient <= 1e-2.
* Freeze patterns, determinism, a workspace poisoned with 0xFF, and a composed model (torch head -> native trunk -> torch tail) under
  autocast + GradScaler against its eager fp32 copy."""
import copy
import ctypes as C

import pytest
import torch
from torch import nn

import sr_gan_fd_b200 as b200
from oracle import rrdbnet_oracle as orc
from sr_gan_fd_b200 import lib as _lib
from test_gen_stages_gpu import make_params, unblock

pytestmark = pytest.mark.gpu

TOL_OUT, TOL_GRAD, TOL_SAME = 5e-3, 1e-2, 1e-6
# (num_blocks, batch, height, width): config-2 geometry, uneven image groups, the per-conv schedule of a large frame
GEOS = [(2, 16, 64, 64), (2, 3, 40, 72), (1, 1, 256, 256)]
GEO_IDS = [f"{nb}rrdb-{n}x{h}x{w}" for nb, n, h, w in GEOS]


class _Raw:
    """one generator or trunk plan driven through the C ABI, on buffers filled with 0xFF (NaN in bf16 and fp32)"""

    def __init__(self, nb, n, h, w, training, trunk, det=False, in_ch=3, n_up=2):
        self.L = _lib.load()
        self.n, self.h, self.w, self.trunk = n, h, w, trunk
        ic, oc, up = (64, 64, 0) if trunk else (in_ch, 3, n_up)
        self.in_ch, self.out_ch, self.scale = ic, oc, 1 << up
        nd = _lib.NetDesc(ic, oc, 64, 32, nb, up, n, h, w, int(training), 0, int(det))
        self.handle = C.c_void_p()
        create = self.L.b200sr_trunk_plan_create if trunk else self.L.b200sr_plan_create
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
        s = self.scale
        y = self._nan(self.n, self.out_ch, s * self.h, s * self.w)
        dt = {torch.float32: _lib.F32, torch.float16: _lib.F16, torch.bfloat16: _lib.BF16}[x.dtype]
        _lib.check(self.L.b200sr_forward(self.handle, C.c_void_p(x.data_ptr()), dt, (C.c_int64 * 4)(*x.stride()),
                                         C.c_void_p(self.pk.data_ptr()), C.c_void_p(self.ws.data_ptr()), C.c_void_p(y.data_ptr()),
                                         self.stream))
        torch.cuda.synchronize()
        return y

    def backward(self, dy, want_dx=True, mask=None):
        g = self._nan(self.numel)
        dx = self._nan(self.n, self.in_ch, self.h, self.w) if want_dx else None
        m = (C.c_uint8 * len(mask))(*mask) if mask is not None else None
        _lib.check(self.L.b200sr_backward_select(self.handle, C.c_void_p(dy.data_ptr()), C.c_void_p(self.pk.data_ptr()),
                                                 C.c_void_p(self.ws.data_ptr()), C.c_void_p(g.data_ptr()),
                                                 C.c_void_p(dx.data_ptr()) if want_dx else None, m, _lib.BUCKET_CB(), None,
                                                 self.stream))
        torch.cuda.synchronize()
        return g, dx

    def region(self, name, dtype):
        off, nbytes = C.c_int64(-1), C.c_int64(-1)
        _lib.check(self.L.b200sr_debug_buffer(self.handle, name.encode(), C.byref(off), C.byref(nbytes)))
        return self.ws[off.value:off.value + nbytes.value].view(dtype)

    def carrier_nchw(self, name):
        """a tile-blocked fp32 carrier as [N, 64, H, W] (contiguous copy)"""
        return unblock(self.region(name, torch.float32), self.n, self.h, self.w).permute(0, 3, 1, 2).contiguous()


def _bits(a, b):
    return torch.equal(a.contiguous().view(torch.int32), b.contiguous().view(torch.int32))


def _trunk_slice(in_ch, nb):
    """the trunk's range of a generator's flat gradient buffer, and its parameter tensors' range of make_params' list"""
    lo = 64 * in_ch * 9 + 64
    return slice(lo, lo + 719_424 * nb), slice(2, 2 + 30 * nb)


@pytest.mark.parametrize("training", [True, False])
@pytest.mark.parametrize("geo", GEOS, ids=GEO_IDS)
def test_trunk_plan_reproduces_the_generator_trunk(geo, training):
    nb, n, h, w = geo
    params = make_params(3, 3, nb, 2, 7, torch.device("cuda", 0))
    gen = _Raw(nb, n, h, w, training, trunk=False)
    gen.pack(params)
    x = torch.rand(n, 3, h, w, device="cuda", generator=torch.Generator(device="cuda").manual_seed(8))
    gen.forward(x)
    t0, tr = gen.carrier_nchw("T0"), gen.carrier_nchw("TR")
    assert bool(torch.isfinite(t0).all()) and bool(torch.isfinite(tr).all())
    trunk = _Raw(nb, n, h, w, training, trunk=True)
    trunk.pack(params[_trunk_slice(3, nb)[1]])
    y = trunk.forward(t0)
    assert _bits(y, tr), f"{int((y != tr).sum())} of {y.numel()} elements differ from the generator's trunk output"
    assert _bits(trunk.carrier_nchw("TR"), tr)
    # channels_last and 16-bit inputs go through the same ingest
    assert _bits(trunk.forward(t0.to(memory_format=torch.channels_last)), tr)
    xh = t0.half()
    ref = trunk.forward(xh.float())
    assert _bits(trunk.forward(xh), ref)


@pytest.mark.parametrize("geo", GEOS, ids=GEO_IDS)
def test_trunk_backward_reproduces_the_generator_backward(geo):
    """deterministic plans: the trunk's weight gradients and its input gradient are the generator's, bit for bit"""
    nb, n, h, w = geo
    dev = torch.device("cuda", 0)
    params = make_params(3, 3, nb, 2, 11, dev)
    gsl, psl = _trunk_slice(3, nb)
    g = torch.Generator(device="cuda").manual_seed(12)
    x = torch.rand(n, 3, h, w, device=dev, generator=g)
    dy = torch.randn(n, 3, 4 * h, 4 * w, device=dev, generator=g)
    gen = _Raw(nb, n, h, w, True, trunk=False, det=True)
    gen.pack(params)
    gen.forward(x)
    nconv = len(params) // 2
    tail_only = [0] * (1 + 15 * nb) + [1] * (nconv - 1 - 15 * nb)
    gen.backward(dy, want_dx=False, mask=tail_only)
    g_out = gen.carrier_nchw("GR")            # conv2's data gradient = the gradient w.r.t. the trunk output
    t0 = gen.carrier_nchw("T0")
    full, _ = gen.backward(dy, want_dx=False)
    g_in = gen.carrier_nchw("GR")             # after the full walk: the gradient w.r.t. the trunk input (without the long skip)
    trunk = _Raw(nb, n, h, w, True, trunk=True, det=True)
    trunk.pack(params[psl])
    trunk.forward(t0)
    grads, dx = trunk.backward(g_out)
    assert _bits(grads, full[gsl]), f"{int((grads != full[gsl]).sum())} trunk gradient elements differ from the generator's"
    assert _bits(dx, g_in), f"{int((dx != g_in).sum())} input-gradient elements differ from the generator's GR"


def _trunk_module(nb, seed=0):
    torch.manual_seed(seed)
    t = b200.RRDBTrunk(num_blocks=nb)
    with torch.no_grad():  # larger trunk weights and non-zero biases: the increment y - x is not negligible
        for name, p in t.named_parameters():
            p.mul_(2.0) if name.endswith("weight") else p.add_(torch.randn_like(p) * 0.05)
    return t


def _oracle(trunk, x, dy):
    p = {"trunk." + k: v.detach().cpu().clone().requires_grad_(True) for k, v in trunk.state_dict().items()}
    xr = x.detach().cpu().float().clone().requires_grad_(True)
    y = xr
    for b in range(len(trunk)):
        y = orc.rrdb_forward(y, p, f"trunk.{b}")
    y.backward(dy.cpu())
    return y.detach(), xr.grad, torch.cat([v.grad.flatten() for v in p.values()])


@pytest.mark.parametrize("layout", ["nchw", "channels_last"])
def test_trunk_against_the_fp32_oracle(layout):
    dev = torch.device("cuda", 0)
    trunk = _trunk_module(3, seed=1)
    g = torch.Generator().manual_seed(2)
    x = torch.randn(4, 64, 40, 48, generator=g)
    dy = torch.randn(4, 64, 40, 48, generator=g)
    y_ref, dx_ref, g_ref = _oracle(trunk, x, dy)
    net = copy.deepcopy(trunk).to(dev)
    xd = x.to(dev)
    if layout == "channels_last":
        xd = xd.to(memory_format=torch.channels_last)
    xd.requires_grad_(True)
    y = net(xd)
    assert y.dtype == torch.float32 and y.shape == x.shape
    y.backward(dy.to(dev))
    flat = torch.cat([p.grad.flatten() for p in net.parameters()]).cpu()
    assert orc.rel_l2(y.cpu(), y_ref) <= TOL_OUT
    assert orc.rel_l2(y.detach().cpu() - x, y_ref - x) <= TOL_GRAD
    assert orc.rel_l2(xd.grad.cpu(), dx_ref) <= TOL_GRAD
    assert orc.rel_l2(flat, g_ref) <= TOL_GRAD
    with torch.no_grad():  # inference plan: same output
        assert orc.rel_l2(net.eval()(xd).cpu(), y_ref) <= TOL_OUT


def _pattern(name, pattern, nb):
    if pattern == "frozen":
        return False
    if pattern == "head+half":
        return int(name.split(".")[0]) >= nb // 2
    if pattern == "one_conv":
        return not name.startswith(f"{nb - 1}.rdb2.conv3.")
    if pattern == "no_bias":
        return not name.endswith(".bias")
    raise ValueError(pattern)


@pytest.mark.parametrize("pattern", ["frozen", "head+half", "one_conv", "no_bias"])
def test_trunk_freeze_patterns(pattern):
    dev = torch.device("cuda", 0)
    nb = 4
    net = _trunk_module(nb, seed=3).to(dev)
    g = torch.Generator(device="cuda").manual_seed(4)
    x = torch.randn(4, 64, 32, 40, device=dev, generator=g)
    dy = torch.randn(4, 64, 32, 40, device=dev, generator=g)

    def run(train):
        for (name, p), t in zip(net.named_parameters(), train):
            p.requires_grad_(t)
            p.grad = None
        xx = x.clone().requires_grad_(True)
        net(xx).backward(dy)
        return [p.grad for p in net.parameters()], xx.grad

    full, full_dx = run([True] * len(list(net.parameters())))
    train = [_pattern(n, pattern, nb) for n, _ in net.named_parameters()]
    got, dx = run(train)
    for (name, _), t, gp, gf in zip(net.named_parameters(), train, got, full):
        if not t:
            assert gp is None, f"{pattern}: {name} is frozen but got a gradient"
            continue
        assert gp is not None, f"{pattern}: {name} is trainable but got no gradient"
        assert orc.rel_l2(gp, gf) <= TOL_SAME, f"{pattern}: {name}"
    assert torch.equal(dx, full_dx), f"{pattern}: dL/dx differs from the full backward's"


def test_trunk_deterministic_repeats_are_bit_identical():
    dev = torch.device("cuda", 0)
    net = _trunk_module(2, seed=5).to(dev)
    g = torch.Generator(device="cuda").manual_seed(6)
    x = torch.randn(16, 64, 64, 64, device=dev, generator=g)
    dy = torch.randn(16, 64, 64, 64, device=dev, generator=g)
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
def test_trunk_poisoned_workspace_gives_finite_outputs(geo):
    nb, n, h, w = geo
    params = make_params(3, 3, nb, 0, 9, torch.device("cuda", 0))[_trunk_slice(3, nb)[1]]
    trunk = _Raw(nb, n, h, w, True, trunk=True)
    trunk.pack(params)
    g = torch.Generator(device="cuda").manual_seed(10)
    x = torch.randn(n, 64, h, w, device="cuda", generator=g)
    y = trunk.forward(x)
    grads, dx = trunk.backward(torch.randn(n, 64, h, w, device="cuda", generator=g))
    assert bool(torch.isfinite(y).all()) and bool(torch.isfinite(grads).all()) and bool(torch.isfinite(dx).all())
    for name in ["TR", "C1", "C2", "GR", "GC1", "GC2"]:
        assert bool(torch.isfinite(trunk.carrier_nchw(name)).all()), name
    for r in range(3 * nb):
        for name in (f"D{r}", f"DYB{r}"):
            assert bool(torch.isfinite(trunk.region(name, torch.bfloat16).float()).all()), name


class _RDB(nn.Module):
    """ESRGAN / BasicSR dense block with its own forward (the eager copy of the composed model runs it)"""

    def __init__(self):
        super().__init__()
        for k in range(1, 6):
            setattr(self, f"conv{k}", nn.Conv2d(64 + 32 * (k - 1), 32 if k < 5 else 64, 3, 1, 1))
        self.lrelu = nn.LeakyReLU(0.2, True)

    def forward(self, x):
        feats = [x]
        for k in range(1, 5):
            feats.append(self.lrelu(getattr(self, f"conv{k}")(torch.cat(feats, 1))))
        return self.conv5(torch.cat(feats, 1)) * 0.2 + x


class _RRDB(nn.Module):
    def __init__(self):
        super().__init__()
        self.rdb1, self.rdb2, self.rdb3 = _RDB(), _RDB(), _RDB()

    def forward(self, x):
        return self.rdb3(self.rdb2(self.rdb1(x))) * 0.2 + x


class _Toy(nn.Module):
    """a generator that is not one of the reference factories: own head, a bottleneck after the trunk, a x2 pixel-shuffle tail"""

    def __init__(self, nb):
        super().__init__()
        self.head = nn.Conv2d(3, 64, 3, 1, 1)
        self.trunk = nn.Sequential(*[_RRDB() for _ in range(nb)])
        self.bottleneck = nn.Conv2d(64, 64, 1)
        self.up = nn.Sequential(nn.Conv2d(64, 256, 3, 1, 1), nn.PixelShuffle(2), nn.LeakyReLU(0.2), nn.Conv2d(64, 3, 3, 1, 1))

    def forward(self, x):
        f = self.head(x)
        return self.up(f + self.bottleneck(self.trunk(f)))


def test_composed_model_under_autocast_and_gradscaler():
    dev = torch.device("cuda", 0)
    torch.manual_seed(13)
    ref = _Toy(3).to(dev)
    mine = copy.deepcopy(ref)
    mine.trunk = b200.native_trunk(mine.trunk)
    lr = torch.rand(4, 3, 32, 40, device=dev)
    gt = torch.rand(4, 3, 64, 80, device=dev)
    prev = torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32
    torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = False
    try:
        sr_ref = ref(lr)
        loss_ref = nn.functional.mse_loss(sr_ref, gt)
        loss_ref.backward()
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = prev
    opt = torch.optim.SGD(mine.parameters(), lr=0.0)
    scaler = torch.amp.GradScaler("cuda", init_scale=1024.0)
    with torch.autocast("cuda", dtype=torch.float16):
        sr = mine(lr)
        loss = nn.functional.mse_loss(sr.float(), gt)
    scaler.scale(loss).backward()
    scaler.unscale_(opt)
    assert orc.rel_l2(sr.float(), sr_ref) <= TOL_OUT
    got = torch.cat([p.grad.float().flatten() for p in mine.parameters()])
    want = torch.cat([p.grad.flatten() for p in ref.parameters()])
    assert orc.rel_l2(got, want) <= TOL_GRAD
    trunk_got = torch.cat([p.grad.flatten() for p in mine.trunk.parameters()])
    trunk_want = torch.cat([p.grad.flatten() for p in ref.trunk.parameters()])
    assert orc.rel_l2(trunk_got, trunk_want) <= TOL_GRAD
    scaler.step(opt)
    scaler.update()
