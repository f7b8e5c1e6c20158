"""U-Net discriminator, stage by stage against float64, teacher-forced from the tensors the kernels stored in the workspace.

A discriminator plan gives every forward activation and every backward gradient a workspace tensor of its own and reuses none
of them, so after one forward + backward every intermediate a kernel wrote is still there (b200sr_debug_buffer names them).
Each stage is recomputed in float64 from the 16-bit tensors the kernel actually read, with the weights rounded to the plan's
16-bit format as the weight packer rounds them, and compared with the tensor the kernel actually wrote.  What is left is one
rounding of the output plus the fp32 accumulation order, so the per-element bars are
    16-bit outputs: |s - r| <= ulp16(|r|) + gamma * M        fp32 outputs (logits, dx, weight / bias gradients): |s - r| <= gamma * M
where M is the same operation on absolute values (conv of |in| with |W|, sum of |x * dy| for a weight gradient, ...), next to a
bar on the relative L2 error of each tensor.  The end-to-end checks against the fp32 oracle (test_disc.py) have to allow
0.1 - 0.2 relative L2 per gradient; a stage that is wrong by a few percent stands out here by orders of magnitude.

Before the forward the workspace, the logits, the input gradient and the weight gradients are filled with 0xFF bytes (NaN in
fp16, bf16 and fp32): every tensor read back must be finite, so no stage reads an element no stage wrote (the module allocates
its workspace with torch.empty), and the outputs documented as OVERWRITTEN are written in full.

Worst case over every stage and case of this file, measured on one B200 (1000 W power limit), and the bars (BARS):
    fp16 stages:  gamma 2.0e-7 (up_block1, 4 x 256^2), rel-L2 2.3e-4        bars gamma 2^-21 = 4.8e-7, rel-L2 8e-4
    bf16 stages:  gamma 1.5e-7 (up_block1),            rel-L2 1.8e-3        bars gamma 2^-21,          rel-L2 6e-3
    fp32 outputs: gamma 3.0e-7 (up1 weight gradient),  rel-L2 5.0e-6 (conv2 weight gradient)   bars gamma 2^-20 = 9.5e-7, rel-L2 1e-5
(gamma = the smallest per-element gamma the stage passes with; the ingest copies are bit-exact.)  The per-stage table is in
DESIGN.md section 6g; the values of a run are appended to disc_stages.jsonl where test_disc.py records its parity values."""
import ctypes as C

import pytest
import torch
import torch.nn.functional as F

from sr_gan_fd_b200 import lib as _lib
from test_disc import _record

# workspace tensors of a discriminator plan: name -> (lattice level: H >> level, channels, U layout?).  A U-layout tensor of
# level l is stored [N, H >> (l+1), W >> (l+1), 4C] with channel (py*2+px)*C + c; every other one [N, H >> l, W >> l, C].
FWD_LAYOUT = {
    "xin": (0, 64, False), "T0u": (0, 64, True), "T1u": (1, 128, True), "T2u": (2, 256, True), "T3": (3, 512, False),
    "B1": (2, 512, False), "A1": (2, 256, False), "B2": (1, 256, False), "A2": (1, 128, False), "B3": (0, 128, False),
    "A3": (0, 64, False), "S3": (0, 64, False), "A4": (0, 64, False), "A5": (0, 64, False),
}
BWD_LAYOUT = {
    "DYP": (0, 64, False), "G5": (0, 64, False), "G4": (0, 64, False), "GS3": (0, 64, False), "G3": (0, 64, False),
    "GB3": (0, 128, False), "GS2": (1, 128, False), "GA2": (1, 128, False), "GB2": (1, 256, False), "GS1": (2, 256, False),
    "GA1": (2, 256, False), "GB1": (2, 512, False), "GT3": (3, 512, False), "GT2": (2, 256, False), "GT1": (1, 128, False),
    "G0": (0, 64, False),
}
# conv order = parameter order: (name, out channels, in channels, kernel); conv1 and conv4 carry a bias
CONVS = [("conv1", 64, None, 3), ("down1", 128, 64, 4), ("down2", 256, 128, 4), ("down3", 512, 256, 4), ("up1", 256, 512, 3),
         ("up2", 128, 256, 3), ("up3", 64, 128, 3), ("conv2", 64, 64, 3), ("conv3", 64, 64, 3), ("conv4", None, 64, 3)]

# per-element gamma and relative-L2 bars by output format
BARS = {"fp16": (2.0 ** -21, 8e-4), "bf16": (2.0 ** -21, 6e-3), "fp32": (2.0 ** -20, 1e-5)}


def _disc_plan(ci, co, n, h, w, training, fp16=True):
    from sr_gan_fd_b200.discriminator import _DiscPlan
    return _DiscPlan(ci, co, 64, n, h, w, training, fp16)


def _lookup(L, handle, name):
    off, nbytes = C.c_int64(-1), C.c_int64(-1)
    rc = L.b200sr_debug_buffer(handle, name.encode(), C.byref(off), C.byref(nbytes))
    return rc, off.value, nbytes.value


def _layout_bytes(name, n, h, w):
    lvl, c, _ = {**FWD_LAYOUT, **BWD_LAYOUT}[name]
    return n * (h >> lvl) * (w >> lvl) * c * 2


# ------------------------------------------------------------------------------------------------------------ CPU
@pytest.fixture(scope="module")
def L():
    from sr_gan_fd_b200.build import build_native
    build_native()
    return _lib.load()


@pytest.mark.parametrize("geom", [(3, 1, 1, 8, 8), (3, 1, 3, 40, 72), (1, 2, 2, 48, 40), (3, 1, 16, 256, 256), (16, 16, 2, 64, 128)])
@pytest.mark.parametrize("training", [True, False])
def test_debug_buffer_regions_match_the_layout_table(L, geom, training):
    ci, co, n, h, w = geom
    plan = _disc_plan(ci, co, n, h, w, training)
    names = list(FWD_LAYOUT) + (list(BWD_LAYOUT) if training else [])
    regions = []
    for name in names:
        rc, off, nbytes = _lookup(L, plan.handle, name)
        assert rc == 0, (name, L.b200sr_last_error())
        assert nbytes == _layout_bytes(name, n, h, w), name
        assert off >= 0 and off % 16 == 0 and off + nbytes <= plan.workspace_bytes, name
        regions.append((off, nbytes, name))
    regions.sort()
    for (o0, b0, n0), (o1, _, n1) in zip(regions, regions[1:]):
        assert o0 + b0 <= o1, f"{n0} overlaps {n1}"
    if not training:
        for name in BWD_LAYOUT:
            assert _lookup(L, plan.handle, name)[0] == -1, name  # B200SR_ERR_INVALID: an inference plan keeps no gradients


def test_debug_buffer_rejects_unknown_and_foreign_names(L):
    plan = _disc_plan(3, 1, 2, 64, 64, True)
    for name in ("nope", "", "t0u", "G6", "xin "):
        rc, _, _ = _lookup(L, plan.handle, name)
        assert rc == -1 and name.encode() in L.b200sr_last_error(), name
    assert L.b200sr_debug_buffer(None, b"xin", C.byref(C.c_int64()), C.byref(C.c_int64())) == -1
    nd = _lib.NetDesc(3, 3, 64, 32, 2, 2, 2, 32, 32, 1, 0)
    handle = C.c_void_p()
    assert L.b200sr_plan_create(C.byref(nd), C.byref(handle)) == 0
    try:
        # a generator plan names its own tensors (test_gen_stages_gpu.py): the names it shares with the discriminator resolve to the
        # generator's regions, every discriminator-only name is rejected
        for name in set(FWD_LAYOUT) | set(BWD_LAYOUT):
            if name not in ("xin", "DYP", "G3"):
                assert _lookup(L, handle, name)[0] == -1, name
        assert _lookup(L, handle, "xin")[2] == 2 * 32 * 32 * 64 * 2    # conv1 input [hi | lo | hi | 0], 64 channels
        assert _lookup(L, handle, "DYP")[2] == 2 * 128 * 128 * 64 * 2  # x4 output gradient, 64 channels
    finally:
        L.b200sr_plan_destroy(handle)
    vd = _lib.VggDesc(2, 32, 32, 15, 1 << 15, -1, 0, (C.c_float * 3)(0.5, 0.5, 0.5), (C.c_float * 3)(0.25, 0.25, 0.25))
    handle = C.c_void_p()
    assert L.b200sr_vgg_plan_create(C.byref(vd), C.byref(handle)) == 0
    try:
        # a VGG plan names its own tensors (test_vgg_stages_gpu.py): every discriminator-only name is rejected
        for name in set(FWD_LAYOUT) | set(BWD_LAYOUT):
            if name not in ("xin", "A1", "A2", "A3", "A4", "A5"):
                assert _lookup(L, handle, name)[0] == -1, name
        assert _lookup(L, handle, "xin")[2] == 2 * 32 * 32 * 64 * 2  # [hi(3) | lo(3) | hi(3) | 0], 64 channels
    finally:
        L.b200sr_plan_destroy(handle)


# ------------------------------------------------------------------------------------------------------------ GPU helpers
def _from_u(t):
    """[N, h, w, 4C] U layout (channel (py*2+px)*C + c) -> plain [N, C, 2h, 2w] float64"""
    n, h, w, c4 = t.shape
    c = c4 // 4
    return t.reshape(n, h, w, 2, 2, c).permute(0, 5, 1, 3, 2, 4).reshape(n, c, 2 * h, 2 * w).double()


def _nchw(t):
    return t.permute(0, 3, 1, 2).double()


def _ulp16(r, fmt):
    mant, emin = (10, -14) if fmt == "fp16" else (7, -126)
    e = torch.floor(torch.log2(r.abs().clamp_min(2.0 ** emin)))
    return torch.exp2(e - mant)


def _dlrelu(a):
    return torch.where(a > 0, 1.0, 0.2).double()


def _conv(x, w, stride=1):
    return F.conv2d(x, w, stride=stride, padding=1)


def _convT(g, w, stride=1):
    return F.conv_transpose2d(g, w, stride=stride, padding=1)


def _wgrad(x, g, w_shape, stride=1):
    return torch.nn.grad.conv2d_weight(x, w_shape, g, stride=stride, padding=1)


def _up(t):
    return F.interpolate(t, scale_factor=2, mode="bilinear", align_corners=False)


def _up_adjoint(g):
    """transpose of the bilinear x2 upsample (autograd of F.interpolate, float64)"""
    n, c, h, w = g.shape
    z = torch.zeros(n, c, h // 2, w // 2, dtype=torch.float64, device=g.device, requires_grad=True)
    return torch.autograd.grad(_up(z), z, g)[0]


class _Stages:
    """collects every stage's worst normalised error before anything is asserted, so one run reports them all; worst_index is
    (image among the checked ones, channel, y, x) of the NCHW view, or the index into the weight / bias gradient"""
    jsonl = "disc_stages.jsonl"

    def __init__(self, case, fmt):
        self.case, self.fmt, self.rows = case, fmt, []

    def check(self, stage, buf, s, r, m, out_fmt=None):
        out_fmt = out_fmt or self.fmt
        s, r, m = s.double(), r.double(), m.double()
        assert s.shape == r.shape == m.shape, (stage, buf, s.shape, r.shape, m.shape)
        diff = (s - r).abs()
        slack = _ulp16(r, out_fmt) if out_fmt != "fp32" else torch.zeros_like(r)
        need = torch.nan_to_num((diff - slack).clamp_min(0) / m.clamp_min(1e-300), nan=float("inf"))
        flat = int(need.flatten().argmax())
        idx = tuple(int(i) for i in torch.unravel_index(torch.tensor(flat), need.shape))
        gamma, rel_bar = BARS[out_fmt]
        row = {"stage": stage, "buffer": buf, "format": out_fmt, "gamma_needed": float(need.flatten()[flat]),
               "rel_l2": float(torch.nan_to_num((s - r).norm() / r.norm().clamp_min(1e-300), nan=float("inf"))),
               "worst_index": idx, "stored": float(s[idx]), "reference": float(r[idx]), "magnitude": float(m[idx])}
        row["ok"] = row["gamma_needed"] <= gamma and row["rel_l2"] <= rel_bar
        self.rows.append(row)

    def exact(self, stage, buf, s, r):
        """bit-exact 16-bit copy"""
        bad = (s.view(torch.int16) != r.view(torch.int16))
        row = {"stage": stage, "buffer": buf, "format": "bits", "mismatches": int(bad.sum()), "ok": not bool(bad.any())}
        if bad.any():
            idx = tuple(int(i) for i in bad.nonzero()[0])
            row.update(worst_index=idx, stored=float(s[idx]), reference=float(r[idx]))
        self.rows.append(row)

    def finish(self):
        for row in self.rows:
            _record(self.case, row, self.jsonl)
        scored = [r for r in self.rows if "gamma_needed" in r]
        if scored:
            worst = max(scored, key=lambda r: r["gamma_needed"] / BARS[r["format"]][0])
            print(f"{self.case}: worst {worst['stage']} ({worst['buffer']}) gamma {worst['gamma_needed']:.2e}")
        bad = [r for r in self.rows if not r["ok"]]
        assert not bad, "stages outside their bars:\n" + "\n".join(
            f"  {r['stage']} -> {r['buffer']} ({r['format']}): " + ", ".join(f"{k} {v}" for k, v in r.items() if k not in ("stage", "buffer", "format", "ok"))
            for r in bad)


def _r16(t, dt):
    return t.to(dt).double()


def _split16(t, dt):
    """(hi, lo) = (r16(t), r16(t - hi)) with the difference taken in fp32, as the ingest and weight-packing kernels do"""
    t = t.float()
    hi = t.to(dt)
    return hi, (t - hi.float()).to(dt)


def _weights(ci, co, seed, dev):
    from sr_gan_fd_b200.discriminator import DiscriminatorUNet
    torch.manual_seed(seed)
    mine = DiscriminatorUNet(in_channels=ci, out_channels=co, channels=64).to(dev).train()
    ws = [mine.conv1.weight, mine.conv1.bias] + [mine._effective_weight(c) for c in mine._sn_convs()] + [mine.conv4.weight, mine.conv4.bias]
    return [t.detach().float().contiguous() for t in ws]


class _Run:
    """one forward (+ backward) through the raw C ABI on 0xFF-filled buffers"""

    def __init__(self, ci, co, n, h, w, training, fp16, seed=0, x=None):
        self.L = L = _lib.load()
        dev = self.dev = torch.device("cuda", 0)
        self.n, self.h, self.w, self.ci, self.co, self.training = n, h, w, ci, co, training
        self.dt = torch.float16 if (fp16 and ci == 3) else torch.bfloat16   # other input widths run in bf16
        self.plan = _disc_plan(ci, co, n, h, w, training, fp16)
        self.params = _weights(ci, co, seed, dev)
        w1, b1, d1, d2, d3, u1, u2, u3, c2, c3, w4, b4 = self.params
        slots = [w1, b1, d1, None, d2, None, d3, None, u1, None, u2, None, u3, None, c2, None, c3, None, w4, b4]
        self.stream = torch.cuda.current_stream().cuda_stream
        g = torch.Generator(device=dev).manual_seed(seed + 1)
        self.x = torch.rand(n, ci, h, w, device=dev, generator=g) if x is None else x
        self.dy = torch.randn(n, co, h, w, device=dev, generator=g)
        self.ws = torch.full((self.plan.workspace_bytes,), 0xFF, dtype=torch.uint8, device=dev)
        self.pk = torch.zeros(self.plan.packed_bytes, dtype=torch.uint8, device=dev)
        self.y = self._nan(n * co * h * w).view(n, co, h, w)
        ptrs = (C.c_void_p * 20)(*[t.data_ptr() if t is not None else None for t in slots])
        _lib.check(L.b200sr_pack_weights(self.plan.handle, ptrs, C.c_void_p(self.pk.data_ptr()), C.c_void_p(self.stream)))
        strides = (C.c_int64 * 4)(*self.x.stride())
        from sr_gan_fd_b200.discriminator import _DTYPES
        _lib.check(L.b200sr_disc_forward(self.plan.handle, C.c_void_p(self.x.data_ptr()), _DTYPES[self.x.dtype], strides,
                                         C.c_void_p(self.pk.data_ptr()), C.c_void_p(self.ws.data_ptr()), C.c_void_p(self.y.data_ptr()),
                                         C.c_void_p(self.stream)))
        if training:
            self.grads, self.dx = self.backward(True, True)
        torch.cuda.synchronize()

    def _nan(self, numel):
        return torch.full((numel,), -1, dtype=torch.int32, device=self.dev).view(torch.float32)  # 0xFFFFFFFF: NaN

    def backward(self, want_grads, want_dx):
        gb = self._nan(self.plan.param_numel) if want_grads else None
        dxb = self._nan(self.n * self.ci * self.h * self.w).view(self.n, self.ci, self.h, self.w) if want_dx else None
        ptr = lambda t: C.c_void_p(t.data_ptr() if t is not None else None)  # noqa: E731
        _lib.check(self.L.b200sr_disc_backward(self.plan.handle, C.c_void_p(self.dy.data_ptr()), ptr(self.pk), ptr(self.ws), ptr(gb),
                                               ptr(dxb), C.c_void_p(self.stream)))
        torch.cuda.synchronize()
        return gb, dxb

    def buf(self, name):
        """the workspace tensor as the kernels left it: [N, h, w, C] (U layout: [N, h/2, w/2, 4C]) in the plan's 16-bit format"""
        rc, off, nbytes = _lookup(self.L, self.plan.handle, name)
        assert rc == 0, name
        lvl, c, u = {**FWD_LAYOUT, **BWD_LAYOUT}[name]
        h, w = self.h >> (lvl + u), self.w >> (lvl + u)
        return self.ws[off:off + nbytes].view(self.dt).view(self.n, h, w, c * (4 if u else 1))


def _check_ingest(st, run):
    xin = run.buf("xin")
    ci = run.ci
    hi, lo = _split16(run.x.permute(0, 2, 3, 1), run.dt)
    ref = torch.cat([hi, lo, hi, torch.zeros(*hi.shape[:3], 64 - 3 * ci, dtype=run.dt, device=hi.device)], dim=3)
    st.exact("ingest", "xin", xin, ref)


def _param_slices(ci, co):
    """(name, weight shape, flat offset of the weight, flat offset of the bias or None) in flat-gradient order"""
    out, off = [], 0
    for name, o, i, k in CONVS:
        o, i = o or co, i or ci
        shape = (o, i, k, k)
        wo = off
        off += o * i * k * k
        bo = None
        if name in ("conv1", "conv4"):
            bo = off
            off += o
        out.append((name, shape, wo, bo))
    return out, off


# ------------------------------------------------------------------------------------------------------------ GPU
CASES = [  # (n, h, w), in / out channels, requested 16-bit format, training
    pytest.param((1, 8, 8), 3, 1, "fp16", True, id="1x8x8-fp16"),
    pytest.param((2, 64, 64), 3, 1, "fp16", True, id="2x64x64-fp16"),
    pytest.param((2, 64, 64), 3, 1, "bf16", True, id="2x64x64-bf16"),
    pytest.param((3, 40, 72), 3, 1, "fp16", True, id="3x40x72-fp16"),
    pytest.param((2, 128, 96), 3, 1, "fp16", True, id="2x128x96-fp16"),
    pytest.param((4, 256, 256), 3, 1, "fp16", True, id="4x256x256-fp16"),
    pytest.param((2, 48, 40), 1, 2, "fp16", True, id="2x48x40-ci1-co2"),   # other input widths fall back to bf16
    pytest.param((2, 48, 56), 3, 1, "fp16", False, id="2x48x56-fp16-eval"),
]


@pytest.mark.gpu
@pytest.mark.parametrize("shape,ci,co,fmt,training", CASES)
def test_gpu_disc_stages_against_fp64(shape, ci, co, fmt, training):
    n, h, w = shape
    run = _Run(ci, co, n, h, w, training, fmt == "fp16")
    dt, f = run.dt, ("fp16" if run.dt == torch.float16 else "bf16")
    st = _Stages(f"{shape} ci={ci} co={co} {f} training={training}", f)
    names = list(FWD_LAYOUT) + (list(BWD_LAYOUT) if training else [])
    for name in names:
        t = run.buf(name)
        if name == "DYP":
            t = t[..., :16]  # the logit-gradient ingest writes 16 channels; conv4's data / weight / bias gradients read those
        assert bool(torch.isfinite(t).all()), f"workspace tensor {name} holds elements no kernel wrote (or non-finite values)"
    assert bool(torch.isfinite(run.y).all()), "logits not written in full"
    if training:
        assert bool(torch.isfinite(run.grads).all()) and bool(torch.isfinite(run.dx).all()), "gradients not written in full"
    _check_ingest(st, run)

    w1, b1, d1, d2, d3, u1, u2, u3, c2, c3, w4, b4 = run.params
    W = {k: _r16(v, dt) for k, v in zip(("d1", "d2", "d3", "u1", "u2", "u3", "c2", "c3", "w4"), (d1, d2, d3, u1, u2, u3, c2, c3, w4))}
    absW = {k: v.abs() for k, v in W.items()}
    w1h, w1l = (t.double() for t in _split16(w1, dt))
    sel = list(range(n)) if n <= 3 else [0, n - 1]   # per-image stages: the first and the last image of a large batch
    P = lambda name: _nchw(run.buf(name)[sel])   # noqa: E731
    U = lambda name: _from_u(run.buf(name)[sel])  # noqa: E731

    # ---- forward
    xin = P("xin")
    hi, lo = xin[:, :ci], xin[:, ci:2 * ci]
    r = _conv(hi, w1h) + _conv(lo, w1h) + _conv(hi, w1l) + b1.double().view(1, -1, 1, 1)
    m = _conv(hi.abs(), w1h.abs()) + _conv(lo.abs(), w1h.abs()) + _conv(hi.abs(), w1l.abs()) + b1.double().abs().view(1, -1, 1, 1)
    st.check("conv1 (3-product split)", "T0u", U("T0u"), r, m)
    for stage, src, dst, key in (("down1", "T0u", "T1u", "d1"), ("down2", "T1u", "T2u", "d2"), ("down3", "T2u", "T3", "d3")):
        a = U(src)
        out = U(dst) if dst != "T3" else P(dst)
        st.check(f"{stage} (4-tap stride 2)", dst, out, F.leaky_relu(_conv(a, W[key], 2), 0.2), _conv(a.abs(), absW[key], 2))
    for stage, lo_in, skip, dst in (("upsample 1", "T3", None, "B1"), ("upsample 2 + skip", "A1", "T2u", "B2"),
                                    ("upsample 3 + skip", "A2", "T1u", "B3")):
        a = P(lo_in)
        s_ = U(skip) if skip else torch.zeros_like(a)
        st.check(stage, dst, P(dst), _up(a + s_), _up(a.abs() + s_.abs()))
    for stage, src, dst, key in (("up_block1", "B1", "A1", "u1"), ("up_block2", "B2", "A2", "u2"), ("up_block3", "B3", "A3", "u3"),
                                 ("conv2", "S3", "A4", "c2"), ("conv3", "A4", "A5", "c3")):
        a = P(src)
        st.check(stage, dst, P(dst), F.leaky_relu(_conv(a, W[key]), 0.2), _conv(a.abs(), absW[key]))
    st.check("skip add (disc_add_u_kernel)", "S3", P("S3"), P("A3") + U("T0u"), P("A3").abs() + U("T0u").abs())
    a5 = P("A5")
    st.check("conv4 (fp32 logits)", "y", run.y[sel].double(), _conv(a5, W["w4"]) + b4.double().view(1, -1, 1, 1),
             _conv(a5.abs(), absW["w4"]) + b4.double().abs().view(1, -1, 1, 1), out_fmt="fp32")

    if training:
        # ---- data gradients
        dyp = run.buf("DYP")
        st.exact("logit-gradient ingest", "DYP", dyp[..., :co], run.dy.permute(0, 2, 3, 1).to(dt))
        st.exact("logit-gradient ingest (zero channels)", "DYP", dyp[..., co:16], torch.zeros_like(dyp[..., co:16]))
        g = P("DYP")[:, :co]
        for stage, src, dst, key, mask in (("conv4 dgrad", None, "G5", "w4", "A5"), ("conv3 dgrad", "G5", "G4", "c3", "A4"),
                                           ("conv2 dgrad", "G4", "GS3", "c2", None), ("up_block3 dgrad", "G3", "GB3", "u3", None),
                                           ("up_block2 dgrad", "GA2", "GB2", "u2", None), ("up_block1 dgrad", "GA1", "GB1", "u1", None)):
            gi = g if src is None else P(src)
            d = _dlrelu(P(mask)) if mask else 1.0
            st.check(stage, dst, P(dst), _convT(gi, W[key]) * d, _convT(gi.abs(), absW[key]) * d)
        st.check("LeakyReLU mask (disc_lrelu_mask_kernel)", "G3", P("G3"), P("GS3") * _dlrelu(P("A3")), P("GS3").abs())
        for stage, src, gs, ga, act in (("bilinear transpose 3", "GB3", "GS2", "GA2", "A2"), ("bilinear transpose 2", "GB2", "GS1", "GA1", "A1"),
                                        ("bilinear transpose 1", "GB1", None, "GT3", "T3")):
            gi = P(src)
            r, m = _up_adjoint(gi), _up_adjoint(gi.abs())
            if gs:
                st.check(stage, gs, P(gs), r, m)
            d = _dlrelu(P(act))
            st.check(stage + " x LeakyReLU'", ga, P(ga), r * d, m * d)
        for stage, src, skip, dst, key, mask in (("down3 dgrad (shuffle + skip + mask)", "GT3", "GS1", "GT2", "d3", "T2u"),
                                                 ("down2 dgrad (shuffle + skip + mask)", "GT2", "GS2", "GT1", "d2", "T1u"),
                                                 ("down1 dgrad (shuffle + skip)", "GT1", "GS3", "G0", "d1", None)):
            gi, sk = P(src), P(skip)
            d = _dlrelu(U(mask)) if mask else 1.0
            st.check(stage, dst, P(dst), (_convT(gi, W[key], 2) + sk) * d, (_convT(gi.abs(), absW[key], 2) + sk.abs()) * d)
        w1r = _r16(w1, dt)
        g0 = P("G0")
        st.check("conv1 dgrad (fp32 dx)", "dx", run.dx[sel].double(), _convT(g0, w1r), _convT(g0.abs(), w1r.abs()), out_fmt="fp32")

        # ---- weight and bias gradients: the whole batch
        A = lambda name: _nchw(run.buf(name))  # noqa: E731
        AU = lambda name: _from_u(run.buf(name))  # noqa: E731
        pairs = {"conv1": (A("xin")[:, :ci], A("G0"), 1), "down1": (AU("T0u"), A("GT1"), 2), "down2": (AU("T1u"), A("GT2"), 2),
                 "down3": (AU("T2u"), A("GT3"), 2), "up1": (A("B1"), A("GA1"), 1), "up2": (A("B2"), A("GA2"), 1),
                 "up3": (A("B3"), A("G3"), 1), "conv2": (A("S3"), A("G4"), 1), "conv3": (A("A4"), A("G5"), 1),
                 "conv4": (A("A5"), A("DYP")[:, :co], 1)}
        slices, total = _param_slices(ci, co)
        assert total == run.plan.param_numel
        grads = run.grads.double()
        for name, shape, wo, bo in slices:
            x_, g_, stride = pairs[name]
            numel = shape[0] * shape[1] * shape[2] * shape[3]
            st.check(f"{name} weight gradient", "flat_grads", grads[wo:wo + numel].view(shape), _wgrad(x_, g_, shape, stride),
                     _wgrad(x_.abs(), g_.abs(), shape, stride), out_fmt="fp32")
            if bo is not None:
                st.check(f"{name} bias gradient", "flat_grads", grads[bo:bo + shape[0]], g_.sum(dim=(0, 2, 3)), g_.abs().sum(dim=(0, 2, 3)),
                         out_fmt="fp32")

        # ---- the two partial backwards against the full one (the workspace is rewritten with the same values)
        _, dx_only = run.backward(False, True)
        assert torch.equal(dx_only, run.dx), "frozen-discriminator backward (no weight gradients) changed dx"
        grads_only, _ = run.backward(True, False)
        assert bool(torch.isfinite(grads_only).all())
        for name, shape, wo, bo in slices:
            x_, g_, stride = pairs[name]
            numel = shape[0] * shape[1] * shape[2] * shape[3]
            m = _wgrad(x_.abs(), g_.abs(), shape, stride).flatten()
            diff = (grads_only[wo:wo + numel].double() - grads[wo:wo + numel]).abs()
            assert bool((diff <= 2 * BARS["fp32"][0] * m).all()), f"{name}: weight gradients without dx differ beyond atomic ordering"
    st.finish()


@pytest.mark.gpu
@pytest.mark.parametrize("x_dtype", [torch.float32, torch.float16, torch.bfloat16])
@pytest.mark.parametrize("channels_last", [False, True])
@pytest.mark.parametrize("ci,fmt", [(3, "fp16"), (3, "bf16"), (1, "bf16")])
def test_gpu_disc_ingest_bit_exact(x_dtype, channels_last, ci, fmt):
    """x -> [hi | lo | hi | 0] in the plan's 16-bit format, for every input dtype and memory layout (RGB: the vectorised kernel,
    other widths: the generic one)"""
    dev = torch.device("cuda", 0)
    g = torch.Generator(device=dev).manual_seed(7)
    x = torch.rand(2, ci, 16, 24, device=dev, generator=g).to(x_dtype)
    if channels_last:
        x = x.contiguous(memory_format=torch.channels_last)
    run = _Run(ci, 1, 2, 16, 24, False, fmt == "fp16", x=x)
    st = _Stages(f"ingest {x_dtype} channels_last={channels_last} ci={ci} {fmt}", fmt)
    _check_ingest(st, run)
    st.finish()
