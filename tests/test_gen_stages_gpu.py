"""RRDBNet generator, stage by stage against float64, teacher-forced from the tensors the kernels stored in the workspace.

A training plan keeps every dense block's activation buffer D{r} and output-gradient buffer DYB{r}, the tail activations and
gradients, and the fp32 carriers the residual epilogues read and write (b200sr_debug_buffer names them).  After one forward and
one backward almost every intermediate a kernel wrote is still there, so each stage is recomputed in float64 from the 16-bit
tensors the kernel actually read, with the weights rounded exactly as pack_weights_kernel rounds them, and compared with what
the kernel stored.  The per-element bar is the one of test_disc_stages_gpu.py:
    |s - r| <= slack + gamma * M        M = the same operation on absolute values
slack = ulp16(|r|) for a 16-bit store, ulp16 of the lo part for a [hi | lo] bf16 pair, 0 for fp32 outputs; where a residual can
only be rebuilt from its bf16 shadow (the carrier was overwritten later), one ulp16 of that shadow times its scale is added.
Next to it each tensor has a relative-L2 bar.  The end-to-end checks against the fp32 oracle (test_model_gpu.py) allow 5e-3 on
the SR output and 1e-2 / 5e-2 on the gradients; a conv that is wrong by a percent or a residual scale of 0.21 stands out here.

Before the forward the workspace, y, the flat gradients and dx are filled with 0xFF bytes (NaN in bf16, fp16 and fp32): every
named tensor, read over its valid pixels and channels, must come back finite, and so must the outputs documented as OVERWRITTEN.

fp32 carriers use the tile-blocked layout of the conv epilogues ([tile][half][16-byte chunk][pixel in half][4 floats] over
8 x 32-pixel tiles, see carrier_base); the upsample convs run as four phase convs on the low-res lattice with the 3x3 kernel
folded per phase (fold_up), pixel-shuffled on store with channel ((y & 1) * 2 + (x & 1)) * 64 + c.

Bars (BARS below, gamma / rel-L2): bf16 2^-21 / 6e-3, fp16 2^-21 / 8e-4, fp32 2^-20 / 1e-5, "split" (a [hi | lo] bf16 pair,
about 16 significant bits) 2^-19 / 1e-5 and "wgrad" (fp32 weight / bias gradients) 2^-20 / 5e-5.  The measured worst values per stage are in DESIGN.md section 6j; every run appends its
rows to gen_stages.jsonl next to disc_stages.jsonl."""
import contextlib
import ctypes as C
import os

import pytest
import torch
import torch.nn.functional as F

from sr_gan_fd_b200 import lib as _lib
from test_disc import _record
from test_disc_stages_gpu import _ulp16

# gamma / rel-L2 per output format.  "split" ([hi | lo] bf16 pair) needs gamma 1.34e-6 (conv3, 1 x 3 x 160 x 264 at x4): K = 3 x 576
# products in one fp32 tensor-core accumulator; "wgrad" (fp32 weight / bias gradients, sums over up to 675 k pixels whose signs
# cancel, so |result| << M) needs rel-L2 2.5e-5 (conv3 weight gradient, same case), gamma 6.3e-7 (config 2)
BARS = {"fp16": (2.0 ** -21, 8e-4), "bf16": (2.0 ** -21, 6e-3), "fp32": (2.0 ** -20, 1e-5), "split": (2.0 ** -19, 1e-5),
        "wgrad": (2.0 ** -20, 5e-5)}
TILE_W, TILE_H = 8, 32          # conv work item (kTileW x kTileH)
CARRIER_TILE_BYTES = 65536      # kCarrierBytesPerTile


# ------------------------------------------------------------------------------------------------------------ helpers
def unblock(t, n, h, w):
    """tile-blocked fp32 carrier (flat) -> [N, H, W, 64]: tile = (n * tiles_y + ty) * tiles_x + tx, y = 32 ty + 16 half + m / 8,
    x = 8 tx + m % 8, c = 4 chunk + lane (add_carriers_to_bf16_kernel); padded pixels are dropped"""
    ty, tx = -(-h // TILE_H), -(-w // TILE_W)
    t = t[:n * ty * tx * CARRIER_TILE_BYTES // 4].view(n, ty, tx, 2, 16, 16, 8, 4)   # n ty tx half chunk my mx lane
    t = t.permute(0, 1, 3, 5, 2, 6, 4, 7).reshape(n, ty * TILE_H, tx * TILE_W, 64)
    return t[:, :h, :w]


def shuffle(t):
    """[N, 4C, h, w] with channel ((a * 2) + b) * C + c -> [N, C, 2h, 2w], pixel (2y + a, 2x + b)"""
    n, c4, h, w = t.shape
    c = c4 // 4
    return t.view(n, 2, 2, c, h, w).permute(0, 3, 4, 1, 5, 2).reshape(n, c, 2 * h, 2 * w)


def unshuffle(t):
    n, c, h2, w2 = t.shape
    return t.view(n, c, h2 // 2, 2, w2 // 2, 2).permute(0, 3, 5, 1, 2, 4).reshape(n, 4 * c, h2 // 2, w2 // 2)


# original 3x3 taps d that fold onto low-res tap t for output phase a (up_phase_taps)
_UP_TAPS = {0: [[0], [1, 2], []], 1: [[], [0, 1], [2]]}


def fold_up(w):
    """[64, 64, 3, 3] -> [256, 64, 3, 3], row phase * 64 + co (kPackUpFwd): the four phase kernels of nearest-x2 + conv on the
    low-res lattice, summed in w's dtype from 0, dy outer, dx inner, as pack_fetch sums them"""
    co = w.shape[0]
    out = torch.zeros(4 * co, *w.shape[1:], dtype=w.dtype, device=w.device)
    for ph in range(4):
        a, b = ph >> 1, ph & 1
        for ty in range(3):
            for tx in range(3):
                acc = torch.zeros(w.shape[:2], dtype=w.dtype, device=w.device)
                for dy in _UP_TAPS[a][ty]:
                    for dx in _UP_TAPS[b][tx]:
                        acc = acc + w[:, :, dy, dx]
                out[ph * co:(ph + 1) * co, :, ty, tx] = acc
    return out


def _conv(x, w):
    return F.conv2d(x, w, padding=1)


def _convT(g, w):
    return F.conv_transpose2d(g, w, padding=1)


def _wgrad(x, g, shape):
    return torch.nn.grad.conv2d_weight(x, shape, g, padding=1)


def _dlrelu(a):
    return torch.where(a > 0, 1.0, 0.2).double()


def _lrelu(v):
    return F.leaky_relu(v, 0.2)


def _nchw(t):
    return t.permute(0, 3, 1, 2).double()


def _split(t, dt=torch.bfloat16):
    """(hi, lo) of an fp32 tensor, the difference taken in fp32 (ingest / pack / split-store epilogues)"""
    t = t.float()
    hi = t.to(dt)
    return hi, (t - hi.float()).to(dt)


def _f32_scale(t, s):
    """fp32 product with the fp32 constant s, as the epilogue forms delta * v"""
    return t.float() * torch.tensor(s, dtype=torch.float32, device=t.device)


# ------------------------------------------------------------------------------------------------------------ names / sizes
def expected_regions(in_ch, out_ch, num_blocks, n_up, n, h, w, training, tail_f16=None):
    """name -> bytes of every workspace tensor a generator plan names"""
    tail_f16 = (not training) if tail_f16 is None else tail_f16
    R, L = 3 * num_blocks, n_up
    P = n * h * w
    carrier = n * (-(-w // TILE_W)) * (-(-h // TILE_H)) * CARRIER_TILE_BYTES
    ts = 64 if (tail_f16 and not training) else 128
    xs = -(-3 * in_ch // 64) * 64
    out = {"xin": P * xs * 2, "T0": carrier, "TR": carrier, "C1": carrier, "C2": carrier}
    for r in range(R if training else 2):
        out[f"D{r}"] = P * 192 * 2
    out["SPLT"] = P * ts * 2
    for lvl in range(L + 1):
        out[f"SPL{lvl}"] = (P << (2 * lvl)) * ts * 2
    out["SPLC"] = (P << (2 * L)) * ts * 2
    if training:
        hr = P << (2 * L)
        out.update(CMASK=hr * out_ch, DYP=hr * 128, G3=hr * 128)
        for lvl in range(1, L + 1):
            out[f"GU{lvl}"] = (P << (2 * (lvl - 1))) * 256 * 2
        out.update(GT=carrier, GTB=P * 128, GR=carrier, GC1=carrier, GC2=carrier, GO1=P * 128)
        for r in range(R):
            out[f"DYB{r}"] = P * 192 * 2
    return out


def _lookup(L, handle, name):
    off, nbytes = C.c_int64(-1), C.c_int64(-1)
    rc = L.b200sr_debug_buffer(handle, name.encode(), C.byref(off), C.byref(nbytes))
    return rc, off.value, nbytes.value


@contextlib.contextmanager
def _env(**kv):
    """plan-creation switches (read in b200sr_plan_create)"""
    old = {k: os.environ.get(k) for k in kv}
    os.environ.update({k: str(v) for k, v in kv.items()})
    try:
        yield
    finally:
        for k, v in old.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v


class _Plan:
    def __init__(self, in_ch, out_ch, num_blocks, n_up, n, h, w, training, env=None):
        self.L = _lib.load()
        nd = _lib.NetDesc(in_ch, out_ch, 64, 32, num_blocks, n_up, n, h, w, 1 if training else 0, 0)
        self.handle = C.c_void_p()
        with _env(**(env or {})):
            _lib.check(self.L.b200sr_plan_create(C.byref(nd), C.byref(self.handle)))
        self.workspace_bytes = int(self.L.b200sr_workspace_bytes(self.handle))
        self.packed_bytes = int(self.L.b200sr_packed_bytes(self.handle))
        self.param_numel = int(self.L.b200sr_param_numel(self.handle))

    def region(self, name):
        rc, off, nbytes = _lookup(self.L, self.handle, name)
        assert rc == 0, (name, self.L.b200sr_last_error())
        return off, nbytes

    def __del__(self):
        if getattr(self, "handle", None):
            self.L.b200sr_plan_destroy(self.handle)


# ------------------------------------------------------------------------------------------------------------ CPU
@pytest.fixture(scope="module")
def L():
    from sr_gan_fd_b200.build import build_native
    build_native()
    return _lib.load()


GEOMS = [  # in_ch, num_blocks, n, h, w
    pytest.param((3, 1, 1, 16, 8), id="3ch-1x16x8"),
    pytest.param((12, 2, 3, 33, 9), id="12ch-3x33x9"),
    pytest.param((48, 23, 16, 64, 64), id="48ch-23rrdb-16x64x64"),
    pytest.param((3, 1, 1, 160, 264), id="3ch-1x160x264-per-conv"),
]


@pytest.mark.parametrize("geom", GEOMS)
@pytest.mark.parametrize("n_up", [0, 1, 2, 3])
@pytest.mark.parametrize("training", [True, False])
def test_gen_debug_buffer_regions(L, geom, n_up, training):
    in_ch, nb, n, h, w = geom
    plan = _Plan(in_ch, 3, nb, n_up, n, h, w, training)
    want = expected_regions(in_ch, 3, nb, n_up, n, h, w, training)
    regions = []
    for name, nbytes in want.items():
        off, got = plan.region(name)
        assert got == nbytes, (name, got, nbytes)
        assert off >= 0 and off % 16 == 0 and off + got <= plan.workspace_bytes, name
        regions.append((off, got, name))
    regions.sort()
    for (o0, b0, n0), (o1, _, n1) in zip(regions, regions[1:]):
        assert o0 + b0 <= o1, f"{n0} overlaps {n1}"
    R = 3 * nb
    rejected = ["nope", "", "d0", "xin ", f"D{R}", "D69", "GU0", f"SPL{n_up + 1}", f"GU{n_up + 1}", "GW", "T0u"]
    if not training:
        rejected += ["D2", "CMASK", "DYP", "G3", "GU1", "GT", "GTB", "GR", "GC1", "GC2", "GO1", "DYB0"]
    for name in rejected:
        rc, _, _ = _lookup(L, plan.handle, name)
        assert rc == -1 and name.encode() in L.b200sr_last_error(), name


def test_gen_debug_buffer_tail_fp16_training(L):
    """B200SR_TAIL_FP16=1 in a training plan keeps the 128-channel tail buffers (fp16 | bf16 twin)"""
    plan = _Plan(3, 3, 1, 2, 2, 16, 8, True, env={"B200SR_TAIL_FP16": 1})
    for name, nbytes in expected_regions(3, 3, 1, 2, 2, 16, 8, True, tail_f16=True).items():
        assert plan.region(name)[1] == nbytes, name
    plan = _Plan(3, 3, 1, 2, 2, 16, 8, False, env={"B200SR_TAIL_FP16": 0})
    assert plan.region("SPLT")[1] == 2 * 16 * 8 * 128 * 2  # split-precision inference tail: [hi | lo]


def test_fold_up_is_nearest_upsample_then_conv():
    g = torch.Generator().manual_seed(3)
    w = torch.randn(64, 64, 3, 3, generator=g, dtype=torch.float64)
    x = torch.randn(2, 64, 5, 7, generator=g, dtype=torch.float64)
    ref = _conv(F.interpolate(x, scale_factor=2, mode="nearest"), w)
    got = shuffle(_conv(x, fold_up(w)))
    assert torch.allclose(got, ref, rtol=1e-12, atol=1e-12)
    assert torch.equal(unshuffle(shuffle(x.repeat(1, 4, 1, 1))), x.repeat(1, 4, 1, 1))
    # each original tap lands on exactly one low-res tap per phase
    ones = fold_up(torch.ones(1, 1, 3, 3, dtype=torch.float64))
    assert ones.view(4, 9).sum(1).tolist() == [9.0] * 4


def test_unblock_matches_carrier_base():
    n, h, w = 2, 40, 13
    ty, tx = -(-h // TILE_H), -(-w // TILE_W)
    flat = torch.full((n * ty * tx * CARRIER_TILE_BYTES // 4,), -1.0, dtype=torch.float64)
    for b in range(n):
        for y in range(h):
            for x in range(w):
                tile = (b * ty + y // TILE_H) * tx + x // TILE_W
                half, m = (y % TILE_H) // 16, (y % 16) * 8 + x % TILE_W
                base = ((tile * 2 + half) * 16 * 128 + m) * 4      # carrier_base(tile, half, m)
                for c in range(64):
                    flat[base + (c >> 2) * 512 + (c & 3)] = ((b * h + y) * w + x) * 64 + c
    got = unblock(flat, n, h, w)
    assert torch.equal(got, torch.arange(n * h * w * 64, dtype=torch.float64).view(n, h, w, 64))


# ------------------------------------------------------------------------------------------------------------ GPU
class _Stages:
    """every stage's worst normalised error is collected before anything is asserted (test_disc_stages_gpu._Stages, with an
    extra slack for residuals rebuilt from bf16 shadows); worst_index is the index into the NCHW view or the gradient tensor"""

    def __init__(self, case):
        self.case, self.rows = case, []

    def check(self, stage, buf, s, r, m, fmt, extra=None, slack=None):
        s, r, m = s.double(), r.double(), m.double()
        assert s.shape == r.shape == m.shape, (stage, buf, s.shape, r.shape, m.shape)
        diff = (s - r).abs()
        if slack is None:
            slack = _ulp16(r, fmt) if fmt in ("bf16", "fp16") else torch.zeros_like(r)
        if extra is not None:
            slack = slack + extra
        need = torch.nan_to_num((diff - slack).clamp_min(0) / m.clamp_min(1e-300), nan=float("inf"))
        flat = int(need.flatten().argmax())
        idx = tuple(int(i) for i in torch.unravel_index(torch.tensor(flat), need.shape))
        gamma, rel_bar = BARS[fmt]
        row = {"stage": stage, "buffer": buf, "format": fmt, "gamma_needed": float(need.flatten()[flat]),
               "rel_l2": float(torch.nan_to_num((s - r).norm() / r.norm().clamp_min(1e-300), nan=float("inf"))),
               "worst_index": idx, "stored": float(s[idx]), "reference": float(r[idx]), "magnitude": float(m[idx])}
        if extra is not None:   # the shadow's own bf16 rounding sits in the difference: the tensor's rel-L2 bar is the bf16 one
            rel_bar = BARS["bf16"][1]
        row["ok"] = row["gamma_needed"] <= gamma and row["rel_l2"] <= rel_bar
        self.rows.append(row)

    def exact(self, stage, buf, s, r):
        bits = torch.int16 if s.element_size() == 2 else (torch.int32 if s.element_size() == 4 else torch.uint8)
        bad = (s.contiguous().view(bits) != r.contiguous().view(bits))
        row = {"stage": stage, "buffer": buf, "format": "bits", "mismatches": int(bad.sum()), "ok": not bool(bad.any())}
        if bad.any():
            idx = tuple(int(i) for i in bad.nonzero()[0])
            row.update(worst_index=idx, stored=float(s[idx]), reference=float(r[idx]))
        self.rows.append(row)

    def truth(self, stage, buf, ok, **info):
        self.rows.append({"stage": stage, "buffer": buf, "format": "logic", "ok": bool(ok), **info})

    def finish(self):
        for row in self.rows:
            _record(self.case, row, "gen_stages.jsonl")
        scored = [r for r in self.rows if "gamma_needed" in r]
        if scored:
            worst = max(scored, key=lambda r: r["gamma_needed"] / BARS[r["format"]][0])
            print(f"{self.case}: {len(self.rows)} checks, worst {worst['stage']} ({worst['buffer']}) gamma {worst['gamma_needed']:.2e}")
        bad = [r for r in self.rows if not r["ok"]]
        assert not bad, "stages outside their bars:\n" + "\n".join(
            f"  {r['stage']} -> {r['buffer']} ({r['format']}): " + ", ".join(f"{k} {v}" for k, v in r.items() if k not in ("stage", "buffer", "format", "ok"))
            for r in bad[:40])


def make_params(in_ch, out_ch, num_blocks, n_up, seed, dev):
    """state_dict-order fp32 weights and biases: Kaiming-scaled head / tail, 0.2x trunk, small random biases, conv4 bias 0.5 (so the
    clamp cuts on both sides)"""
    g = torch.Generator().manual_seed(seed)
    dims = [(64, in_ch)]
    for _ in range(3 * num_blocks):
        dims += [(32, 64), (32, 96), (32, 128), (32, 160), (64, 192)]
    dims += [(64, 64)] * (1 + n_up + 1) + [(out_ch, 64)]
    out = []
    ntrunk = 1 + 15 * num_blocks
    for i, (o, c) in enumerate(dims):
        scale = 0.2 if 1 <= i < ntrunk else 1.0
        wt = torch.randn(o, c, 3, 3, generator=g) * (2.0 / (9 * c)) ** 0.5 * scale
        b = torch.randn(o, generator=g) * 0.05
        if i == len(dims) - 1:
            b = b + 0.5
        out += [wt.to(dev).contiguous(), b.to(dev).contiguous()]
    return out


class _Run:
    """one forward + backward through the raw C ABI on 0xFF-filled buffers"""

    def __init__(self, in_ch, out_ch, num_blocks, n_up, n, h, w, training=True, env=None, seed=0, x=None):
        dev = self.dev = torch.device("cuda", 0)
        self.in_ch, self.out_ch, self.nb, self.L, self.n, self.h, self.w = in_ch, out_ch, num_blocks, n_up, n, h, w
        self.R, self.training = 3 * num_blocks, training
        env = env or {}
        self.tail_f16 = bool(int(env["B200SR_TAIL_FP16"])) if "B200SR_TAIL_FP16" in env else not training
        self.ts = 64 if (self.tail_f16 and not training) else 128
        self.plan = _Plan(in_ch, out_ch, num_blocks, n_up, n, h, w, training, env)
        self.lib = self.plan.L
        self.params = make_params(in_ch, out_ch, num_blocks, n_up, seed, dev)
        self.stream = torch.cuda.current_stream().cuda_stream
        g = torch.Generator(device=dev).manual_seed(seed + 1)
        self.x = torch.rand(n, in_ch, h, w, device=dev, generator=g) if x is None else x
        s = 1 << n_up
        self.dy = torch.randn(n, out_ch, s * h, s * w, device=dev, generator=g)
        self.ws = torch.full((self.plan.workspace_bytes,), 0xFF, dtype=torch.uint8, device=dev)
        self.pk = torch.zeros(self.plan.packed_bytes, dtype=torch.uint8, device=dev)
        self.y = self._nan(n * out_ch * s * h * s * w).view(n, out_ch, s * h, s * w)
        ptrs = (C.c_void_p * len(self.params))(*[t.data_ptr() for t in self.params])
        _lib.check(self.lib.b200sr_pack_weights(self.plan.handle, ptrs, C.c_void_p(self.pk.data_ptr()), C.c_void_p(self.stream)))
        dt = {torch.float32: _lib.F32, torch.float16: _lib.F16, torch.bfloat16: _lib.BF16}[self.x.dtype]
        strides = (C.c_int64 * 4)(*self.x.stride())
        _lib.check(self.lib.b200sr_forward(self.plan.handle, C.c_void_p(self.x.data_ptr()), dt, strides, C.c_void_p(self.pk.data_ptr()),
                                           C.c_void_p(self.ws.data_ptr()), C.c_void_p(self.y.data_ptr()), C.c_void_p(self.stream)))
        if training:
            self.grads, self.dx = self.backward(True)
        torch.cuda.synchronize()

    def _nan(self, numel):
        return torch.full((numel,), -1, dtype=torch.int32, device=self.dev).view(torch.float32)

    def backward(self, want_dx):
        gb = self._nan(self.plan.param_numel)
        dxb = self._nan(self.n * self.in_ch * self.h * self.w).view(self.n, self.in_ch, self.h, self.w) if want_dx else None
        _lib.check(self.lib.b200sr_backward(self.plan.handle, C.c_void_p(self.dy.data_ptr()), C.c_void_p(self.pk.data_ptr()),
                                            C.c_void_p(self.ws.data_ptr()), C.c_void_p(gb.data_ptr()),
                                            C.c_void_p(dxb.data_ptr()) if want_dx else None, _lib.BUCKET_CB(), None,
                                            C.c_void_p(self.stream)))
        torch.cuda.synchronize()
        return gb, dxb

    def raw(self, name, dtype):
        off, nbytes = self.plan.region(name)
        return self.ws[off:off + nbytes].view(dtype)

    def pix(self, name, c, level=0, dtype=torch.bfloat16):
        """[N, h, w, c] NHWC view of a workspace tensor on the lattice of upsample level `level`"""
        return self.raw(name, dtype).view(self.n, self.h << level, self.w << level, c)

    def carrier(self, name):
        return unblock(self.raw(name, torch.float32), self.n, self.h, self.w)


def _fin(t):
    return bool(torch.isfinite(t.float()).all())


def _finite_checks(st, run):
    n_up, R = run.L, run.R
    tdt = torch.float16 if run.tail_f16 else torch.bfloat16
    xs = run.plan.region("xin")[1] // (run.n * run.h * run.w * 2)
    names = {"xin": run.pix("xin", xs)}
    for c in ("T0", "TR", "C1", "C2"):
        names[c] = run.carrier(c)
    for r in range(R if run.training else 2):
        names[f"D{r}"] = run.pix(f"D{r}", 192)
    names["SPLT"] = run.pix("SPLT", run.ts, 0, tdt)
    for lvl in range(n_up + 1):
        names[f"SPL{lvl}"] = run.pix(f"SPL{lvl}", run.ts, lvl, tdt)
    names["SPLC"] = run.pix("SPLC", run.ts, n_up, tdt)
    if run.tail_f16 and run.training:   # channels [64, 128): the bf16 twin of the fp16 value
        for k in [k for k in names if k.startswith("SP")]:
            names[k + " twin"] = names[k][..., 64:].view(torch.bfloat16)
            names[k] = names[k][..., :64]
    if run.training:
        names["DYP"] = run.pix("DYP", 64, n_up)[..., :16]   # the gradient ingest writes 16 channels; every reader reads those
        names["G3"] = run.pix("G3", 64, n_up)
        for lvl in range(1, n_up + 1):
            names[f"GU{lvl}"] = run.pix(f"GU{lvl}", 256, lvl - 1)
        for c in ("GT", "GR", "GC1", "GC2"):
            names[c] = run.carrier(c)
        names["GTB"], names["GO1"] = run.pix("GTB", 64), run.pix("GO1", 64)
        for r in range(R):
            names[f"DYB{r}"] = run.pix(f"DYB{r}", 192)
    bad = [k for k, t in names.items() if not _fin(t)]
    st.truth("every named tensor finite (no element left unwritten)", ",".join(bad) or "all", not bad)
    st.truth("y finite", "y", _fin(run.y))
    if run.training:
        st.truth("flat gradients finite", "flat_grads", _fin(run.grads))
        st.truth("dx finite", "dx", _fin(run.dx))


def check_ingest(st, run):
    xs = run.plan.region("xin")[1] // (run.n * run.h * run.w * 2)
    hi, lo = _split(run.x.permute(0, 2, 3, 1))
    c = run.in_ch
    ref = torch.cat([hi, lo, hi, torch.zeros(run.n, run.h, run.w, xs - 3 * c, dtype=torch.bfloat16, device=hi.device)], dim=3)
    st.exact("ingest", "xin", run.pix("xin", xs), ref)


class _Weights:
    """the packed weights, rebuilt in float64 the way pack_weights_kernel rounds them"""

    def __init__(self, run):
        p = run.params
        self.R, self.L = run.R, run.L
        self.ntrunk = 1 + 5 * self.R
        bf = lambda t: t.to(torch.bfloat16).double()  # noqa: E731
        self.w1h, self.w1l = (t.double() for t in _split(p[0]))
        self.b = [p[2 * i + 1].double() for i in range(len(p) // 2)]
        self.W = [bf(p[2 * i]) for i in range(len(p) // 2)]            # bf16(w): trunk and every dgrad pack
        self.tail = {}
        for i in range(self.ntrunk, len(p) // 2):
            w = p[2 * i]
            is_up = self.ntrunk + 1 <= i <= self.ntrunk + self.L
            f = fold_up(w) if is_up else w                                # fp32 fold, rounded after
            if run.tail_f16:
                self.tail[i] = [f.to(torch.float16).double()]
            else:
                hi, lo = _split(f)
                self.tail[i] = [hi.double(), lo.double()]
            if is_up:
                self.W[i] = f.to(torch.bfloat16).double()                 # up-dgrad: bf16 of the fold

    def rdb(self, r, k):
        return 1 + 5 * r + (k - 1)


def _tail_conv(run, Wt, idx, a, a_lo):
    """forward of one tail conv on the 16-bit operands: split form hi*Wh + lo*Wh + hi*Wl, or one fp16 product"""
    ws = Wt.tail[idx]
    if run.tail_f16:
        return _conv(a, ws[0]), _conv(a.abs(), ws[0].abs())
    r = _conv(a, ws[0]) + _conv(a_lo, ws[0]) + _conv(a, ws[1])
    m = _conv(a.abs(), ws[0].abs()) + _conv(a_lo.abs(), ws[0].abs()) + _conv(a.abs(), ws[1].abs())
    return r, m


def _tail_check(st, run, stage, name, buf, r, m, lvl):
    """a tail activation store: [hi | lo] bf16 pair, or fp16 (+ bf16 twin in training)"""
    if run.tail_f16:
        s = _nchw(buf[..., :64])
        st.check(stage, name, s, r, m, "fp16")
        if run.training:
            twin = _nchw(buf[..., 64:128].view(torch.bfloat16))
            # one bf16 ulp of the fp16 value (plus the fp16 subnormal spacing, which is coarser than bf16's below 2^-14)
            st.check(stage + " (bf16 twin)", name, twin, s, torch.zeros_like(s), "bf16", slack=_ulp16(s, "bf16") + _ulp16(s, "fp16"))
    else:
        hi, lo = _nchw(buf[..., :64]), _nchw(buf[..., 64:128])
        st.check(stage, name, hi + lo, r, m, "split", slack=_ulp16(lo, "bf16"))


def _tail_operand(run, name, lvl, sel):
    """(fwd operand, lo operand or None, weight-gradient operand) of a tail activation buffer, NCHW float64"""
    tdt = torch.float16 if run.tail_f16 else torch.bfloat16
    t = run.pix(name, run.ts, lvl, tdt)[sel]
    if run.tail_f16:
        twin = run.pix(name, run.ts, lvl, torch.bfloat16)[sel][..., 64:128] if run.training else None
        return _nchw(t[..., :64]), None, (_nchw(twin) if twin is not None else None)
    return _nchw(t[..., :64]), _nchw(t[..., 64:128]), _nchw(t[..., :64])


def check_forward(st, run, Wt, sel, blocks):
    R, nb = run.R, run.nb
    bias = lambda i: Wt.b[i].view(1, -1, 1, 1)  # noqa: E731
    xs = run.plan.region("xin")[1] // (run.n * run.h * run.w * 2)
    xin = _nchw(run.pix("xin", xs)[sel])
    c = run.in_ch
    hi, lo = xin[:, :c], xin[:, c:2 * c]
    r = _conv(hi, Wt.w1h) + _conv(lo, Wt.w1h) + _conv(hi, Wt.w1l) + bias(0)
    m = _conv(hi.abs(), Wt.w1h.abs()) + _conv(lo.abs(), Wt.w1h.abs()) + _conv(hi.abs(), Wt.w1l.abs()) + bias(0).abs()
    T0 = run.carrier("T0")[sel]
    st.check("conv1 (3-product split)", "T0", _nchw(T0), r, m, "fp32")
    if run.training:
        st.exact("conv1 bf16 shadow", "D0[:64]", run.pix("D0", 64 * 3)[sel][..., :64], T0.to(torch.bfloat16))
    D = {}
    for r_ in blocks:
        D[r_] = run.pix(f"D{r_ if run.training else r_ & 1}", 192)[sel]
    car = {k: _nchw(run.carrier(k)[sel]) for k in ("T0", "TR", "C1", "C2")}
    for r_ in blocks:
        d = _nchw(D[r_])
        for k in range(1, 5):
            cin = 64 + 32 * (k - 1)
            i = Wt.rdb(r_, k)
            a = d[:, :cin]
            pre = _conv(a, Wt.W[i]) + bias(i)
            st.check(f"dense conv{k}", f"D{r_}[{cin}:{cin + 32}]", d[:, cin:cin + 32], _lrelu(pre),
                     _conv(a.abs(), Wt.W[i].abs()) + bias(i).abs(), "bf16")
    # conv5 + residual epilogue: v = alpha (acc + b) + beta1 r1 + beta2 r2
    last_b = nb - 1
    for r_ in blocks:
        j, b = r_ % 3, r_ // 3
        i = Wt.rdb(r_, 5)
        d = _nchw(D[r_])
        acc = _conv(d, Wt.W[i]) + bias(i)
        macc = _conv(d.abs(), Wt.W[i].abs()) + bias(i).abs()
        alpha = 0.04 if j == 2 else 0.2

        def shadow(rr):  # bf16 shadow of the block-rr input carrier, None where the plan no longer has it
            if rr in D:
                return _nchw(D[rr][..., :64])
            return None
        terms = []   # (scale, value, exact?)
        if j == 0:
            terms.append((1.0, car["T0"] if b == 0 else shadow(r_), b == 0))
        elif j == 1:
            terms.append((1.0, car["C1"] if b == last_b else shadow(r_), b == last_b))
        else:
            terms.append((0.2, car["C2"] if b == last_b else shadow(r_), b == last_b))
            terms.append((1.0, car["T0"] if b == 0 else shadow(r_ - 2), b == 0))
        if any(t[1] is None for t in terms):
            continue
        ref = alpha * acc + sum(s * v for s, v, _ in terms)
        mag = alpha * macc + sum(s * v.abs() for s, v, _ in terms)
        extra = sum(s * _ulp16(v, "bf16") for s, v, ex in terms if not ex)
        all_exact = all(ex for _, _, ex in terms)
        out_c = ("C1", "C2", "TR")[j]
        survives = b == last_b
        if survives and all_exact:
            st.check(f"conv5 + residual (j={j}, fp32 carrier)", f"{out_c} (block {r_})", car[out_c], ref, mag, "fp32")
        if r_ < R - 1:
            s16 = _nchw(D[r_ + 1][..., :64]) if (r_ + 1) in D else None
            if s16 is not None:
                st.check(f"conv5 + residual (j={j}, bf16 shadow)", f"D{r_ + 1}[:64]", s16, ref, mag, "bf16",
                         extra=None if all_exact else extra)
                if survives:
                    st.exact(f"conv5 shadow == bf16(carrier) (j={j})", f"D{r_ + 1}[:64]", D[r_ + 1][..., :64],
                             run.carrier(out_c)[sel].to(torch.bfloat16))
        else:
            s = _tail_operand(run, "SPLT", 0, sel)
            st.check(f"conv5 + residual (j={j}, tail input)", "SPLT", s[0] + (s[1] if s[1] is not None else 0), ref, mag,
                     "fp16" if run.tail_f16 else "split", extra=None if all_exact else extra,
                     slack=_ulp16(ref, "fp16") if run.tail_f16 else _ulp16(s[1], "bf16"))
    # tail input == 16-bit copy of the final trunk carrier, bit for bit
    tr = run.carrier("TR")[sel]
    splt = run.pix("SPLT", run.ts, 0, torch.float16 if run.tail_f16 else torch.bfloat16)[sel]
    if run.tail_f16:
        st.exact("SPLT == fp16(TR)", "SPLT", splt[..., :64], tr.to(torch.float16))
        if run.training:
            st.exact("SPLT twin == bf16(TR)", "SPLT[64:]", splt[..., 64:].view(torch.bfloat16), tr.to(torch.bfloat16))
    else:
        h_, l_ = _split(tr)
        st.exact("SPLT == [bf16(TR) | bf16(TR - bf16(TR))]", "SPLT", splt, torch.cat([h_, l_], -1))
    # tail convs
    ic2 = Wt.ntrunk
    a, alo, _ = _tail_operand(run, "SPLT", 0, sel)
    r, m = _tail_conv(run, Wt, ic2, a, alo)
    r, m = r + bias(ic2) + car["T0"], m + bias(ic2).abs() + car["T0"].abs()
    _tail_check(st, run, "conv2 + long skip", "SPL0", run.pix("SPL0", run.ts, 0, torch.float16 if run.tail_f16 else torch.bfloat16)[sel], r, m, 0)
    tdt = torch.float16 if run.tail_f16 else torch.bfloat16
    for lvl in range(1, run.L + 1):
        iu = ic2 + lvl
        a, alo, _ = _tail_operand(run, f"SPL{lvl - 1}", lvl - 1, sel)
        r, m = _tail_conv(run, Wt, iu, a, alo)
        b4 = Wt.b[iu].repeat(4).view(1, -1, 1, 1)
        r, m = shuffle(_lrelu(r + b4)), shuffle(m + b4.abs())
        _tail_check(st, run, f"upsample {lvl} (phase form, shuffled)", f"SPL{lvl}", run.pix(f"SPL{lvl}", run.ts, lvl, tdt)[sel], r, m, lvl)
    ic3 = ic2 + run.L + 1
    a, alo, _ = _tail_operand(run, f"SPL{run.L}", run.L, sel)
    r, m = _tail_conv(run, Wt, ic3, a, alo)
    _tail_check(st, run, "conv3", "SPLC", run.pix("SPLC", run.ts, run.L, tdt)[sel], _lrelu(r + bias(ic3)), m + bias(ic3).abs(), run.L)
    ic4 = ic3 + 1
    a, alo, _ = _tail_operand(run, "SPLC", run.L, sel)
    r, m = _tail_conv(run, Wt, ic4, a, alo)
    pre, mag = r + bias(ic4), m + bias(ic4).abs()
    y = run.y[sel].double()
    bar = BARS["fp32"][0] * mag
    inside = (pre > bar) & (pre < 1 - bar)
    st.check("conv4 (fp32, unclamped elements)", "y", torch.where(inside, y, pre), pre, mag, "fp32")
    st.truth("conv4 clamp", "y", bool(((pre <= -bar) <= (y == 0)).all() and ((pre >= 1 + bar) <= (y == 1)).all()),
             inside=int(inside.sum()), total=int(pre.numel()))
    if run.training:
        cm = run.raw("CMASK", torch.uint8).view(run.n, run.out_ch, run.h << run.L, run.w << run.L)[sel]
        clear = ((pre.abs() > bar) & ((pre - 1).abs() > bar))
        ok_ref = bool((((cm == 1) == ((pre >= 0) & (pre <= 1))) | ~clear).all())
        ok_y = bool(((cm == 1) | (y == 0) | (y == 1)).all() and (((y > 0) & (y < 1)) <= (cm == 1)).all())
        st.truth("CMASK against the fp64 pre-activation", "CMASK", ok_ref)
        st.truth("CMASK consistent with y", "CMASK", ok_y)
    return car


def check_backward(st, run, Wt, sel):
    R, nb, L = run.R, run.nb, run.L
    dyp = run.pix("DYP", 64, L)
    cm = run.raw("CMASK", torch.uint8).view(run.n, run.out_ch, run.h << L, run.w << L)
    st.exact("output-gradient ingest", "DYP", dyp[..., :run.out_ch],
             torch.where(cm == 1, run.dy, torch.zeros_like(run.dy)).permute(0, 2, 3, 1).to(torch.bfloat16))
    st.exact("output-gradient ingest (zero channels)", "DYP", dyp[..., run.out_ch:16], torch.zeros_like(dyp[..., run.out_ch:16]))
    ic2 = Wt.ntrunk
    ic3, ic4 = ic2 + L + 1, ic2 + L + 2
    tdt = torch.float16 if run.tail_f16 else torch.bfloat16
    mask = lambda name, lvl: _dlrelu(_nchw(run.pix(name, run.ts, lvl, tdt)[sel][..., :64]))  # noqa: E731
    g = _nchw(dyp[sel][..., :run.out_ch])
    st.check("conv4 dgrad x lrelu'(SPLC)", "G3", _nchw(run.pix("G3", 64, L)[sel]), _convT(g, Wt.W[ic4]) * mask("SPLC", L),
             _convT(g.abs(), Wt.W[ic4].abs()), "bf16")
    g = _nchw(run.pix("G3", 64, L)[sel])
    gt = run.carrier("GT")[sel]
    if L >= 1:
        st.check("conv3 dgrad x lrelu'(SPL{L}), unshuffled", f"GU{L}", _nchw(run.pix(f"GU{L}", 256, L - 1)[sel]),
                 unshuffle(_convT(g, Wt.W[ic3]) * mask(f"SPL{L}", L)), unshuffle(_convT(g.abs(), Wt.W[ic3].abs())), "bf16")
    else:
        st.check("conv3 dgrad (fp32)", "GT", _nchw(gt), _convT(g, Wt.W[ic3]), _convT(g.abs(), Wt.W[ic3].abs()), "fp32")
    for lvl in range(L, 0, -1):
        iu = ic2 + lvl
        g = _nchw(run.pix(f"GU{lvl}", 256, lvl - 1)[sel])
        r, m = _convT(g, Wt.W[iu]), _convT(g.abs(), Wt.W[iu].abs())
        if lvl >= 2:
            d = mask(f"SPL{lvl - 1}", lvl - 1)
            st.check(f"upsample {lvl} dgrad x lrelu'(SPL{lvl - 1}), unshuffled", f"GU{lvl - 1}",
                     _nchw(run.pix(f"GU{lvl - 1}", 256, lvl - 2)[sel]), unshuffle(r * d), unshuffle(m), "bf16")
        else:
            st.check("upsample 1 dgrad (fp32)", "GT", _nchw(gt), r, m, "fp32")
    st.exact("GTB == bf16(GT)", "GTB", run.pix("GTB", 64)[sel], gt.to(torch.bfloat16))
    # conv2 dgrad: g_trunk = convT(GTB, W2) is the gradient at the trunk output, exact up to gamma (GR is overwritten later)
    gtb = _nchw(run.pix("GTB", 64)[sel])
    g_trunk, m_trunk = _convT(gtb, Wt.W[ic2]), _convT(gtb.abs(), Wt.W[ic2].abs())
    DYB = {r_: _nchw(run.pix(f"DYB{r_}", 192)[sel]) for r_ in range(R)}
    st.check("conv2 dgrad x 0.04", f"DYB{R - 1}[:64]", DYB[R - 1][:, :64], 0.04 * g_trunk, 0.04 * m_trunk, "bf16")
    # dense blocks, last first
    offs = {5: 0, 4: 64, 3: 96, 2: 128, 1: 160}
    car = {k: _nchw(run.carrier(k)[sel]) for k in ("GR", "GC1", "GC2")}
    for r_ in range(R - 1, -1, -1):
        j, b = r_ % 3, r_ // 3
        d, dyb = _nchw(run.pix(f"D{r_}", 192)[sel]), DYB[r_]
        gD = torch.zeros_like(d)
        mD = torch.zeros_like(d)
        for k in range(5, 0, -1):
            i = Wt.rdb(r_, k)
            cin = 64 + 32 * (k - 1)
            gk = dyb[:, offs[k]:offs[k] + (64 if k == 5 else 32)]
            gD[:, :cin] += _convT(gk, Wt.W[i])
            mD[:, :cin] += _convT(gk.abs(), Wt.W[i].abs())
            if k > 1:  # gD of slice o_{k-1} is complete once conv k's contribution is in
                sl = k - 1
                cs = 64 + 32 * (sl - 1)
                st.check(f"dense dgrad slice o{sl} x lrelu'", f"DYB{r_}[{offs[sl]}:{offs[sl] + 32}]", dyb[:, offs[sl]:offs[sl] + 32],
                         gD[:, cs:cs + 32] * _dlrelu(d[:, cs:cs + 32]), mD[:, cs:cs + 32], "bf16")
        gx, mx = gD[:, :64], mD[:, :64]
        # block-input epilogue (xslice_epilogue)
        gr_in = (g_trunk, m_trunk, True) if b == nb - 1 else (DYB[3 * b + 2][:, :64] / 0.04, None, False)
        if j == 2:
            terms, delta, out_c = [(0.2, gr_in)], 0.2, "GC2"
        elif j == 1:
            terms, delta, out_c = [(1.0, (car["GC2"], car["GC2"].abs(), True) if b == 0 else (DYB[3 * b + 1][:, :64] / 0.2, None, False))], 0.2, "GC1"
        else:
            terms = [(1.0, (car["GC1"], car["GC1"].abs(), True) if b == 0 else (DYB[3 * b][:, :64] / 0.2, None, False)), (1.0, gr_in)]
            delta, out_c = 0.04, "GR"
        ref = gx + sum(s * t[0] for s, t in terms)
        mag = mx + sum(s * (t[1] if t[1] is not None else t[0].abs()) for s, t in terms)
        all_exact = all(t[2] for _, t in terms)
        # shadow slack: a residual rebuilt as stored / delta' carries ulp16(stored) / delta'
        extra = None
        if not all_exact:
            extra = torch.zeros_like(ref)
            for s, t in terms:
                if not t[2]:
                    scale = 0.04 if t is gr_in else 0.2
                    extra = extra + s * _ulp16(t[0] * scale, "bf16") / scale
        if b == 0 and all_exact:
            st.check(f"block-input gradient (j={j}, fp32 carrier)", f"{out_c} (block {r_})", car[out_c], ref, mag, "fp32")
        if r_ > 0:
            st.check(f"block-input gradient x {delta} (j={j})", f"DYB{r_ - 1}[:64]", DYB[r_ - 1][:, :64], delta * ref, delta * mag,
                     "bf16", extra=None if extra is None else delta * extra)
            if b == 0:
                st.exact(f"block-input gradient shadow == bf16({delta} carrier) (j={j})", f"DYB{r_ - 1}[:64]",
                         run.pix(f"DYB{r_ - 1}", 192)[sel][..., :64], _f32_scale(run.carrier(out_c)[sel], delta).to(torch.bfloat16))
    go1 = (run.carrier("GR") + run.carrier("GT")).to(torch.bfloat16)
    st.exact("GO1 == bf16(GR + GT)", "GO1", run.pix("GO1", 64), go1)
    g = _nchw(run.pix("GO1", 64)[sel])
    w1 = Wt.W[0]
    st.check("conv1 dgrad (fp32 dx)", "dx", run.dx[sel].double(), _convT(g, w1), _convT(g.abs(), w1.abs()), "fp32")


def param_slices(run):
    """(conv index, weight shape, flat weight offset, flat bias offset) in state_dict order"""
    out, off = [], 0
    for i in range(len(run.params) // 2):
        shape = tuple(run.params[2 * i].shape)
        numel = shape[0] * shape[1] * 9
        out.append((i, shape, off, off + numel))
        off += numel + shape[0]
    return out, off


def check_weight_grads(st, run, Wt):
    """every weight and bias gradient over the whole batch, from the operands the weight-gradient kernels read; returns the
    slices and {conv: (weight M, bias M)} for the repeated-backward check"""
    L, R = run.L, run.R
    ic2 = Wt.ntrunk
    xs = run.plan.region("xin")[1] // (run.n * run.h * run.w * 2)
    allp = slice(None)
    offs = {5: 0, 4: 64, 3: 96, 2: 128, 1: 160}

    def operands():  # (conv index, stage name, X, dY), one dense block at a time
        yield 0, "conv1", _nchw(run.pix("xin", xs))[:, :run.in_ch], _nchw(run.pix("GO1", 64))   # the kernel flushes the hi rows only
        for r_ in range(R):
            d, dyb = _nchw(run.pix(f"D{r_}", 192)), _nchw(run.pix(f"DYB{r_}", 192))
            for k in range(1, 6):
                yield Wt.rdb(r_, k), f"dense conv{k}", d[:, :64 + 32 * (k - 1)], dyb[:, offs[k]:offs[k] + (64 if k == 5 else 32)]
        yield ic2, "conv2", _tail_operand(run, "SPLT", 0, allp)[2], _nchw(run.pix("GTB", 64))
        for lvl in range(1, L + 1):
            a = _tail_operand(run, f"SPL{lvl - 1}", lvl - 1, allp)[2]
            yield (ic2 + lvl, f"upsample {lvl}", F.interpolate(a, scale_factor=2, mode="nearest"),
                   shuffle(_nchw(run.pix(f"GU{lvl}", 256, lvl - 1))))
        yield ic2 + L + 1, "conv3", _tail_operand(run, f"SPL{L}", L, allp)[2], _nchw(run.pix("G3", 64, L))
        yield ic2 + L + 2, "conv4", _tail_operand(run, "SPLC", L, allp)[2], _nchw(run.pix("DYP", 64, L))[:, :run.out_ch]

    slices, total = param_slices(run)
    assert total == run.plan.param_numel
    grads = run.grads.double()
    mags = {}
    for i, name, x_, g_ in operands():
        _, shape, wo, bo = slices[i]
        numel = shape[0] * shape[1] * 9
        m, mb = _wgrad(x_.abs(), g_.abs(), shape), g_.abs().sum(dim=(0, 2, 3))
        where = f"flat_grads[conv {i}]"
        st.check(f"{name} weight gradient", where, grads[wo:wo + numel].view(shape), _wgrad(x_, g_, shape), m, "wgrad")
        st.check(f"{name} bias gradient", where, grads[bo:bo + shape[0]], g_.sum(dim=(0, 2, 3)), mb, "wgrad")
        mags[i] = (m.flatten(), mb)
    return slices, mags


# (in_ch, out_ch, num_blocks, n_up, (n, h, w), training, env, images checked per stage (None: all))
CASES = [
    pytest.param(3, 3, 1, 2, (1, 16, 8), True, {}, None, id="1rrdb-x4-1x16x8"),
    pytest.param(3, 3, 1, 2, (3, 33, 9), True, {}, None, id="1rrdb-x4-3x33x9"),
    pytest.param(3, 3, 2, 2, (1, 20, 12), True, {}, None, id="2rrdb-x4-1x20x12"),
    pytest.param(3, 3, 1, 0, (2, 24, 16), True, {}, None, id="1rrdb-x1-2x24x16"),
    pytest.param(3, 3, 1, 1, (2, 20, 12), True, {}, None, id="1rrdb-x2-2x20x12"),
    pytest.param(3, 3, 1, 3, (1, 12, 8), True, {}, None, id="1rrdb-x8-1x12x8"),
    pytest.param(12, 3, 1, 2, (2, 16, 24), True, {}, None, id="real-x2-12ch"),
    pytest.param(48, 3, 1, 2, (1, 16, 16), True, {}, None, id="real-x1-48ch"),
    pytest.param(1, 1, 1, 2, (2, 16, 8), True, {}, None, id="1ch-in-1ch-out"),
    pytest.param(3, 3, 2, 2, (1, 20, 12), True, {"B200SR_REASSOC": 0}, None, id="2rrdb-per-conv-schedule"),
    pytest.param(3, 3, 1, 2, (1, 160, 264), True, {}, None, id="1rrdb-x4-1x160x264-per-conv"),
    pytest.param(3, 3, 1, 2, (2, 16, 16), True, {"B200SR_TAIL_FP16": 1}, None, id="1rrdb-fp16-tail-training"),
    pytest.param(3, 3, 2, 2, (2, 40, 24), False, {}, None, id="2rrdb-inference-2x40x24"),
    pytest.param(3, 3, 23, 2, (16, 64, 64), True, {}, [0, 15], id="config2-23rrdb-16x64x64"),
]


@pytest.mark.gpu
@pytest.mark.parametrize("in_ch,out_ch,nb,n_up,shape,training,env,sel", CASES)
def test_gpu_gen_stages_against_fp64(in_ch, out_ch, nb, n_up, shape, training, env, sel):
    n, h, w = shape
    run = _Run(in_ch, out_ch, nb, n_up, n, h, w, training, env)
    st = _Stages(f"gen {in_ch}->{out_ch} rrdb={nb} n_up={n_up} {shape} training={training} {env}")
    _finite_checks(st, run)
    check_ingest(st, run)
    Wt = _Weights(run)
    sel = list(range(n)) if sel is None else sel
    blocks = list(range(run.R)) if training else [run.R - 2, run.R - 1]
    check_forward(st, run, Wt, sel, blocks)
    if training:
        check_backward(st, run, Wt, sel)
        slices, mags = check_weight_grads(st, run, Wt)
        # a second backward without dx: the same gradients up to the order of the fp32 atomics; a third with dx: the same dx
        grads0, dx0 = run.grads.clone(), run.dx.clone()
        g1, _ = run.backward(False)
        st.truth("backward without dx: gradients finite", "flat_grads", _fin(g1))
        worst = 0.0
        for i, shape_, wo, bo in slices:
            numel = shape_[0] * shape_[1] * 9
            mw, mb = mags[i]
            for a, b_, m in ((g1[wo:wo + numel], grads0[wo:wo + numel], mw), (g1[bo:bo + shape_[0]], grads0[bo:bo + shape_[0]], mb)):
                excess = ((a.double() - b_.double()).abs() - 2 * BARS["fp32"][0] * m).max()
                worst = max(worst, float(excess))
        st.truth("backward without dx == first backward (2 gamma M)", "flat_grads", worst <= 0.0, worst_excess=worst)
        _, dx2 = run.backward(True)
        st.truth("third backward: dx bit-identical", "dx", torch.equal(dx2.view(torch.int32), dx0.view(torch.int32)))
    st.finish()


@pytest.mark.gpu
@pytest.mark.parametrize("x_dtype", [torch.float32, torch.float16, torch.bfloat16])
@pytest.mark.parametrize("channels_last", [False, True])
@pytest.mark.parametrize("in_ch", [3, 12, 48])
def test_gpu_gen_ingest_bit_exact(x_dtype, channels_last, in_ch):
    """x -> [hi | lo | hi | 0] bf16, for every input dtype, memory layout and the three conv1 widths (48: xin_stride 192)"""
    dev = torch.device("cuda", 0)
    g = torch.Generator(device=dev).manual_seed(11)
    x = torch.rand(2, in_ch, 16, 24, device=dev, generator=g).to(x_dtype)
    if channels_last:
        x = x.contiguous(memory_format=torch.channels_last)
    run = _Run(in_ch, 3, 1, 0, 2, 16, 24, False, x=x)
    st = _Stages(f"gen ingest {x_dtype} channels_last={channels_last} in_ch={in_ch}")
    check_ingest(st, run)
    st.finish()
