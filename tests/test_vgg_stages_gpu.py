"""VGG19 feature path, stage by stage against float64, teacher-forced from the tensors the kernels stored in the workspace.

A VGG plan keeps every conv's post-ReLU activation A{l}, every max-pool P{l}, the fp32 feature nodes F{l} and, with a gradient
request, the gradient G{l} w.r.t. every conv's pre-activation output and GP{l} on each pooled lattice (b200sr_debug_buffer names
them; the table is in include/b200sr.h).  After one forward, the L1 sums and one backward every intermediate a kernel wrote is
still there, so each stage is recomputed in float64 from the 16-bit tensors the kernel actually read, with the weights rounded as
pack_weights_kernel rounds them (conv 0 [w_hi | w_hi | w_lo] against the [hi | lo | hi] input, every other conv and every dgrad
bf16(w)), and compared with what the kernel stored.  The per-element bar is the one of test_disc_stages_gpu.py:
    bf16 outputs: |s - r| <= ulp16(|r|) + gamma * M        fp32 outputs (features, dx): |s - r| <= gamma * M
where M is the same operation on absolute values, next to a bar on the relative L2 error of each tensor.  The copies are bit-exact:
the ingest, the max-pools, the L1 gradient and the pool backward.  The L1 sums must match the fp64 sum over the stored features
within 2^-23 relative.  The end-to-end checks against fp32 (test_vgg.py) allow 1 % on the loss and up to 0.33 relative L2 on the
16-conv-deep input gradient; a dropped ReLU mask, a wrong tie rule or a bias off by 1 % stands out here.

The weights are plain seeded tensors (He-normal, small random biases); no torchvision network is built.  Before the forward the
workspace and dx are filled with 0xFF bytes (NaN in bf16 and fp32): every named tensor must come back finite, so no stage reads an
element no stage wrote, and dx must be written in full.

Worst case over every stage and case of this file, measured on one B200 (1000 W power limit), and the bars (BARS of
test_disc_stages_gpu.py, whose convs reach the same K = 4608; all VGG stages fit them, so none was changed):
    bf16 stages:  gamma 2.0e-7 (conv 8 dgrad onto the pooled lattice GP7, 16 x 256^2), rel-L2 1.8e-3    bars 2^-21 = 4.8e-7, 6e-3
    fp32 outputs: gamma 6.7e-7 (feature F11 after the ReLU, 3 x 48 x 80), rel-L2 3.6e-6 (F15)        bars 2^-20 = 9.5e-7, 1e-5
    L1 sums:      2.3e-10 relative                                                                   bar  2^-23 = 1.2e-7
The per-stage table is in DESIGN.md section 6f; the values of a run are appended to vgg_stages.jsonl next to disc_stages.jsonl."""
import ctypes as C
import re

import pytest
import torch
import torch.nn.functional as F

from sr_gan_fd_b200 import lib as _lib
from test_disc_stages_gpu import _Stages as _DiscStages
from test_disc_stages_gpu import _lookup

COUT = [64, 64, 128, 128, 256, 256, 256, 256, 512, 512, 512, 512, 512, 512, 512, 512]
CIN = [3] + COUT[:-1]
POOL_AFTER = {1, 3, 7, 11}
MEAN, STD = (0.485, 0.456, 0.406), (0.229, 0.224, 0.225)
L1_REL_BAR = 2.0 ** -23


def _lattices(h, w, last):
    """(h_l, w_l) of conv 0 .. last: floor-halved after every pool"""
    out = []
    for l in range(last + 1):
        out.append((h, w))
        if l in POOL_AFTER:
            h, w = h // 2, w // 2
    return out


def _expected_names(n, h, w, last, feats, gc, nb):
    """name -> bytes of every tensor a plan of this geometry names (the table in include/b200sr.h)"""
    out = {"xin": n * h * w * 64 * 2}
    bwd = gc >= 0 and nb > 0
    for l, (hl, wl) in enumerate(_lattices(h, w, last)):
        c = COUT[l]
        out[f"A{l}"] = n * hl * wl * c * 2
        if l in feats:
            out[f"F{l}"] = n * hl * wl * c * 4
        if l in POOL_AFTER and l < last:
            out[f"P{l}"] = n * (hl // 2) * (wl // 2) * c * 2
        if bwd and l <= gc:
            out[f"G{l}"] = nb * hl * wl * c * 2
            if l in POOL_AFTER and l < gc:
                out[f"GP{l}"] = nb * (hl // 2) * (wl // 2) * c * 2
    return out


def _desc(n, h, w, last, feats, gc, nb, det):
    mask = sum(1 << l for l in feats)
    return _lib.VggDesc(n, h, w, last, mask, gc, nb, (C.c_float * 3)(*MEAN), (C.c_float * 3)(*STD), 1 if det else 0)


class _Plan:
    def __init__(self, L, n, h, w, last, feats, gc, nb, det=False):
        self.L, self.handle = L, C.c_void_p()
        _lib.check(L.b200sr_vgg_plan_create(C.byref(_desc(n, h, w, last, feats, gc, nb, det)), C.byref(self.handle)))
        self.workspace_bytes = int(L.b200sr_workspace_bytes(self.handle))
        self.packed_bytes = int(L.b200sr_packed_bytes(self.handle))

    def close(self):
        if self.handle:
            self.L.b200sr_plan_destroy(self.handle)
            self.handle = None


# ------------------------------------------------------------------------------------------------------------ CPU
@pytest.fixture(scope="module")
def L():
    from sr_gan_fd_b200.build import build_native
    build_native()
    return _lib.load()


PLAN_GEOMS = [  # images (sr + gt), H, W, last_conv, feature nodes, grad_conv, deterministic
    (4, 33, 47, 15, {15}, 15, False),            # odd sizes at every pool
    (2, 16, 16, 15, {15}, 15, True),             # the smallest input conv5_4 accepts: 1 x 1 at the last four convs
    (2, 24, 40, 0, {0}, 0, False),               # conv1_1 alone
    (4, 40, 56, 7, {7}, 7, True),                # features.16
    (6, 48, 80, 15, {1, 3, 7, 11, 15}, -1, False),  # the five BSRGAN nodes, inference
    (4, 32, 32, 3, {1, 3}, 1, False),            # gradient of a node before the last conv
    (2, 64, 96, 11, {5, 11}, 5, True),
    (2, 20, 28, 9, {2, 9}, -1, True),
]


@pytest.mark.parametrize("geom", PLAN_GEOMS)
def test_vgg_debug_buffer_regions_match_the_layout_table(L, geom):
    n, h, w, last, feats, gc, det = geom
    nb = n // 2 if gc >= 0 else 0
    plan = _Plan(L, n, h, w, last, feats, gc, nb, det)
    try:
        expected = _expected_names(n, h, w, last, feats, gc, nb)
        regions = []
        for name, size in expected.items():
            rc, off, nbytes = _lookup(L, plan.handle, name)
            assert rc == 0, (name, L.b200sr_last_error())
            assert nbytes == size, (name, nbytes, size)
            assert off >= 0 and off % 16 == 0 and off + nbytes <= plan.workspace_bytes, name
            regions.append((off, nbytes, name))
        regions.sort()
        for (o0, b0, n0), (o1, _, n1) in zip(regions, regions[1:]):
            assert o0 + b0 <= o1, f"{n0} overlaps {n1}"
        # every other name of the family is rejected: convs past last_conv / grad_conv, absent nodes and pools
        for l in range(17):
            for name in (f"A{l}", f"F{l}", f"P{l}", f"G{l}", f"GP{l}"):
                if name not in expected:
                    rc, _, _ = _lookup(L, plan.handle, name)
                    assert rc == -1 and name.encode() in L.b200sr_last_error(), name
        for name in ("a0", "G-1", "A", "xin0", "F"):
            assert _lookup(L, plan.handle, name)[0] == -1, name
    finally:
        plan.close()


@pytest.mark.parametrize("gc,nb", [(-1, 0), (7, 0)])
def test_vgg_inference_plans_name_no_gradients(L, gc, nb):
    plan = _Plan(L, 4, 32, 48, 7, {3, 7}, gc, nb)
    try:
        for l in range(16):
            assert _lookup(L, plan.handle, f"G{l}")[0] == -1 and _lookup(L, plan.handle, f"GP{l}")[0] == -1, l
        assert _lookup(L, plan.handle, "A7")[0] == 0 and _lookup(L, plan.handle, "P3")[0] == 0
    finally:
        plan.close()


@pytest.mark.parametrize("h,w,last,bad_conv", [(15, 16, 15, 12), (16, 15, 12, 12), (8, 8, 12, 12), (7, 64, 8, 8), (1, 1, 2, 2),
                                               (3, 40, 4, 4)])
def test_vgg_plan_rejects_an_input_too_small_naming_the_conv(L, h, w, last, bad_conv):
    handle = C.c_void_p()
    assert L.b200sr_vgg_plan_create(C.byref(_desc(2, h, w, last, {last}, -1, 0, False)), C.byref(handle)) == -1
    assert f"conv {bad_conv}".encode() in L.b200sr_last_error()
    # one conv earlier fits
    plan = _Plan(L, 2, h, w, bad_conv - 1, {bad_conv - 1}, bad_conv - 1, 1)
    plan.close()


# ------------------------------------------------------------------------------------------------------------ GPU helpers
class _Stages(_DiscStages):
    jsonl = "vgg_stages.jsonl"

    def rel(self, stage, buf, s, r, bar):
        err = abs(s - r) / max(abs(r), 1e-300)
        self.rows.append({"stage": stage, "buffer": buf, "format": "sum", "rel_err": err, "stored": s, "reference": r, "ok": err <= bar})

    def truth(self, stage, buf, ok, **info):
        self.rows.append({"stage": stage, "buffer": buf, "format": "logic", "ok": bool(ok), **info})


def _nchw(t):
    return t.permute(0, 3, 1, 2).double()


def _conv(x, w):
    return F.conv2d(x, w, padding=1)


def _convT(g, w):
    return F.conv_transpose2d(g, w, padding=1)


def _bias(b):
    return b.double().view(1, -1, 1, 1)


def _weights(last, seed, dev):
    """He-normal OIHW weights and small random biases, fp32, in pack order (conv l weight at 2l, bias at 2l + 1)"""
    g = torch.Generator().manual_seed(seed)
    out = []
    for l in range(last + 1):
        out.append((torch.randn(COUT[l], CIN[l], 3, 3, generator=g) * (2.0 / (9 * CIN[l])) ** 0.5).to(dev))
        out.append((0.1 * torch.randn(COUT[l], generator=g)).to(dev))
    return out


def _pair_images(pairs, h, w, seed, dev):
    g = torch.Generator().manual_seed(seed)
    gt = torch.rand(pairs, 3, h, w, generator=g)
    sr = (gt + 0.1 * torch.randn(pairs, 3, h, w, generator=g)).clamp(0, 1)
    return torch.cat([sr, gt]).to(dev).contiguous()


def _flat_block_images(pairs, h, w, seed, dev, block=8):
    """k/255 colours, constant over block x block squares, sr = gt with a third of the blocks one or two levels off: pool windows
    inside a square hold equal maxima, and the ReLU leaves many of them all zero"""
    g = torch.Generator().manual_seed(seed)
    hb, wb = -(-h // block), -(-w // block)
    gt = torch.randint(0, 256, (pairs, 3, hb, wb), generator=g)
    sr = (gt + torch.randint(-2, 3, gt.shape, generator=g) * (torch.rand(gt.shape, generator=g) < 0.33)).clamp(0, 255)
    up = lambda t: t.repeat_interleave(block, 2).repeat_interleave(block, 3)[:, :, :h, :w]  # noqa: E731
    return (torch.cat([up(sr), up(gt)]).float() / 255.0).to(dev).contiguous()


class _Run:
    """one forward, the L1 sum of every feature node and (with grad_conv >= 0) one backward, through the raw C ABI on 0xFF-filled
    buffers"""

    def __init__(self, pairs, h, w, last, feats, gc, det=False, images="random", seed=0, upstream=0.7):
        self.L = L = _lib.load()
        dev = self.dev = torch.device("cuda", 0)
        self.pairs, self.n, self.nb = pairs, 2 * pairs, (pairs if gc >= 0 else 0)
        self.h, self.w, self.last, self.feats, self.gc, self.upstream = h, w, last, sorted(feats), gc, upstream
        self.lat = _lattices(h, w, last)
        self.plan = _Plan(L, self.n, h, w, last, feats, gc, self.nb, det)
        stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
        try:
            self.params = _weights(last, seed, dev)
            make = _pair_images if images == "random" else _flat_block_images
            self.x = make(pairs, h, w, seed + 1, dev)
            self.ws = torch.full((self.plan.workspace_bytes,), 0xFF, dtype=torch.uint8, device=dev)
            self.pk = torch.zeros(self.plan.packed_bytes, dtype=torch.uint8, device=dev)
            ptrs = (C.c_void_p * len(self.params))(*[t.data_ptr() for t in self.params])
            _lib.check(L.b200sr_pack_weights(self.plan.handle, ptrs, C.c_void_p(self.pk.data_ptr()), stream))
            strides = (C.c_int64 * 4)(*self.x.stride())
            _lib.check(L.b200sr_vgg_forward(self.plan.handle, C.c_void_p(self.x.data_ptr()), strides, C.c_void_p(self.pk.data_ptr()),
                                            C.c_void_p(self.ws.data_ptr()), stream))
            self.sums = self.l1_sums()
            self.dx = None
            if gc >= 0:
                self.dx = torch.full((self.nb * 3 * h * w,), -1, dtype=torch.int32, device=dev).view(torch.float32).view(self.nb, 3, h, w)
                up = torch.tensor([upstream], dtype=torch.float32, device=dev)
                _lib.check(L.b200sr_vgg_backward(self.plan.handle, C.c_void_p(up.data_ptr()), C.c_void_p(self.pk.data_ptr()),
                                                 C.c_void_p(self.ws.data_ptr()), C.c_void_p(self.dx.data_ptr()), stream))
            torch.cuda.synchronize()
        except BaseException:
            self.plan.close()
            raise

    def l1_sums(self):
        out = torch.full((len(self.feats),), float("nan"), dtype=torch.float64, device=self.dev)
        stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
        for i, l in enumerate(self.feats):
            _lib.check(self.L.b200sr_vgg_feature_l1(self.plan.handle, C.c_void_p(self.ws.data_ptr()), l, self.pairs,
                                                    C.c_void_p(out[i:].data_ptr()), stream))
        torch.cuda.synchronize()
        return out.cpu()

    def buf(self, name):
        """the workspace tensor as the kernels left it: [images, h, w, C], bf16 (fp32 for F{l})"""
        rc, off, nbytes = _lookup(self.L, self.plan.handle, name)
        assert rc == 0, name
        if name == "xin":
            return self.ws[off:off + nbytes].view(torch.bfloat16).view(self.n, self.h, self.w, 64)
        kind, l = re.fullmatch(r"(A|F|P|G|GP)(\d+)", name).groups()
        l = int(l)
        hl, wl = self.lat[l]
        if kind in ("P", "GP"):
            hl, wl = hl // 2, wl // 2
        imgs = self.nb if kind in ("G", "GP") else self.n
        dt = torch.float32 if kind == "F" else torch.bfloat16
        return self.ws[off:off + nbytes].view(dt).view(imgs, hl, wl, COUT[l])

    def names(self):
        return list(_expected_names(self.n, self.h, self.w, self.last, set(self.feats), self.gc, self.nb))


def _pool_bwd_ref(a, gp):
    """ReLU + MaxPool2d(2, 2) backward from the stored activation a [n, h, w, C] and pooled-lattice gradient gp [n, h/2, w/2, C]:
    the first maximum of each window in row-major order receives the gradient if it is > 0; floor-dropped rows / columns get 0"""
    n, h, w, c = a.shape
    ho, wo = h // 2, w // 2
    win = a[:, :2 * ho, :2 * wo].float().reshape(n, ho, 2, wo, 2, c).permute(0, 1, 3, 5, 2, 4).reshape(n, ho, wo, c, 4)
    vmax, first = win[..., 0], torch.zeros(win.shape[:-1], dtype=torch.long, device=a.device)
    for k in range(1, 4):  # a later element wins only if strictly larger
        later = win[..., k] > vmax
        vmax, first = torch.where(later, win[..., k], vmax), torch.where(later, k, first)
    hit = F.one_hot(first, 4).bool() & (vmax > 0).unsqueeze(-1)
    vals = torch.where(hit, gp.float().unsqueeze(-1), 0.0)  # +0 elsewhere, as the kernel stores it
    out = torch.zeros(n, h, w, c, dtype=torch.float32, device=a.device)
    out[:, :2 * ho, :2 * wo] = vals.reshape(n, ho, wo, c, 2, 2).permute(0, 1, 4, 2, 5, 3).reshape(n, 2 * ho, 2 * wo, c)
    return out.to(torch.bfloat16)


def _check_forward(st, run, sel):
    dt = torch.bfloat16
    # ---- ingest: (x - mean) / std in fp32 (IEEE division), split into hi / lo with the difference taken in fp32
    x = run.x.cpu()
    v = (x - torch.tensor(MEAN).view(1, 3, 1, 1)) / torch.tensor(STD).view(1, 3, 1, 1)
    hi = v.to(dt)
    lo = (v - hi.float()).to(dt)
    ref = torch.cat([hi, lo, hi, torch.zeros(run.n, 55, run.h, run.w, dtype=dt)], dim=1).permute(0, 2, 3, 1)
    st.exact("ingest (vgg_ingest_kernel)", "xin", run.buf("xin").cpu(), ref)
    del x, v, hi, lo, ref

    P = lambda name: _nchw(run.buf(name)[sel])  # noqa: E731
    for l in range(run.last + 1):
        wt, b = run.params[2 * l], run.params[2 * l + 1]
        if l == 0:
            xin = P("xin")
            xh, xl = xin[:, 0:3], xin[:, 3:6]
            wh = wt.to(dt)
            wl = (wt - wh.float()).to(dt)
            wh, wl = wh.double(), wl.double()
            pre = _conv(xh, wh) + _conv(xl, wh) + _conv(xh, wl) + _bias(b)
            m = _conv(xh.abs(), wh.abs()) + _conv(xl.abs(), wh.abs()) + _conv(xh.abs(), wl.abs()) + _bias(b.abs())
            stage = "conv 0 (3-product split)"
            del xin, xh, xl
        else:
            src = f"P{l - 1}" if (l - 1) in POOL_AFTER else f"A{l - 1}"
            a = P(src)
            wr = wt.to(dt).double()
            pre = _conv(a, wr) + _bias(b)
            m = _conv(a.abs(), wr.abs()) + _bias(b.abs())
            stage = f"conv {l} from {src}"
            del a
        post = pre.clamp_min(0)
        st.check(stage + " + ReLU", f"A{l}", P(f"A{l}"), post, m)
        if l in run.feats:
            fr = pre if l == run.last else post
            st.check(stage + (" (fp32 feature, before the ReLU)" if l == run.last else " (fp32 feature, after the ReLU)"), f"F{l}",
                     P(f"F{l}"), fr, m, out_fmt="fp32")
        del pre, post, m
        if l in POOL_AFTER and l < run.last:
            a = run.buf(f"A{l}")[sel]
            ref = F.max_pool2d(a.permute(0, 3, 1, 2).float(), 2).to(dt).permute(0, 2, 3, 1)
            st.exact(f"max-pool {l} (vgg_maxpool_kernel)", f"P{l}", run.buf(f"P{l}")[sel], ref)
            del a, ref


def _check_losses(st, run):
    for i, l in enumerate(run.feats):
        f = run.buf(f"F{l}").double()
        ref = float((f[:run.pairs] - f[run.pairs:]).abs().sum())
        st.rel(f"L1 sum of node {l} (vgg_l1_pair_sum_kernel)", f"F{l}", float(run.sums[i]), ref, L1_REL_BAR)
        del f


def _check_backward(st, run, selb):
    dt = torch.bfloat16
    gc, nb = run.gc, run.nb
    # ---- L1 gradient: bf16(sign(F_sr - F_gt) * fp32(upstream / numel)), times the ReLU derivative for a post-ReLU node
    f = run.buf(f"F{gc}")
    fs, fg = f[:nb], f[nb:]
    hl, wl = run.lat[gc]
    s = torch.tensor(run.upstream, dtype=torch.float32) / torch.tensor(float(nb * hl * wl * COUT[gc]), dtype=torch.float32)
    g = torch.sign(fs - fg) * s.to(fs.device)
    if gc < run.last:
        g = torch.where(fs > 0, g, 0.0)
    st.exact("L1 gradient (vgg_l1_grad_kernel)" + (" x ReLU'" if gc < run.last else ""), f"G{gc}", run.buf(f"G{gc}"), g.to(dt))
    del f, fs, fg, g

    P = lambda name: _nchw(run.buf(name)[selb])  # noqa: E731
    for l in range(gc, -1, -1):
        gi = P(f"G{l}")
        wr = run.params[2 * l].to(dt).double()
        r, m = _convT(gi, wr), _convT(gi.abs(), wr.abs())
        del gi
        if l == 0:
            st.check("conv 0 dgrad (fp32 dx, NCHW)", "dx", run.dx[selb].double(), r, m, out_fmt="fp32")
        elif (l - 1) in POOL_AFTER:
            st.check(f"conv {l} dgrad onto the pooled lattice", f"GP{l - 1}", P(f"GP{l - 1}"), r, m)
            # sr images are the first nb of the batch, so A's image i pairs with G's image i
            ref = _pool_bwd_ref(run.buf(f"A{l - 1}")[selb], run.buf(f"GP{l - 1}")[selb])
            st.exact(f"ReLU + max-pool {l - 1} backward (vgg_maxpool_relu_bwd_kernel)", f"G{l - 1}", run.buf(f"G{l - 1}")[selb], ref)
            del ref
        else:
            d = (P(f"A{l - 1}") > 0).double()
            st.check(f"conv {l} dgrad x ReLU'", f"G{l - 1}", P(f"G{l - 1}"), r * d, m * d)
            del d
        del r, m


# ------------------------------------------------------------------------------------------------------------ GPU
CASES = [  # pairs, (H, W), last_conv, feature nodes, grad_conv, deterministic, images
    pytest.param(1, (16, 16), 15, {15}, 15, False, "random", id="1x16x16-conv15"),      # the 512-channel layers at 2 x 2 and 1 x 1
    pytest.param(2, (33, 47), 15, {15}, 15, False, "random", id="2x33x47-conv15"),      # odd sizes at all four pools
    pytest.param(1, (24, 40), 0, {0}, 0, False, "random", id="1x24x40-conv0"),          # conv1_1 straight to dx
    pytest.param(2, (40, 56), 7, {7}, 7, False, "random", id="2x40x56-conv7"),          # features.16
    pytest.param(3, (48, 80), 15, {1, 3, 7, 11, 15}, -1, False, "random", id="3x48x80-five-nodes"),  # BSRGAN's nodes, forward only
    pytest.param(2, (32, 32), 3, {1, 3}, 1, False, "random", id="2x32x32-grad-conv1-of-3"),  # gradient of a post-ReLU node
    pytest.param(2, (64, 72), 7, {3, 7}, 7, False, "flat", id="2x64x72-ties"),          # equal maxima and all-zero pool windows
    pytest.param(2, (64, 72), 7, {3, 7}, 7, True, "flat", id="2x64x72-ties-det"),
]


def _run_case(pairs, hw, last, feats, gc, det, images):
    run = _Run(pairs, hw[0], hw[1], last, feats, gc, det=det, images=images)
    try:
        st = _Stages(f"vgg pairs={pairs} {hw} last={last} feats={sorted(feats)} grad={gc} det={det} {images}", "bf16")
        for name in run.names():
            st.truth("written in full", name, bool(torch.isfinite(run.buf(name)).all()))
        if run.dx is not None:
            st.truth("written in full", "dx", bool(torch.isfinite(run.dx).all()))
        n, nb = run.n, run.nb
        sel = list(range(n)) if n <= 6 else [0, pairs - 1, pairs, n - 1]
        selb = list(range(nb)) if nb <= 3 else [0, nb - 1]
        _check_forward(st, run, sel)
        _check_losses(st, run)
        if det:
            again = run.l1_sums()
            st.truth("deterministic L1 sums repeat bit for bit", "out_sum", torch.equal(again, run.sums))
        if gc >= 0:
            _check_backward(st, run, selb)
        st.finish()
    finally:
        run.plan.close()


@pytest.mark.gpu
@pytest.mark.parametrize("pairs,hw,last,feats,gc,det,images", CASES)
def test_gpu_vgg_stages_against_fp64(pairs, hw, last, feats, gc, det, images):
    _run_case(pairs, hw, last, feats, gc, det, images)


@pytest.mark.gpu
def test_gpu_vgg_stages_gan_step_shape():
    """the benchmarked GAN step's content loss: 16 pairs at 256^2, features.34, its input gradient (images 0, 15, 16, 31 in the
    forward, sr images 0 and 15 in the backward: every conv works per image, so teacher forcing a subset is exact)"""
    _run_case(16, (256, 256), 15, {15}, 15, False, "random")
    torch.cuda.empty_cache()
