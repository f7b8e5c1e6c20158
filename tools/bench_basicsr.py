"""Time of BasicSR's RRDBNet layout (the Real-ESRGAN release generator) at config 2: 16 x 3 x 64^2 -> 256^2, 23 RRDBs, an L1 loss
against a fixed target, forward + backward.

Training-step arms, each timed with CUDA events after `--warmup` untimed calls, the median of `--iters` calls per round, the arms
ALTERNATING over `--rounds` rounds so that box drift hits them alike:
  (a) the layout in plain torch / cuDNN: fp32 with TF32 off, and fp16 autocast + channels_last (the faster one is reported);
  (b) the same module with its body swapped for native_trunk(body): torch head, long skip and HR tail around the native trunk;
  (c) BasicSRRRDBNet: the whole unclamped generator in the native kernels;
  (d) the clamped native generator rrdbnet_x4 on the same input, the reference rate.
Inference arms (no_grad forward) for (b), (c) and (d), reported in output Mpix/s.  The card's name, power limit and max SM clock are
read in the same run.

    python tools/bench_basicsr.py [--iters 10] [--rounds 3] [--warmup 3] [--out results/bench_basicsr.json]
"""
from __future__ import annotations

import argparse
import copy
import json
import os
import statistics
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from bench_partial_grad import card  # noqa: E402


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=10)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    import torch
    import torch.nn.functional as F
    import sr_gan_fd_b200 as b200
    from sr_gan_fd_b200.function import eager_trunk
    if not torch.cuda.is_available():
        raise SystemExit("bench_basicsr needs a CUDA device")
    torch.backends.cudnn.benchmark = True
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    dev = torch.device("cuda", 0)
    N, H, W, NB = 16, 64, 64, 23
    torch.manual_seed(0)
    net = b200.BasicSRRRDBNet(3, 3, scale=4, num_block=NB).to(dev)
    net_cl = copy.deepcopy(net).to(memory_format=torch.channels_last)
    native_body = b200.native_trunk(copy.deepcopy(net.body))
    gen = b200.rrdbnet_x4(num_blocks=NB).to(dev)
    g = torch.Generator().manual_seed(1)
    lr = torch.rand(N, 3, H, W, generator=g).to(dev)
    gt = torch.rand(N, 3, 4 * H, 4 * W, generator=g).to(dev)
    lr_cl = lr.to(memory_format=torch.channels_last)

    def torch_layout(m, body):
        """BasicSR's RRDBNet.forward on m's children, with `body` for the RRDB stack"""
        def f(x):
            feat = m.conv_first(x)
            feat = feat + m.conv_body(body(feat))
            feat = m.lrelu(m.conv_up1(F.interpolate(feat, scale_factor=2, mode="nearest")))
            feat = m.lrelu(m.conv_up2(F.interpolate(feat, scale_factor=2, mode="nearest")))
            return m.conv_last(m.lrelu(m.conv_hr(feat)))
        return f

    torch_fwd = torch_layout(net, lambda t: eager_trunk(net.body, t))
    torch_cl_fwd = torch_layout(net_cl, lambda t: eager_trunk(net_cl.body, t))
    composed_fwd = torch_layout(net, native_body)

    def step(fwd, params_of, x=lr, amp=False):
        def f():
            with torch.autocast("cuda", dtype=torch.float16, enabled=amp):
                y = fwd(x)
            F.l1_loss(y.float(), gt).backward()
            params_of.zero_grad(set_to_none=True)
        return f

    def infer(fwd):
        def f():
            with torch.no_grad():
                fwd(lr)
        return f

    class _Both(torch.nn.Module):  # zero_grad over the composed model's torch children and its native body
        def __init__(self):
            super().__init__()
            self.a, self.b = net, native_body

    both = _Both()
    arms = {"a_torch_fp32": step(torch_fwd, net), "a_torch_fp16_cl": step(torch_cl_fwd, net_cl, lr_cl, amp=True),
            "b_native_trunk": step(composed_fwd, both), "c_basicsr_native": step(net, net), "d_rrdbnet_x4": step(gen, gen),
            "b_infer": infer(composed_fwd), "c_infer": infer(net), "d_infer": infer(gen)}
    for f in arms.values():
        for _ in range(args.warmup):
            f()
    torch.cuda.synchronize()
    times = {k: [] for k in arms}
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(args.rounds):
        for k, f in arms.items():
            for _ in range(args.iters):
                ev0.record()
                f()
                ev1.record()
                ev1.synchronize()
                times[k].append(ev0.elapsed_time(ev1))
    med = {k: statistics.median(v) for k, v in times.items()}
    spread = {k: [round(min(v), 3), round(max(v), 3)] for k, v in times.items()}
    best_torch = min(("a_torch_fp32", "a_torch_fp16_cl"), key=lambda k: med[k])
    out_mpix = N * 4 * H * 4 * W / 1e6
    res = {"card": card(), "shape": [N, 3, H, W], "num_blocks": NB, "iters": args.iters, "rounds": args.rounds,
           "step_ms": {k: round(v, 3) for k, v in med.items() if not k.endswith("_infer")},
           "step_ms_min_max": {k: v for k, v in spread.items() if not k.endswith("_infer")},
           "infer_ms": {k: round(v, 3) for k, v in med.items() if k.endswith("_infer")},
           "infer_mpix_per_s": {k: round(out_mpix / (v / 1e3), 1) for k, v in med.items() if k.endswith("_infer")},
           "best_torch": best_torch,
           "ratios_over_d": {k: round(med[k] / med["d_rrdbnet_x4"], 3) for k in (best_torch, "b_native_trunk", "c_basicsr_native")}}
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
