"""Time of the RRDB trunk as a module of its own (RRDBTrunk), at the config-2 trunk shape: 16 x 64 x 64^2 input, 23 RRDBs.

Arms, each timed with CUDA events after `--warmup` untimed calls, the median of `--iters` calls per round, the arms ALTERNATING over
`--rounds` rounds so that box drift hits them alike:
  * native forward (training plan: autograd graph kept, then dropped);
  * native forward + backward (every parameter gradient and dx);
  * the same Sequential through torch / cuDNN, forward + backward: fp32 (TF32 off), fp16 autocast, fp16 autocast + channels_last;
  * composed model at config 2: torch conv1 + native trunk + torch tail (conv2 + long skip, 2 x (nearest x2 + conv + LeakyReLU),
    conv3 + LeakyReLU, conv4, clamp), fwd + bwd of an L1 loss, against the native generator (rrdbnet_x4) on the same input.
TFLOP/s = b200sr_flops of the trunk plan over the median time.  The card's name and power limit are read in the same run.

    python tools/bench_trunk.py [--iters 20] [--rounds 3] [--warmup 3] [--out results/bench_trunk.json]
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
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    import torch
    import torch.nn.functional as F
    from torch import nn
    import sr_gan_fd_b200 as b200
    from sr_gan_fd_b200.function import eager_trunk
    if not torch.cuda.is_available():
        raise SystemExit("bench_trunk needs a CUDA device")
    torch.backends.cudnn.benchmark = True
    torch.backends.cudnn.allow_tf32 = False
    dev = torch.device("cuda", 0)
    torch.manual_seed(0)
    N, H, W, NB = 16, 64, 64, 23
    trunk = b200.RRDBTrunk(num_blocks=NB).to(dev)
    g = torch.Generator().manual_seed(1)
    x = torch.randn(N, 64, H, W, generator=g).to(dev)
    dy = torch.randn(N, 64, H, W, generator=g).to(dev)
    x_cl = x.to(memory_format=torch.channels_last)
    trunk_cl = copy.deepcopy(trunk).to(memory_format=torch.channels_last)

    class Eager(nn.Module):  # the same Sequential's math through torch ops (cuDNN convs)
        def __init__(self, t):
            super().__init__()
            self.t = t

        def forward(self, v):
            return eager_trunk(self.t, v)

    eager, eager_cl = Eager(trunk), Eager(trunk_cl)

    def native_fwd():
        xx = x.requires_grad_(True)
        trunk(xx)
        x.requires_grad_(False)

    def native_fb():
        xx = x.detach().requires_grad_(True)
        trunk(xx).backward(dy)
        trunk.zero_grad(set_to_none=True)

    def torch_fb(model, inp, amp):
        def f():
            xx = inp.detach().requires_grad_(True)
            with torch.autocast("cuda", dtype=torch.float16, enabled=amp):
                y = model(xx)
            y.float().backward(dy)
            model.zero_grad(set_to_none=True)
        return f

    # composed model vs the native generator, config 2 (16 x 3 x 64^2 -> 256^2)
    gen = b200.rrdbnet_x4(num_blocks=NB).to(dev)

    class Composed(nn.Module):
        def __init__(self, net):
            super().__init__()
            net = copy.deepcopy(net)
            self.conv1, self.conv2, self.conv3, self.conv4 = net.conv1, net.conv2, net.conv3, net.conv4
            self.up = nn.ModuleList([net.upsampling1, net.upsampling2])
            self.trunk = b200.native_trunk(net.trunk)

        def forward(self, v):
            head = self.conv1(v)
            t = head + self.conv2(self.trunk(head))
            for u in self.up:
                t = u(F.interpolate(t, scale_factor=2, mode="nearest"))
            return torch.clamp(self.conv4(self.conv3(t)), 0.0, 1.0)

    comp = Composed(gen)
    lr = torch.rand(N, 3, H, W, generator=g).to(dev)
    gt = torch.rand(N, 3, 4 * H, 4 * W, generator=g).to(dev)

    def step(model):
        def f():
            F.l1_loss(model(lr), gt).backward()
            model.zero_grad(set_to_none=True)
        return f

    arms = {"native_fwd": native_fwd, "native_fwd_bwd": native_fb,
            "torch_fp32_fwd_bwd": torch_fb(eager, x, False), "torch_fp16_fwd_bwd": torch_fb(eager, x, True),
            "torch_fp16_cl_fwd_bwd": torch_fb(eager_cl, x_cl, True),
            "composed_step": step(comp), "generator_step": step(gen)}
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
    plan = trunk._runtime().last_plan
    fl_f, fl_b = plan.flops_fwd, plan.flops_bwd
    best_torch = min(("torch_fp32_fwd_bwd", "torch_fp16_fwd_bwd", "torch_fp16_cl_fwd_bwd"), key=lambda k: med[k])
    res = {"card": card(), "shape": [N, 64, H, W], "num_blocks": NB, "iters": args.iters, "rounds": args.rounds,
           "ms": {k: round(v, 3) for k, v in med.items()},
           "tflops": {"native_fwd": round(fl_f / med["native_fwd"] / 1e9, 1),
                      "native_fwd_bwd": round((fl_f + fl_b) / med["native_fwd_bwd"] / 1e9, 1),
                      best_torch: round((fl_f + fl_b) / med[best_torch] / 1e9, 1)},
           "best_torch": best_torch, "speedup_fwd_bwd_vs_best_torch": round(med[best_torch] / med["native_fwd_bwd"], 2),
           "composed_over_generator": round(med["composed_step"] / med["generator_step"], 3)}
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
