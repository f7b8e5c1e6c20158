"""Step time of config 2 (16 x 64^2 -> 256^2, 23 RRDBs, L1 loss, fwd + bwd through the module API) for freeze patterns:
full, frozen generator + dL/dx, tail only, conv1 + the first 12 RRDBs frozen, conv1 + the first 22 RRDBs frozen.

The patterns ALTERNATE inside one process (each of `--rounds` rounds runs `--steps` timed steps of every pattern in turn,
after `--warmup` untimed steps per pattern), so box drift hits every pattern alike.  Each step is timed with CUDA events around
forward + loss + backward; the median over all timed steps is reported, with the backward launch count of the pattern
(b200sr_backward_launches) and the card's name and power limit read in the same run.

    python tools/bench_partial_grad.py [--steps 20] [--rounds 3] [--warmup 3]
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def trainable(name: str, pattern: str) -> bool:
    if pattern == "full":
        return True
    if pattern == "frozen+dx":
        return False
    if pattern == "tail":
        return not (name.startswith("conv1.") or name.startswith("trunk."))
    k = int(pattern.split("+")[1])  # "head+k": conv1 and RRDBs 0 .. k-1 frozen
    return not (name.startswith("conv1.") or (name.startswith("trunk.") and int(name.split(".")[1]) < k))


PATTERNS = ["full", "frozen+dx", "tail", "head+12", "head+22"]


def card() -> dict:
    import torch
    out = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader,nounits"],
                           capture_output=True, text=True, timeout=30).stdout.strip().split(",")
        out["power_limit_w"], out["sm_max_mhz"] = float(q[0]), float(q[1])
    except Exception as e:  # the card name alone still identifies the measurement
        out["power_limit_w"] = f"unavailable ({e})"
    return out


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--patterns", default=",".join(PATTERNS))
    args = ap.parse_args()
    import torch
    import torch.nn.functional as F
    import sr_gan_fd_b200 as b200
    if not torch.cuda.is_available():
        raise SystemExit("bench_partial_grad needs a CUDA device")
    dev = torch.device("cuda", 0)
    torch.manual_seed(0)
    net = b200.rrdbnet_x4(num_blocks=23).to(dev).train()
    g = torch.Generator().manual_seed(1)
    lr = torch.rand(16, 3, 64, 64, generator=g).to(dev)
    gt = torch.rand(16, 3, 256, 256, generator=g).to(dev)
    patterns = args.patterns.split(",")
    names = [n for n, _ in net.named_parameters()]
    flags = {p: [trainable(n, p) for n in names] for p in patterns}

    def step(p):
        for prm, t in zip(net.parameters(), flags[p]):
            prm.requires_grad_(t)
        x = lr.requires_grad_(p == "frozen+dx")
        F.l1_loss(net(x), gt).backward()
        net.zero_grad(set_to_none=True)
        lr.grad = None

    for _ in range(args.warmup):
        for p in patterns:
            step(p)
    torch.cuda.synchronize()
    times = {p: [] for p in patterns}
    for _ in range(args.rounds):
        for p in patterns:
            for _ in range(args.steps):
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                step(p)
                b.record()
                torch.cuda.synchronize()
                times[p].append(a.elapsed_time(b))
    plan = net._runtime().last_plan
    res = {"card": card(), "config": "16x3x64x64 -> 256x256, 23 RRDB, L1, fwd+bwd", "steps_per_pattern": args.steps * args.rounds,
           "lib": os.environ.get("B200SR_LIB", "in-tree"), "patterns": {}}
    for p in patterns:
        t = times[p]
        res["patterns"][p] = {"ms_per_step_median": round(statistics.median(t), 3), "ms_min": round(min(t), 3),
                              "ms_max": round(max(t), 3),
                              "bwd_launches": plan.backward_launches(flags[p], with_dx=(p == "frozen+dx"))}
        print(f"{p:10s} {statistics.median(t):8.3f} ms/step (min {min(t):.3f}, max {max(t):.3f})  "
              f"backward launches {res['patterns'][p]['bwd_launches']}")
    print(json.dumps(res))


if __name__ == "__main__":
    main()
