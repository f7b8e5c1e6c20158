"""Cost of deterministic mode (torch.use_deterministic_algorithms): default and deterministic plans alternate in one process.

  * config-2 generator step: 16 x 64 x 64, 23 RRDBs, forward + L1 + backward (median of --steps steps per mode);
  * the discriminator update at 16 x 256 x 256 (fp16): forward + backward with weight gradients;
  * the all-native GAN step of tools/gan_step.py (generator, U-Net discriminator, VGG content loss, fused Adam + EMA).

Prints one JSON line with the medians, the workspace bytes of both modes, the card and its power limit.
Usage: CUBLAS_WORKSPACE_CONFIG=:4096:8 python tools/bench_deterministic.py [--steps 60]"""
import argparse
import json
import os
import statistics
import subprocess
import sys

import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))


def card():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                              capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception:
        return torch.cuda.get_device_name(0)


def timed(fn, det, n):
    torch.use_deterministic_algorithms(det, warn_only=True)
    ms = []
    for _ in range(n):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        e1.synchronize()
        ms.append(e0.elapsed_time(e1))
    torch.use_deterministic_algorithms(False)
    return ms


def compare(fn, steps, rounds=4):
    out = {False: [], True: []}
    for det in (False, True):
        timed(fn, det, 3)  # warm: plans, descriptors
    for _ in range(rounds):
        for det in (False, True):
            out[det] += timed(fn, det, steps // rounds)
    return {"default_ms": statistics.median(out[False]), "deterministic_ms": statistics.median(out[True])}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=60)
    args = ap.parse_args()
    os.environ.setdefault("CUBLAS_WORKSPACE_CONFIG", ":4096:8")
    dev = torch.device("cuda", 0)
    import gan_step
    import sr_gan_fd_b200 as b200
    from sr_gan_fd_b200.discriminator import discriminator_unet
    res = {"card": card()}

    torch.manual_seed(0)
    g = b200.rrdbnet_x4(num_blocks=23).to(dev).train()
    lr = torch.rand(16, 3, 64, 64, device=dev)
    gt = torch.rand(16, 3, 256, 256, device=dev)

    def gen_step():
        F.l1_loss(g(lr), gt).backward()
        g.zero_grad(set_to_none=True)
    res["generator_config2"] = compare(gen_step, args.steps)
    res["generator_config2"]["workspace_bytes"] = {str(k[-1]): p.workspace_bytes for k, p in g._runtime().plans.items()}

    d = discriminator_unet(in_channels=3, out_channels=1, channels=64).to(dev).train()
    hr = torch.rand(16, 3, 256, 256, device=dev)

    def disc_step():
        d(hr).square().mean().backward()
        d.zero_grad(set_to_none=True)
    res["discriminator_16x256"] = compare(disc_step, args.steps)
    res["discriminator_16x256"]["workspace_bytes"] = {str(k[-1]): p.workspace_bytes for k, p in d._runtime().plans.items()}

    dm, gm, content = gan_step.build("b200", dev, seed=0, content="b200", disc="b200")
    dm.train(); gm.train()
    step = gan_step.GanStep(dm, gm, content, dev, optimizer="fused", ema=True)
    res["gan_step_16x64"] = compare(lambda: step(lr, gt), max(args.steps // 2, 8))
    for v in res.values():
        if isinstance(v, dict) and "default_ms" in v:
            v["overhead_pct"] = 100.0 * (v["deterministic_ms"] / v["default_ms"] - 1.0)
    print(json.dumps(res), flush=True)


if __name__ == "__main__":
    main()
