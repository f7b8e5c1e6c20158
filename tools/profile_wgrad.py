"""Where the weight-gradient time of the config-2 training step goes (torch.profiler, CUDA activities).

    python tools/profile_wgrad.py [--steps 5] [--warmup 3] [--label new] [--out DIR]     # GPU: one JSON line
    python tools/profile_wgrad.py --flops-only                                          # CPU: MMA work per dense block

Per profiled step it takes the kernel trace and reports
  * wgrad_sum_ms:  summed duration of all wgrad3x3_kernel launches;
  * dense_median_us: median duration of the weight-gradient launches that start after the trunk data-gradient chain (the 69
    dense-block launches and conv1's single launch);
  * tail_ms: wall time from the end of the trunk data-gradient chain (the third chain launch of a step) to the end of the last
    wgrad3x3_kernel of the step.
Run it in a process of its own: tracing slows the host, so end-to-end step times come from bench.py, not from here.  B200SR_LIB
selects another build of the library (same-box A/B).

--flops-only restates the dense-block problem list of build_plan (b200sr.cu) and prints the MMA work it executes against the work
the five convs' weight and bias gradients need, per dense block at config 2 (16 x 64 x 64 pixels).
"""
import argparse
import json
import os
import statistics
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

# (CTA-units per pixel tile, N) of every problem; one unit runs M = 128 rows x N columns x 16 pixels per MMA, 3 vertical-tap
# accumulators.  A unit is one CTA's share of one pixel split.
PACKED = [("x,o1,o2 x [dY5..dY2], 3 taps", 3, 3, 160), ("(o3,o4 @dx2 | ones) x [dY5..dY2]", 1, 3, 160),
          ("(o3,o4 @dx0 | o3,o4 @dx1) x [dY5|dY4]", 1, 3, 96), ("(x @dx0 | x @dx1) x dY1", 1, 3, 32),
          ("(x @dx2 | ones) x dY1", 1, 3, 32)]


def dense_block_flops(pixels):
    """GFLOP (2 per multiply-add) per dense block: executed by the problem list, and needed by the gradients themselves."""
    useful = 0
    for k in range(1, 6):
        cin, cout = 64 + 32 * (k - 1), (64 if k == 5 else 32)
        useful += 9 * cin * cout + cout  # weight gradient (9 taps) + bias gradient, multiply-adds per pixel
    out = {"useful_gflop": 2 * useful * pixels / 1e9}
    macs = sum(units * nacc * 128 * n for _, units, nacc, n in PACKED)
    out["packed_gflop"] = 2 * macs * pixels / 1e9
    out["packed_ratio"] = macs / useful
    out["packed_columns_per_tile"] = sum(units * nacc * n for _, units, nacc, n in PACKED) / 3
    return out


def profile(args):
    import torch
    import torch.nn.functional as F
    from torch.profiler import ProfilerActivity, profile as tprofile
    import sr_gan_fd_b200 as b200

    dev = torch.device("cuda", 0)
    torch.manual_seed(0)
    net = b200.rrdbnet_x4(num_blocks=23).to(dev).train()
    g = torch.Generator().manual_seed(1234)
    lr = torch.rand(16, 3, 64, 64, generator=g).to(dev)
    gt = torch.rand(16, 3, 256, 256, generator=g).to(dev)

    def step():
        net.zero_grad(set_to_none=True)
        F.l1_loss(net(lr), gt).backward()

    for _ in range(args.warmup):
        step()
    torch.cuda.synchronize()
    with tprofile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(args.steps):
            step()
        torch.cuda.synchronize()
    out_dir = args.out or tempfile.mkdtemp(prefix="profile_wgrad_")
    os.makedirs(out_dir, exist_ok=True)
    trace = os.path.join(out_dir, f"wgrad_{args.label}.pt.trace.json")
    prof.export_chrome_trace(trace)
    with open(trace) as f:
        ev = [e for e in json.load(f)["traceEvents"] if e.get("cat") == "kernel"]
    ev.sort(key=lambda e: e["ts"])
    chains = [e for e in ev if "conv3x3_chain_kernel" in e["name"]]
    wg = [e for e in ev if "wgrad3x3_kernel" in e["name"]]
    if len(chains) != 3 * args.steps:
        raise RuntimeError(f"expected 3 chain launches per step, found {len(chains)} in {args.steps} steps")
    per_step = []
    for i in range(args.steps):
        t0 = chains[3 * i]["ts"]
        t1 = chains[3 * i + 3]["ts"] if i + 1 < args.steps else float("inf")
        trunk_end = chains[3 * i + 2]["ts"] + chains[3 * i + 2]["dur"]
        mine = [e for e in wg if t0 <= e["ts"] < t1]
        after = [e for e in mine if e["ts"] >= trunk_end]
        per_step.append({"wgrad_launches": len(mine), "after_trunk": len(after),
                         "wgrad_sum_ms": sum(e["dur"] for e in mine) / 1e3,
                         "dense_median_us": statistics.median(e["dur"] for e in after),
                         "tail_ms": (max(e["ts"] + e["dur"] for e in mine) - trunk_end) / 1e3})
    med = {k: statistics.median(s[k] for s in per_step) for k in ("wgrad_sum_ms", "dense_median_us", "tail_ms")}
    return {"label": args.label, "steps": args.steps, "lib": os.environ.get("B200SR_LIB", "in-tree"), "median": med, "per_step": per_step, "trace": trace}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--label", default="run")
    ap.add_argument("--out", help="directory for the chrome trace (default: a new temporary directory)")
    ap.add_argument("--flops-only", action="store_true")
    args = ap.parse_args()
    res = {"dense_block_flops_config2": dense_block_flops(16 * 64 * 64)}
    if not args.flops_only:
        res.update(profile(args))
    print(json.dumps(res))


if __name__ == "__main__":
    main()
