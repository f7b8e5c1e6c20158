#!/usr/bin/env python
"""Benchmark contract for the B200-native RRDBNet generator (MiNeves00/SR-GAN-FD hot path).

    python bench.py --gpus N --steps K --warmup W [--impl reference] [--dump-outputs DIR]

Workload at every N = BASELINE.json configs[1]/[2]: RRDBNet x4 (23 RRDB, 64 ch, growth 32) L1 pre-training step,
forward + backward, 16 synthetic 64x64 LR images per GPU -> 256x256 GT, bf16 tensor-core arithmetic with fp32
accumulation (weak scaling: N=8 is exactly config 3's global batch 128); for N>1 the 16.7 M-parameter gradient is
all-reduced (NCCL, averaged; by default ONE coalesced call issued when backward has enqueued its last kernel -- see
sr_gan_fd_b200/dist.py).  One "step" = one fwd+bwd(+all-reduce) of the
generator.  `value` = images/s with inputs resident in HBM, `e2e` = the same step driven through the public module API
with pinned-host inputs copied in (side stream, one step ahead, like the reference's CUDAPrefetcher) and every step's loss
copied back to pinned host memory and read by the host one step later (`e2e.sync_readback`: the same with a blocking
`loss.item()` per step).  Rank 0 prints ONE JSON line.

`--impl reference` times the reference's own CPU implementation of the same step on all host cores: the UNMODIFIED
`ESRGAN/model.py::rrdbnet_x4` from the staged copy under baseline/_ref (git-ignored; `__graft_entry__.stage_reference()`
makes it in the build container and it travels to the GPU box, where /root/reference is absent), driven as
train_rrdbnet.py:252-261 does (`cpu_baseline.kind = "reference"`); without the staged copy, the fp32 oracle restatement
(asserted bit-equal to the reference classes in tests/; `kind = "port"`).  Full 16-image batch per step.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "RRDBNet x4 train imgs/s (L1 pretraining fwd+bwd; BASELINE configs[1]/[2])"
UNIT = "img/s"
BATCH_PER_GPU, LR_HW, SCALE, NUM_BLOCKS = 16, 64, 4, 23
WORKLOAD = ("RRDBNet x4 L1 pretraining step fwd+bwd, batch 16/GPU, 64x64 LR -> 256x256 GT, 23 RRDB, 64 ch, growth 32 "
            "(BASELINE.json configs[1]; N>1 = configs[2] data-parallel)")


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return float(d.get("bf16_tflops", 1590.0)), float(d.get("bf16_tflops_sustained", 1400.0)), "measured"
    return 1590.0, 1400.0, "fallback"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md recipe)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index = index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, pw, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2])); pw.append(float(f[3]))
            except ValueError:
                continue
            for nm, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None, "samples": len(sm), "reasons": sorted(reasons)}


# ------------------------------------------------------------------------------------------------ reference arm
def _reference_generator():
    """The UNMODIFIED reference generator, if a staged copy of the reference tree travels with the repo (`baseline/_ref/ESRGAN/model.py`,
    git-ignored; /root/reference itself does not exist on the GPU box): `rrdbnet_x4` built with rrdbnet_config.py's values.  None if the
    copy is absent (then the oracle restatement stands in, `kind: "port"`)."""
    path = os.path.join(ROOT, "baseline", "_ref", "ESRGAN", "model.py")
    if not os.path.exists(path):
        return None
    import importlib.util
    import torch
    try:
        spec = importlib.util.spec_from_file_location("_reference_esrgan_model", path)
        mod = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mod)
        torch.manual_seed(0)
        net = mod.rrdbnet_x4(in_channels=3, out_channels=3, channels=64, growth_channels=32, num_blocks=NUM_BLOCKS)
        return net.train()
    except Exception as exc:  # e.g. torchvision missing on the box: say so and fall back to the port
        sys.stderr.write(f"bench.py: staged reference not usable ({exc!r}); using the oracle port\n")
        return None


def cpu_reference_step(batch, threads):
    """One L1 fwd+bwd (fp32, CPU) on `batch` 64x64 LR images: the reference's own RRDBNet driven as ESRGAN/train_rrdbnet.py:252-261 does
    (zero_grad, forward, L1 criterion, backward; its CUDA autocast / GradScaler are no-ops on CPU tensors) when the staged reference is
    present, else the oracle restatement.  Returns seconds."""
    import torch
    torch.set_num_threads(threads)
    lr = torch.rand(batch, 3, LR_HW, LR_HW)
    gt = torch.rand(batch, 3, LR_HW * SCALE, LR_HW * SCALE)
    net = cpu_reference_step.net
    if net is not None:
        t0 = time.perf_counter()
        net.zero_grad(set_to_none=True)
        loss = torch.nn.functional.l1_loss(net(lr), gt)
        loss.backward()
        loss.item()
        return time.perf_counter() - t0
    from oracle import rrdbnet_oracle as orc
    t0 = time.perf_counter()
    orc.rrdbnet_l1_step(cpu_reference_step.params, lr, gt)
    return time.perf_counter() - t0


def cpu_full_batch(warmup, steps, budget_s=420.0):
    """THE CPU method of both arms: the reference generator (staged copy of ESRGAN/model.py; else the oracle restatement) in fp32 on torch
    CPU with every host thread, on the FULL workload batch (16 images, 64x64 LR -> 256x256, fwd+bwd L1), `warmup` untimed + `steps`
    timed steps.  Only if the first step shows the whole run would exceed `budget_s` is the per-step sample cut to 8 / 4 images (and
    said so in `sample`)."""
    import torch
    torch.manual_seed(0)
    threads = os.cpu_count() or 1
    cpu_reference_step.net = _reference_generator()
    if cpu_reference_step.net is None:
        from oracle import rrdbnet_oracle as orc
        cpu_reference_step.params = orc.init_params(seed=0, num_blocks=NUM_BLOCKS, upscale_factor=SCALE)
    kind = "reference" if cpu_reference_step.net is not None else "port"
    what = ("the reference's own RRDBNet (baseline/_ref/ESRGAN/model.py, unmodified) driven as train_rrdbnet.py does" if kind == "reference"
            else "oracle restatement of ESRGAN/model.py")
    cpu_reference_step(1, threads)  # allocator / oneDNN primitive warm-up (1 image, untimed)
    batch = BATCH_PER_GPU
    t_first = cpu_reference_step(batch, threads)  # counts as the first warm-up step
    while batch > 4 and t_first * (batch / BATCH_PER_GPU) * (warmup + steps) > budget_s:
        batch //= 2
    for _ in range(max(warmup - 1, 0)):
        cpu_reference_step(batch, threads)
    times = [cpu_reference_step(batch, threads) for _ in range(steps)]
    sec = sum(times) / len(times)
    sample = (f"{batch} of {BATCH_PER_GPU} images per step ({'the full batch' if batch == BATCH_PER_GPU else 'bounded sample'}), "
              f"{steps} timed steps after {max(warmup, 1)} warm-up, fp32 fwd+bwd L1, {what}, torch CPU")
    return {"value": batch / sec, "unit": UNIT, "cores": threads, "kind": kind, "sample": sample,
            "sec_per_step": sec, "batch": batch}


def bench_config(world):
    return {"workload": WORKLOAD, "global_batch": world * BATCH_PER_GPU, "parallelism": f"dp{world}",
            "l2_policy": "activation working set per step (3.1 GB) is far larger than the 126 MB L2, no flush needed",
            "host": "python cyclic GC collected before and disabled inside each timed region",
            "precision": "bf16 operands / fp32 accumulate in the trunk, fp32 residual carrier, hi+lo split bf16 in head/tail"}


def seeded_inputs(rank=0):
    """The LR and GT batches of one rank's training step: the same on every run."""
    import torch
    torch.manual_seed(1234 + rank)
    return torch.rand(BATCH_PER_GPU, 3, LR_HW, LR_HW), torch.rand(BATCH_PER_GPU, 3, LR_HW * SCALE, LR_HW * SCALE)


GRAD_SAMPLE = 1 << 23  # entries of the 16.7 M-entry flat gradient that --dump-outputs writes (34 MB; 46 MB with sr.npy)


def dump_outputs(out_dir, sr, loss, net):
    """Write what one training step hands its caller, as float32 .npy files under `out_dir`: `sr` (the SR batch), `loss` (the L1
    loss) and `grad_sample` -- the parameter gradients flattened in `net.parameters()` order, sampled at GRAD_SAMPLE fixed
    positions (a seed-0 permutation, ascending), because the whole gradient (67 MB) next to the SR batch (13 MB) would not fit
    the dump's 64 MB."""
    import numpy as np
    import torch
    os.makedirs(out_dir, exist_ok=True)
    flat = torch.cat([p.grad.flatten() for p in net.parameters()])
    idx = torch.randperm(flat.numel(), generator=torch.Generator().manual_seed(0))[:GRAD_SAMPLE].sort().values
    for name, t in (("sr", sr), ("loss", loss), ("grad_sample", flat[idx.to(flat.device)])):
        np.save(os.path.join(out_dir, name + ".npy"), t.float().cpu().numpy())


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cb = cpu_full_batch(args.warmup, args.steps)
    sec, batch = cb.pop("sec_per_step"), cb.pop("batch")
    value = cb["value"]
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": sec * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": bench_config(max(args.gpus, 1)),
        "cpu_baseline": cb,
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------ library baseline
def library_baseline(net, lr_dev, gt_dev, iters=5):
    """The reference generator graph through stock torch / cuDNN on the SAME GPU (SURVEY 8d: "the bar becomes: beat what
    torch+cuDNN runs"): the drop-in's own nn.Conv2d children driven by plain torch ops (cat / conv2d / leaky_relu /
    interpolate -- the op sequence of ESRGAN/model.py:49-60,77-86,211-232; /root/reference itself is absent on the GPU box),
    same batch, same L1 step as ESRGAN/train_rrdbnet.py:256-261, cudnn.benchmark on as in rrdbnet_config.py:25."""
    import copy
    import torch
    import torch.nn.functional as F
    from sr_gan_fd_b200.function import eager_forward
    out = {"what": "same generator, stock torch ops on cuDNN/cuBLAS kernels, fwd+bwd L1, 16 x 64x64 LR, img/s (higher is better)"}
    prev = (torch.backends.cudnn.benchmark, torch.backends.cudnn.allow_tf32)
    torch.backends.cudnn.benchmark = True
    variants = [("fp32_tf32_nchw", None, False, True), ("fp32_tf32_channels_last", None, True, True),
                ("fp32_strict_nchw", None, False, False),
                ("fp16_autocast_nchw", torch.float16, False, True), ("fp16_autocast_channels_last", torch.float16, True, True),
                ("bf16_autocast_nchw", torch.bfloat16, False, True), ("bf16_autocast_channels_last", torch.bfloat16, True, True)]
    for name, dtype, cl, tf32 in variants:
        try:
            torch.backends.cudnn.allow_tf32 = tf32
            m = copy.deepcopy(net)
            x = lr_dev
            if cl:
                m = m.to(memory_format=torch.channels_last)
                x = lr_dev.contiguous(memory_format=torch.channels_last)

            def step():
                m.zero_grad(set_to_none=True)
                with torch.autocast("cuda", dtype=dtype or torch.float16, enabled=dtype is not None):
                    loss = F.l1_loss(eager_forward(m, x), gt_dev)
                (loss * (1024.0 if dtype is torch.float16 else 1.0)).backward()

            for _ in range(3):
                step()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(iters):
                step()
            e1.record()
            torch.cuda.synchronize()
            out[name] = BATCH_PER_GPU / (e0.elapsed_time(e1) / iters * 1e-3)
            del m
            torch.cuda.empty_cache()
        except Exception as exc:  # a baseline variant that cannot run is reported, not fatal
            out[name] = f"failed: {type(exc).__name__}: {str(exc)[:80]}"
    torch.backends.cudnn.benchmark, torch.backends.cudnn.allow_tf32 = prev
    nums = [v for v in out.values() if isinstance(v, float)]
    out["best"] = max(nums) if nums else None
    return out


# ------------------------------------------------------------------------------------------------------ our arm
def widened_components(dev, steps=5):
    """SURVEY.md section 8(f) components next to the path, timed in the same run (N = 1 only; short): the U-Net discriminator's three
    passes (native vs the same module through stock torch ops: fp16 autocast as the reference scripts run it, and channels_last on
    top -- the fastest library arm) and the BSRGAN GAN step (BASELINE configs[4]) with every component native."""
    import importlib.util

    import torch
    out = {}
    try:
        from sr_gan_fd_b200.discriminator import discriminator_unet
        torch.manual_seed(0)
        d = discriminator_unet(in_channels=3, out_channels=1, channels=64).to(dev).train()
        x = torch.rand(BATCH_PER_GPU, 3, LR_HW * SCALE, LR_HW * SCALE, device=dev)
        dy = torch.randn(BATCH_PER_GPU, 1, LR_HW * SCALE, LR_HW * SCALE, device=dev) / x[:, :1].numel()

        def t(fn, n=steps):
            for _ in range(3):
                fn()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(n):
                fn()
            e1.record()
            torch.cuda.synchronize()
            return e0.elapsed_time(e1) / n

        def passes(xin, autocast):
            def d_update():
                for p in d.parameters():
                    p.requires_grad = True
                d.zero_grad(set_to_none=True)
                with torch.autocast("cuda", dtype=torch.float16, enabled=autocast):
                    y = d(xin)
                y.float().backward(dy)

            def g_update():
                for p in d.parameters():
                    p.requires_grad = False
                xr = xin.detach().requires_grad_(True)
                with torch.autocast("cuda", dtype=torch.float16, enabled=autocast):
                    y = d(xr)
                y.float().backward(dy)
            return {"d_update_ms": t(d_update), "g_update_ms": t(g_update)}

        rec = {"shape": [BATCH_PER_GPU, 3, LR_HW * SCALE, LR_HW * SCALE], "b200": passes(x, False)}
        plan = d._runtime().last_plan
        rec["b200_d_update_tflops"] = (plan.flops_fwd + plan.flops_bwd_d) / (rec["b200"]["d_update_ms"] * 1e-3) / 1e12
        d.use_native = False
        rec["torch_fp16_autocast"] = passes(x, True)
        d = d.to(memory_format=torch.channels_last)
        rec["torch_fp16_autocast_channels_last"] = passes(x.contiguous(memory_format=torch.channels_last), True)
        out["discriminator_unet"] = rec
        del d, x, dy
        torch.cuda.empty_cache()
    except Exception as exc:  # a widened component must never take the headline line down
        out["discriminator_unet"] = {"error": repr(exc)[:200]}
    try:
        spec = importlib.util.spec_from_file_location("_gan_step", os.path.join(ROOT, "tools", "gan_step.py"))
        gs = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(gs)
        d_model, g_model, content = gs.build("b200", dev, content="b200", disc="b200")
        d_model.train(); g_model.train()
        step = gs.GanStep(d_model, g_model, content, dev, 1, optimizer="fused", ema=True)
        lr = torch.rand(BATCH_PER_GPU, 3, LR_HW, LR_HW, device=dev)
        gt = torch.rand(BATCH_PER_GPU, 3, LR_HW * SCALE, LR_HW * SCALE, device=dev)
        for _ in range(3):
            step(lr, gt)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            step(lr, gt)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / steps
        out["bsrgan_gan_step"] = {"ms_per_step": ms, "img_per_s": BATCH_PER_GPU / (ms * 1e-3),
                                  "config": "BASELINE configs[4]: generator + U-Net discriminator x3 + VGG19 content loss (seeded random-init VGG19) + fused Adam/EMA, "
                                            "autocast + GradScaler, all components from sr_gan_fd_b200"}
        del step, d_model, g_model, content
        torch.cuda.empty_cache()
    except Exception as exc:
        out["bsrgan_gan_step"] = {"error": repr(exc)[:200]}
    return out


def run_b200(args):
    import torch
    import torch.distributed as dist
    import torch.nn.functional as F
    import sr_gan_fd_b200 as b200
    from sr_gan_fd_b200 import dist as b200dist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py needs a CUDA device (the B200 path has no CPU fallback); use --impl reference for the CPU arm")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    torch.manual_seed(0)  # identical replicas on every rank (same seed, rrdbnet_config.py:20-23)
    net = b200.rrdbnet_x4(in_channels=3, out_channels=3, channels=64, growth_channels=32, num_blocks=NUM_BLOCKS).to(dev)
    net.train()
    dp_err = None
    if world > 1:
        # data-parallel equivalence, checked on every run before anything is timed: `world` ranks x 2 images with the NCCL
        # gradient averaging must equal ONE replica on the 2*world-image global batch (flat-gradient rel-L2)
        g = torch.Generator().manual_seed(77)
        xs = torch.rand(2 * world, 3, 32, 32, generator=g).to(dev)
        ys = torch.rand(2 * world, 3, 128, 128, generator=g).to(dev)
        F.l1_loss(net(xs), ys).backward()
        ref_flat = torch.cat([p.grad.flatten() for p in net.parameters()]).double()
        net.zero_grad(set_to_none=True)
    reducer = b200dist.make_data_parallel(net) if world > 1 else None
    if world > 1:
        sl = slice(2 * rank, 2 * rank + 2)
        F.l1_loss(net(xs[sl]), ys[sl]).backward()
        got_flat = torch.cat([p.grad.flatten() for p in net.parameters()]).double()
        err = ((got_flat - ref_flat).norm() / ref_flat.norm()).reshape(1)
        dist.all_reduce(err, op=dist.ReduceOp.MAX)
        dp_err = float(err.item())
        net.zero_grad(set_to_none=True)
        del xs, ys, ref_flat, got_flat
        if not dp_err < 2e-3:
            raise RuntimeError(f"data-parallel gradients differ from the single-replica gradients: rel-L2 {dp_err:.3e}")

    lr_host, gt_host = (t.pin_memory() for t in seeded_inputs(rank))
    lr_dev, gt_dev = lr_host.to(dev), gt_host.to(dev)
    last = {}  # what the latest resident step returned (detached: the autograd graph is not kept alive), for --dump-outputs

    def step_resident():
        net.zero_grad(set_to_none=True)
        sr = net(lr_dev)
        loss = F.l1_loss(sr, gt_dev)
        loss.backward()
        last.update(sr=sr.detach(), loss=loss.detach())
        return loss

    # End to end through the public API.  Like the reference's CUDAPrefetcher (ESRGAN/dataset.py:196-236) the NEXT batch is
    # copied host->device on a side stream while the current step computes; every step still moves its own inputs from
    # pinned host memory inside the timed region and reads its loss back to the host.
    copy_stream = torch.cuda.Stream(device=dev)
    # two pre-allocated device staging pairs (no allocator traffic in the loop): the copy into pair 1-i is ordered after the
    # step that last read it (event) and runs while step i computes
    stage = [(torch.empty_like(lr_dev), torch.empty_like(gt_dev)) for _ in range(2)]
    copied = [torch.cuda.Event() for _ in range(2)]
    consumed = [torch.cuda.Event() for _ in range(2)]
    state = {"i": 0, "primed": False}

    def prefetch(i):
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(consumed[i])
            stage[i][0].copy_(lr_host, non_blocking=True)
            stage[i][1].copy_(gt_host, non_blocking=True)
            copied[i].record(copy_stream)

    # The loss is read back to the host EVERY step, asynchronously: the scalar goes device -> pinned host right behind the
    # backward pass and the host picks it up one step later (the last one before the closing timestamp), so the host can
    # enqueue step i+1 while the GPU finishes step i.  (A blocking loss.item() per step -- the reference loop's
    # `losses.update(loss.item(), ...)` -- leaves the GPU idle while Python re-enters the module: reported as e2e.sync_readback.)
    loss_host = [torch.empty((), dtype=torch.float32).pin_memory() for _ in range(2)]
    loss_ready = [torch.cuda.Event() for _ in range(2)]
    losses_read = []

    def read_pending():
        j = state.get("pending")
        if j is not None:
            loss_ready[j].synchronize()
            losses_read.append(float(loss_host[j]))
            state["pending"] = None

    def step_e2e(sync_readback=False):
        i = state["i"]
        if not state["primed"]:
            consumed[0].record(); consumed[1].record()
            prefetch(i)
            state["primed"] = True
        cur = torch.cuda.current_stream()
        cur.wait_event(copied[i])
        lr, gt = stage[i]
        prefetch(1 - i)  # next step's inputs, overlapped with this step's compute
        net.zero_grad(set_to_none=True)
        loss = F.l1_loss(net(lr), gt)
        loss.backward()
        consumed[i].record(cur)
        state["i"] = 1 - i
        if sync_readback:
            return loss.item()  # blocking device -> host read of the step's result
        loss_host[i].copy_(loss.detach(), non_blocking=True)  # device -> host read of the step's result (4 bytes, pinned)
        loss_ready[i].record(cur)
        read_pending()          # the PREVIOUS step's loss
        state["pending"] = i

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps, flush=None):
        # Python's cyclic GC is collected up front and held off inside the timed region (as timeit does): one generation-2
        # sweep over torch's object graph costs ~30 ms of host time, which lands in whichever 20-step window it fires in
        # (measured: end-to-end 14.3 ms/step at --steps 20 against 12.7 at --steps 10 and 40 before this)
        import gc
        gc.collect()
        gc.disable()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        if flush:
            flush()  # (end to end: the last step's loss is read on the host before the closing timestamp)
        e1.record()
        barrier()
        gc.enable()
        ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms

    for _ in range(max(args.warmup, 3)):
        step_resident()
    sampler = ClockSampler(local_rank) if rank == 0 else None
    if sampler:
        sampler.start()
    ms_total = timed(step_resident, args.steps)
    clocks = sampler.stop() if sampler else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, last["sr"], last["loss"], net)
    last.clear()
    plan = net._runtime().last_plan
    bucketed = world > 1 and net._runtime().grad_bucket_hook is not None
    ms_step = ms_total / args.steps
    value = world * BATCH_PER_GPU / (ms_step * 1e-3)

    # end-to-end through the public API, host buffers in / loss out every step
    for _ in range(2):
        step_e2e()
    read_pending()
    ms_e2e = timed(step_e2e, args.steps, flush=read_pending) / args.steps
    assert len(losses_read) == args.steps + 2 and all(v == v and v > 0 for v in losses_read), losses_read
    ms_e2e_sync = timed(lambda: step_e2e(True), args.steps) / args.steps
    e2e_value = world * BATCH_PER_GPU / (ms_e2e * 1e-3)

    # dominant kernel (conv3x3_chain_kernel: every forward conv and every data-gradient conv): the forward pass is ONE
    # launch of it over 351 layers (+1 tiny ingest kernel), so forward FLOPs / forward time is its achieved rate,
    # measured live here with CUDA events on the launching stream.
    # (training-mode forward = exactly the launch that runs inside the timed step; the eval-mode forward with ping-pong
    # buffers is timed as well for the inference throughput figure)
    fwd_iters = max(3, min(args.steps, 20))
    for _ in range(3):
        net(lr_dev)
    ms_fwd = timed(lambda: net(lr_dev), fwd_iters) / fwd_iters
    iplan = net._runtime().last_plan
    net.eval()
    with torch.no_grad():
        for _ in range(3):
            net(lr_dev)
        ms_fwd_eval = timed(lambda: net(lr_dev), fwd_iters) / fwd_iters
    net.train()

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    burst, sustained, how = measured_peaks()
    achieved = iplan.flops_fwd / (ms_fwd * 1e-3) / 1e12
    step_tflops = (plan.flops_fwd + plan.flops_bwd) / (ms_step * 1e-3) / 1e12
    traffic = None
    tp = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tp):
        try:
            traffic = json.load(open(tp)).get("conv3x3_chain_kernel_bytes_per_launch")
        except Exception:
            traffic = None
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
        "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16",
        "data": "synthetic",
        "config": bench_config(world),
        "step_tflops": step_tflops, "step_frac_of_peak": step_tflops / burst,
        "infer_out_mpix_per_s": world * BATCH_PER_GPU * (LR_HW * SCALE) ** 2 / (ms_fwd_eval * 1e-3) / 1e6,
        "roofline": {"bound": "tensor", "kernel": "conv3x3_chain_kernel (the whole forward pass = 1 launch, 351 conv layers = 2.3497 TFLOP algorithmic)", "achieved": achieved,
                     "peak": burst, "unit": "TFLOP/s", "frac": achieved / burst, "frac_of_sustained": achieved / sustained,
                     "peak_source": how, "traffic": traffic, "ms_forward": ms_fwd},
        "e2e": {"value": e2e_value, "unit": UNIT, "ms_per_step": ms_e2e,
                "readback": "every step's loss copied device -> pinned host behind its backward pass, read by the host one step later (last one before the closing timestamp)",
                "sync_readback": {"value": world * BATCH_PER_GPU / (ms_e2e_sync * 1e-3), "ms_per_step": ms_e2e_sync, "readback": "blocking loss.item() every step"},
                "h2d_bytes_per_step": int(lr_host.numel() * 4 + gt_host.numel() * 4), "d2h_bytes_per_step": 4},
        # kernels of libb200sr.so launched inside the timed region (chain / wgrad / bias-grad / ingest / unpack / add); with the
        # data-parallel bucket hook (N > 1) the gradient unpack runs once per bucket instead of once per step
        "gpu_launches": int((plan.launches_fwd + (plan.launches_bwd_bucketed if bucketed else plan.launches_bwd)) * args.steps),
        "clocks": clocks,
    }
    if dp_err is not None:
        line["dp_equiv_rel_l2"] = dp_err
    if world == 1 and not args.no_library_baseline:
        line["library_baseline"] = library_baseline(net, lr_dev, gt_dev)
        if line["library_baseline"].get("best"):
            line["vs_library_best"] = value / line["library_baseline"]["best"]
    if world == 1 and not args.no_widened:
        line["widened"] = widened_components(dev)
    if world == 1 and not args.no_cpu_baseline:
        del net
        torch.cuda.empty_cache()
        cb = cpu_full_batch(1, 2)  # same method as the --impl reference arm: the full 16-image batch, 2 timed steps
        cb.pop("sec_per_step"); cb.pop("batch")
        line["cpu_baseline"] = cb
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


# ------------------------------------------------------------------------------------- config 4: large-frame inference
def run_c4(args):
    """BASELINE.json configs[3]: ONE 3x1024x1024 LR frame -> 4096x4096 SR, halo-tiled across the ranks (row bands, no
    collective on the data path; ESRGAN/inference.py:68-69 runs the whole frame in one call).  Every rank super-resolves its
    band(s) with `--halo` extra LR rows on interior edges; the HR rows are then gathered on rank 0.  Reports output Mpix/s
    (compute only, max over ranks, and including the gather) and the rel-L2 of the stitched frame against the whole frame."""
    import torch
    import torch.distributed as dist
    import sr_gan_fd_b200 as b200
    from sr_gan_fd_b200 import tile

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    torch.manual_seed(0)
    net = b200.rrdbnet_x4(num_blocks=NUM_BLOCKS)
    # in-range weights (same transformation as the test fixture, restated here: bench does not import oracle/ on this path)
    sd = net.state_dict()
    with torch.no_grad():
        for k in ("conv1.weight", "conv2.weight", "upsampling1.0.weight", "upsampling2.0.weight", "conv3.0.weight", "conv4.weight"):
            sd[k].mul_(3.7)
        sd["conv4.bias"].fill_(0.5)
    net = net.to(dev).eval()
    H = W = args.frame
    g = torch.Generator().manual_seed(4)
    lr = torch.rand(1, 3, H, W, generator=g).to(dev)
    bands = world * args.bands_per_rank
    out_rows = H * SCALE

    out_buf = torch.zeros((1, 3, out_rows, W * SCALE), dtype=torch.float32, device=dev) if bands > 1 else None

    def compute():
        with torch.no_grad():
            if bands == 1:
                return net(lr), (0, out_rows)
            return tile.tiled_forward(net, lr, SCALE, bands, args.halo, rank, world, out=out_buf)

    def gather(out, rows):
        if world == 1:
            return out
        mine = out[:, :, rows[0]:rows[1]].contiguous()
        parts = [torch.empty_like(mine) for _ in range(world)] if rank == 0 else None  # equal bands: H divisible by bands
        dist.gather(mine, parts, dst=0)
        return torch.cat(parts, 2) if rank == 0 else None

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(max(args.warmup, 3)):
        o, rows = compute()
        full = gather(o, rows)
    sampler = ClockSampler(local_rank) if rank == 0 else None
    if sampler:
        sampler.start()
    times = {}
    for name, with_gather in (("compute", False), ("with_gather", True)):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(args.steps):
            o, rows = compute()
            if with_gather:
                full = gather(o, rows)
        e1.record()
        barrier()
        ms = e0.elapsed_time(e1) / args.steps
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        times[name] = ms
    clocks = sampler.stop() if sampler else None
    err = None
    if rank == 0:
        with torch.no_grad():
            whole = net(lr)
        if full is not None and bands > 1:
            err = float(((full.double() - whole.double()).norm() / whole.double().norm()).item())
        del whole
    if rank == 0:
        mpix = out_rows * W * SCALE / 1e6
        plan = net._runtime().last_plan
        burst, sustained, how = measured_peaks()
        flops_frame = 35.853696e6 * H * W  # algorithmic: 35.854 MFLOP per LR pixel (SURVEY 8d), no credit for the halo rows
        line = {
            "metric": "RRDBNet x4 output Mpix/s (BASELINE configs[3]: 1x3x%dx%d LR -> %dx%d SR, halo-tiled inference)" % (H, W, out_rows, W * SCALE),
            "value": mpix / (times["compute"] * 1e-3), "unit": "Mpix/s", "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": times["compute"], "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": {"workload": "config 4 large-frame inference", "bands": bands, "halo_lr_rows": args.halo,
                       "redundant_rows_fraction": tile.redundant_fraction(H, bands, args.halo) if bands > 1 else 0.0,
                       "l2_policy": "one frame's activations (>10 GB workspace traffic) are far larger than L2"},
            "with_gather": {"value": mpix / (times["with_gather"] * 1e-3), "unit": "Mpix/s", "ms_per_step": times["with_gather"]},
            "tiled_vs_whole_rel_l2": err,
            "frac_of_peak": flops_frame / (times["compute"] * 1e-3) / 1e12 / (burst * world),
            "gpu_launches": int(plan.launches_fwd * args.bands_per_rank * args.steps * 2), "clocks": clocks,
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-library-baseline", action="store_true")
    ap.add_argument("--no-widened", action="store_true", help="skip the short section-8(f) component timings (discriminator, GAN step)")
    ap.add_argument("--workload", default="train", choices=["train", "c4"],
                    help="train: the contract's workload (configs[1]/[2]); c4: large-frame halo-tiled inference (configs[3])")
    ap.add_argument("--frame", type=int, default=1024)
    ap.add_argument("--halo", type=int, default=16)
    ap.add_argument("--bands-per-rank", type=int, default=1)
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one computed to DIR/{sr,loss,grad_sample}.npy (see dump_outputs); "
                         "the inputs are seeded, so two builds run with the same arguments can be compared output for output")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl != "b200" or args.workload != "train"):
        ap.error("--dump-outputs applies to the train workload of --impl b200")
    if args.gpus > 1 and "WORLD_SIZE" not in os.environ:
        # convenience: the driver launches N>1 through torch.distributed.run itself; do the same when run by hand
        os.execvp(sys.executable, [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={args.gpus}",
                                   "--master-addr", "127.0.0.1", "--master-port", "29533", os.path.abspath(__file__)] + sys.argv[1:])
    if args.impl == "reference":
        run_reference(args)
    elif args.workload == "c4":
        run_c4(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
