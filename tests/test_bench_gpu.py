"""bench.py on the GPU at a few steps: the JSON line reports the number of timed steps asked for, and ``--dump-outputs`` writes what
the last timed step computed -- checked against the fp32 CPU oracle on the inputs bench.py seeds, with the tolerances of
test_model_gpu.py (SR rel-L2 <= 5e-3, gradient rel-L2 <= 1e-2)."""
import importlib.util
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from oracle import rrdbnet_oracle as orc

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.gpu
def test_dump_outputs_hold_the_last_timed_step(tmp_path):
    spec = importlib.util.spec_from_file_location("_bench_for_test", os.path.join(ROOT, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    out = tmp_path / "dump"
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", "3", "--warmup", "1",
                        "--no-cpu-baseline", "--no-library-baseline", "--no-widened", "--dump-outputs", str(out)],
                       cwd=tmp_path, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-2000:] + "\n" + r.stderr[-3000:]
    assert json.loads(r.stdout.strip().splitlines()[-1])["steps"] == 3
    assert sorted(os.listdir(out)) == ["grad_sample.npy", "loss.npy", "sr.npy"]
    assert sum(os.path.getsize(out / f) for f in os.listdir(out)) <= 64 << 20
    sr, loss, grad = (torch.from_numpy(np.load(out / f"{n}.npy")) for n in ("sr", "loss", "grad_sample"))
    assert sr.dtype == loss.dtype == grad.dtype == torch.float32
    assert sr.shape == (bench.BATCH_PER_GPU, 3, bench.LR_HW * bench.SCALE, bench.LR_HW * bench.SCALE)

    import sr_gan_fd_b200 as b200
    torch.manual_seed(0)
    params = {k: v.detach() for k, v in b200.rrdbnet_x4(num_blocks=bench.NUM_BLOCKS).state_dict().items()}
    lr, gt = bench.seeded_inputs()
    sr_ref, loss_ref, grads_ref = orc.rrdbnet_l1_step(params, lr, gt)
    flat_ref = torch.cat([g.flatten() for g in grads_ref.values()])
    idx = torch.randperm(flat_ref.numel(), generator=torch.Generator().manual_seed(0))[:bench.GRAD_SAMPLE].sort().values
    e_sr, e_grad = orc.rel_l2(sr, sr_ref), orc.rel_l2(grad, flat_ref[idx])
    print(f"bench dump vs fp32 oracle: SR rel-L2 {e_sr:.3e}, sampled gradient rel-L2 {e_grad:.3e}")
    assert e_sr <= 5e-3 and e_grad <= 1e-2
    # the dumped loss is the L1 of the dumped SR batch: it differs from the oracle's by at most their mean distance
    assert abs(float(loss) - float(loss_ref)) <= float((sr - sr_ref).abs().mean()) + 1e-6
