"""Packed dense-block weight gradients (B200SR_WGRAD_PACK) against the unpacked problem list.

Both forms multiply the same bf16 operands and sum the products in fp32, only in another order (other pixel-split counts, other
``red.global.add`` interleavings), so every weight and bias gradient must agree to fp32 reordering noise.  The switch is read once
per process: each mode runs in a subprocess of its own (this file is also that worker) and saves its gradients.

* config 2 (16 x 64x64 LR, 23 RRDB) and an edge shape (one image, 20 x 12 LR: a partial 16-row pixel tile in y and a partial
  8-column tile in x, 2 RRDB): per-tensor relative L2 of every parameter gradient <= 1e-4 between the modes.  Two floors are
  printed beside it: the unpacked form run twice (same pixel splits, only the atomic order differs) and the unpacked form with all
  SMs per launch instead of half (other pixel-split counts: the kind of reordering packing causes).  At config 2 a dense-block
  weight gradient sums 65536 pixels of products with random signs, an HR-tail one a million, so reordering alone moves a tensor by
  up to about 1e-4 (B200: packed vs unpacked 2.0e-5, unpacked with other splits 1.2e-4 on conv4); a dropped, doubled or
  mis-tapped 128-pixel tile moves it by 1e-2 or more.
* the edge-shape net in every mode against the fp32 CPU oracle, within the flat-gradient bar of test_model_gpu.py (1e-2).
"""
import os
import subprocess
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CASES = {"config2": (23, (16, 3, 64, 64)), "edge": (2, (1, 3, 20, 12))}
TOL_MODE, TOL_GRAD = 1e-4, 1e-2


def _inputs(shape):
    g = torch.Generator().manual_seed(1)
    lr = torch.rand(*shape, generator=g)
    gt = torch.rand(shape[0], 3, shape[2] * 4, shape[3] * 4, generator=g)
    return lr, gt


def _params(num_blocks):
    import sr_gan_fd_b200 as b200
    torch.manual_seed(0)
    return {k: v.detach().clone() for k, v in b200.rrdbnet_x4(num_blocks=num_blocks).state_dict().items()}


def _worker(out_path):
    """One L1 training step per case on cuda:0; saves {case: {name: grad}}."""
    import torch.nn.functional as F
    import sr_gan_fd_b200 as b200
    dev = torch.device("cuda", 0)
    res = {}
    for case, (nb, shape) in CASES.items():
        params = _params(nb)
        net = b200.rrdbnet_x4(num_blocks=nb)
        net.load_state_dict(params)
        net = net.to(dev).train()
        lr, gt = _inputs(shape)
        F.l1_loss(net(lr.to(dev)), gt.to(dev)).backward()
        res[case] = {n: p.grad.detach().cpu().clone() for n, p in net.named_parameters()}
        del net
        torch.cuda.synchronize()
    torch.save(res, out_path)


def _run_mode(tmp_path, tag, env_extra):
    out = tmp_path / f"{tag}.pt"
    env = dict(os.environ, PYTHONDONTWRITEBYTECODE="1", **env_extra)
    r = subprocess.run([sys.executable, os.path.abspath(__file__), str(out)], cwd=tmp_path, env=env, capture_output=True, text=True,
                       timeout=900)
    assert r.returncode == 0, r.stdout[-2000:] + "\n" + r.stderr[-3000:]
    return torch.load(out)


def _rel_l2(a, b):
    d = float((a.double() - b.double()).norm())
    n = float(b.double().norm())
    return d / n if n > 0 else d


@pytest.mark.gpu
def test_packed_wgrad_matches_unpacked(tmp_path):
    from oracle import rrdbnet_oracle as orc
    base = _run_mode(tmp_path, "pack0", {"B200SR_WGRAD_PACK": "0"})
    again = _run_mode(tmp_path, "pack0_again", {"B200SR_WGRAD_PACK": "0"})
    resplit = _run_mode(tmp_path, "pack0_all_sms", {"B200SR_WGRAD_PACK": "0", "B200SR_WGRAD_SMS": str(torch.cuda.get_device_properties(0).multi_processor_count)})
    packed = _run_mode(tmp_path, "pack1", {"B200SR_WGRAD_PACK": "1"})
    for case in CASES:
        names = list(base[case].keys())
        floor = max((_rel_l2(again[case][n], base[case][n]), n) for n in names)
        floor_split = max((_rel_l2(resplit[case][n], base[case][n]), n) for n in names)
        worst = max((_rel_l2(packed[case][n], base[case][n]), n) for n in names)
        dense = max((_rel_l2(packed[case][n], base[case][n]), n) for n in names if n.startswith("trunk."))
        print(f"{case}: worst per-tensor rel-L2 packed vs unpacked {worst[0]:.3e} ({worst[1]}; dense blocks {dense[0]:.3e}), "
              f"unpacked vs unpacked {floor[0]:.3e} ({floor[1]}), other pixel splits {floor_split[0]:.3e} ({floor_split[1]})")
        assert worst[0] <= TOL_MODE, (case, worst, floor)
        for n in names:  # the packed form covers every weight and bias exactly once: no tensor may be left at zero
            assert (float(packed[case][n].norm()) > 0) == (float(base[case][n].norm()) > 0), (case, n)

    nb, shape = CASES["edge"]
    params = _params(nb)
    lr, gt = _inputs(shape)
    _, _, grads_ref = orc.rrdbnet_l1_step(params, lr, gt)
    flat_ref = torch.cat([g.flatten() for g in grads_ref.values()])
    for tag, res in (("pack0", base), ("pack1", packed)):
        flat = torch.cat([res["edge"][n].flatten() for n in grads_ref.keys()])
        err = orc.rel_l2(flat, flat_ref)
        print(f"edge shape, {tag}: flat gradient rel-L2 vs fp32 oracle {err:.3e}")
        assert err <= TOL_GRAD, (tag, err)


if __name__ == "__main__":
    sys.path.insert(0, ROOT)
    _worker(sys.argv[1])
