"""Generates tests/golden/*.pt by EXECUTING the unmodified reference generator classes from /root/reference
(build container only).  The fixtures travel to the GPU box, where the reference tree does not exist.

    PYTHONDONTWRITEBYTECODE=1 python -m oracle.make_golden

Each fixture: seed, constructor kwargs, the LR input, the reference SR output, the L1 loss against a stored GT and a
selection of parameter gradients (full tensors for a few layers + the norm of every gradient tensor).  Weights are NOT
stored: ``torch.manual_seed(seed)`` + the constructor reproduces them (the fixture stores a checksum to prove it).
"""
import os
import sys

import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import reference_loader as rl  # noqa: E402
from oracle import rrdbnet_oracle as orc  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden")
# intra-op threads of torch's CPU kernels the fixtures are computed with: fp32 sums (oneDNN convolutions, bias gradients) are split
# by thread count, so the oracle reproduces the fixtures bit for bit only at this count
THREADS = 8
KEEP = ["conv1.weight", "conv1.bias", "trunk.0.rdb1.conv1.weight", "trunk.0.rdb2.conv3.bias", "trunk.0.rdb3.conv5.bias",
        "conv2.bias", "upsampling1.0.bias", "conv3.0.bias", "conv4.weight", "conv4.bias"]

CASES = [
    # name, flavour, scale, blocks, shape, in_range
    ("esrgan_x4_b1", "esrgan", 4, 1, (1, 3, 24, 20), True),
    ("esrgan_x4_b1_rand", "esrgan", 4, 1, (2, 3, 16, 16), False),
    ("bsrgan_x2_b1", "bsrgan", 2, 1, (1, 3, 19, 13), True),
    ("real_x4_b1", "real", 4, 1, (1, 3, 17, 9), True),
    # the full 23-RRDB depth of every BASELINE config (round 2)
    ("esrgan_x4_b23", "esrgan", 4, 23, (2, 3, 32, 32), True),
]


def main():
    os.makedirs(OUT, exist_ok=True)
    only = set(sys.argv[1:])  # optional: names of the cases to (re)generate
    for name, flavour, scale, blocks, shape, in_range in CASES:
        if only and name not in only:
            continue
        torch.manual_seed(0)
        net = rl.build_generator(flavour, scale, blocks)
        params = {k: v.detach().clone() for k, v in net.state_dict().items()}
        if in_range:
            params = orc.in_range_fixture(params)
            net.load_state_dict(params)
        g = torch.Generator().manual_seed(42)
        lr = torch.rand(*shape, generator=g)
        gt = torch.rand(shape[0], 3, shape[2] * scale, shape[3] * scale, generator=g)
        net.train()
        sr = net(lr)
        loss = F.l1_loss(sr, gt)
        loss.backward()
        grads = {k: p.grad.detach().clone() for k, p in net.named_parameters()}
        fix = {
            "flavour": flavour, "scale": scale, "num_blocks": blocks, "in_range": in_range, "seed": 0,
            "lr": lr, "gt": gt, "sr": sr.detach().clone(), "loss": loss.detach().clone(),
            "grads": {k: grads[k] for k in KEEP if k in grads},
            "grad_norms": {k: float(v.double().norm()) for k, v in grads.items()},
            "param_checksum": float(sum(v.double().sum() for v in params.values())),
            "param_abs_checksum": float(sum(v.double().abs().sum() for v in params.values())),
            "torch_version": str(torch.__version__),
        }
        torch.save(fix, os.path.join(OUT, name + ".pt"))
        print(name, "sr mean", float(sr.detach().mean()), "loss", float(loss.detach()), os.path.getsize(os.path.join(OUT, name + ".pt")) // 1024, "KiB")


DISC_KEEP = ["conv1.weight", "conv1.bias", "conv3.0.weight_orig", "conv4.weight", "conv4.bias"]


def main_disc():
    """tests/golden/disc/*.pt: the reference DiscriminatorUNet (BSRGAN/model.py:91-167) executed on a seeded input."""
    out = os.path.join(OUT, "disc")
    os.makedirs(out, exist_ok=True)
    m = rl.load_module("bsrgan")
    for name, seed, shape in [("disc_unet_s0", 0, (2, 3, 32, 40))]:
        torch.manual_seed(seed)
        net = m.DiscriminatorUNet(3, 1, 64)
        params = {k: v.detach().clone() for k, v in net.state_dict().items()}
        g = torch.Generator().manual_seed(42)
        x = torch.rand(*shape, generator=g)
        dy = torch.randn(shape[0], 1, shape[2], shape[3], generator=g)
        net.train()
        xr = x.clone().requires_grad_(True)
        y = net(xr)
        y.backward(dy)
        grads = {k: p.grad.detach().clone() for k, p in net.named_parameters()}
        after = net.state_dict()
        fix = {
            "seed": seed, "x": x, "dy": dy, "y": y.detach().clone(), "dx": xr.grad.detach().clone(),
            "grads": {k: grads[k] for k in DISC_KEEP},
            "grad_norms": {k: float(v.double().norm()) for k, v in grads.items()},
            "buffers": {k: after[k].detach().clone() for k in after if k.endswith(("weight_u", "weight_v"))},
            "param_checksum": float(sum(v.double().sum() for v in params.values())),
            "torch_version": str(torch.__version__),
        }
        torch.save(fix, os.path.join(out, name + ".pt"))
        print(name, "logit mean", float(y.detach().mean()), os.path.getsize(os.path.join(out, name + ".pt")) // 1024, "KiB")


if __name__ == "__main__":
    torch.set_num_threads(THREADS)
    if "disc" in sys.argv[1:]:
        main_disc()
    else:
        main()
