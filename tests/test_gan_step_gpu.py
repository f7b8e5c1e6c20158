"""BASELINE configs[4] harness check (1 GPU): one BSRGAN GAN iteration (``BSRGAN/train_bsrgan.py:412-470``) with a
``DiscriminatorUNet`` and a ``ContentLoss`` (seeded random-init VGG19 patched into torchvision: no ImageNet weights offline),
a discriminator optimizer step BETWEEN the generator's forward and backward, and the generator backward under the summed
(20 x L1 + 1 x content + 0.5 x adversarial) x 65536 upstream gradient.  The generator's parameter gradients must match the fp32
oracle driven by the SAME upstream gradient.  The critics are the reference's own classes where its tree is present
($SRGANFD_REFERENCE), else the drop-in critics through their stock torch paths -- the reference's op sequences (the
discriminator's pinned against it by tests/golden/disc).  A log of a run on a B200 with the reference's critics is kept in
profiles/r2_gan_step_test.log."""
import os
import sys

import pytest
import torch

from oracle import rrdbnet_oracle as orc

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
from sr_gan_fd_b200.compat._passthrough import reference_root
# $SRGANFD_REFERENCE, /root/reference (build container), or -- on the GPU box -- the unmodified copy staged by
# __graft_entry__.stage_reference() under baseline/_ref (git-ignored, travels with the snapshot)
REF = reference_root()
os.environ["SRGANFD_REFERENCE"] = REF
CRITICS = "reference" if os.path.isfile(os.path.join(REF, "BSRGAN", "model.py")) else "torch"
pytestmark = pytest.mark.gpu


def test_generator_gradients_inside_the_gan_step():
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    import gan_step
    dev = torch.device("cuda", 0)
    d_model, g_model, content = gan_step.build("b200", dev, seed=0, content=CRITICS, disc=CRITICS)
    d_model.train(); g_model.train()
    params = {k: v.detach().cpu().clone() for k, v in g_model.state_dict().items()}
    params = orc.in_range_fixture(params)
    g_model.load_state_dict(params)
    step = gan_step.GanStep(d_model, g_model, content, dev)
    g = torch.Generator().manual_seed(8)
    lr = torch.rand(4, 3, 32, 32, generator=g)
    gt = torch.rand(4, 3, 128, 128, generator=g)
    d_before = [p.detach().clone() for p in d_model.parameters()]
    sr, g_loss, d_loss = step(lr.to(dev), gt.to(dev), step_d=True, step_g=False, keep_sr_grad=True)
    assert any(not torch.equal(a, b) for a, b in zip(d_before, d_model.parameters())), "the discriminator step did not happen"
    dy = step.sr_grad.float().cpu()
    assert float(dy.abs().max()) > 1.0  # carries the GradScaler's 65536
    leaves = {k: v.clone().requires_grad_(True) for k, v in params.items()}
    sr_ref = orc.rrdbnet_forward(leaves, lr)
    assert orc.rel_l2(sr.detach().float().cpu(), sr_ref.detach()) <= 5e-3
    ref = torch.autograd.grad(sr_ref, list(leaves.values()), grad_outputs=dy)
    got = [p.grad.detach().float().cpu() for p in g_model.parameters()]
    flat, flat_ref = torch.cat([t.flatten() for t in got]), torch.cat([t.flatten() for t in ref])
    err = orc.rel_l2(flat, flat_ref)
    print(f"GAN step: generator flat-grad rel-L2 vs oracle {err:.3e} (|dy|max {float(dy.abs().max()):.3g}, g_loss {float(g_loss):.4f}, d_loss {float(d_loss):.4f})")
    assert torch.isfinite(flat).all() and err <= 1e-2, err
