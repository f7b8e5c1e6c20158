"""CPU: the oracle restatement is pinned (a) against the committed golden fixtures that oracle/make_golden.py produced
by executing the reference's own model.py, and (b) -- when /root/reference is present (build container) -- against the
reference classes directly, bit-equal in fp32."""
import glob
import os

import pytest
import torch
import torch.nn.functional as F

from oracle import make_golden
from oracle import reference_loader as rl
from oracle import rrdbnet_oracle as orc

GOLDEN = sorted(glob.glob(os.path.join(os.path.dirname(__file__), "golden", "*.pt")))


@pytest.fixture
def golden_threads():
    """the thread count the fixtures were computed with (bit equality depends on it), whatever the host or an earlier test set"""
    n = torch.get_num_threads()
    torch.set_num_threads(make_golden.THREADS)
    yield
    torch.set_num_threads(n)


def _drop_in(fix):
    import sr_gan_fd_b200 as b200
    torch.manual_seed(fix["seed"])
    if fix["flavour"] == "esrgan":
        net = b200.RRDBNet(3, 3, 64, 32, fix["num_blocks"], fix["scale"])
    elif fix["flavour"] == "bsrgan":
        net = b200.BSRGAN(3, 3, 64, 32, fix["num_blocks"], fix["scale"])
    else:
        net = b200.RealRRDBNet(3, 3, 64, 32, fix["num_blocks"], fix["scale"])
    params = {k: v.detach().clone() for k, v in net.state_dict().items()}
    if fix["in_range"]:
        params = orc.in_range_fixture(params)
    return net, params


@pytest.mark.usefixtures("golden_threads")
@pytest.mark.parametrize("path", GOLDEN, ids=[os.path.basename(p) for p in GOLDEN])
def test_oracle_matches_golden(path):
    """seed + drop-in constructor reproduces the reference weights; oracle forward/backward reproduce the reference
    output, loss and gradients stored in the fixture (bit-equal: same ATen CPU kernels, same op order)."""
    fix = torch.load(path)
    _, params = _drop_in(fix)
    assert abs(float(sum(v.double().sum() for v in params.values())) - fix["param_checksum"]) < 1e-9
    assert abs(float(sum(v.double().abs().sum() for v in params.values())) - fix["param_abs_checksum"]) < 1e-9
    sr, loss, grads = orc.rrdbnet_l1_step(params, fix["lr"], fix["gt"])
    assert torch.equal(sr, fix["sr"])
    assert torch.equal(loss, fix["loss"])
    for k, g in fix["grads"].items():
        assert torch.allclose(grads[k], g, rtol=1e-5, atol=1e-9), k
    for k, nrm in fix["grad_norms"].items():
        assert abs(float(grads[k].double().norm()) - nrm) <= 1e-5 * max(nrm, 1e-12), k


@pytest.mark.skipif(not rl.available(), reason="reference tree not present (GPU box)")
@pytest.mark.parametrize("flavour,scale", [("esrgan", 4), ("esrgan", 2), ("esrgan", 8), ("esrgan", 1), ("bsrgan", 2),
                                           ("bsrgan", 4), ("real", 4), ("real", 2), ("aesrgan", 2)])
def test_oracle_bit_equal_to_reference(flavour, scale):
    torch.manual_seed(0)
    ref = rl.build_generator(flavour, scale, 2, channels=16, growth=8)
    params = {k: v.detach() for k, v in ref.state_dict().items()}
    pu = {2: 2, 1: 4}.get(scale, 1) if flavour == "real" else 1
    for shape, train in [((2, 3, 12 * pu, 8 * pu), False), ((1, 3, 7 * pu, 9 * pu), True)]:
        x = torch.rand(*shape)
        ref.train(train)
        with torch.no_grad():
            y_ref = ref(x)
        y = orc.rrdbnet_forward(params, x, pixel_unshuffle=pu)
        assert torch.equal(y, y_ref)


@pytest.mark.skipif(not rl.available(), reason="reference tree not present (GPU box)")
@pytest.mark.parametrize("flavour,kw", [("esrgan", dict(upscale_factor=4)), ("esrgan", dict(upscale_factor=8)),
                                        ("bsrgan", dict(upscale_factor=2)), ("real", dict(upscale_factor=4)),
                                        ("real", dict(upscale_factor=2))])
def test_drop_in_state_dict_and_init_equal_reference(flavour, kw):
    """Same state_dict keys / order / shapes / dtypes and -- under the same seed -- the same initial values."""
    import sr_gan_fd_b200 as b200
    torch.manual_seed(0)
    ref = rl.build_generator(flavour, kw["upscale_factor"], 2)
    torch.manual_seed(0)
    cls = {"esrgan": b200.RRDBNet, "bsrgan": b200.BSRGAN, "real": b200.RealRRDBNet}[flavour]
    mine = cls(3, 3, 64, 32, 2, kw["upscale_factor"])
    a, b = ref.state_dict(), mine.state_dict()
    assert list(a.keys()) == list(b.keys())
    for k in a:
        assert a[k].shape == b[k].shape and a[k].dtype == b[k].dtype
        assert torch.equal(a[k], b[k]), k
    assert [n for n, _ in ref.named_parameters()] == [n for n, _ in mine.named_parameters()]
    assert len(list(mine.buffers())) == len(list(ref.buffers())) == 0


def test_flop_model_matches_baseline_md():
    assert orc.flops_per_lr_pixel() == 35_853_696
    assert orc.flops_per_lr_pixel(backward=True) == 71_703_936
    assert orc.flops_per_lr_pixel(n_up=1) == 33_747_840 + 0  # BSRGAN x2 forward (SURVEY.md section 8a)


def test_iqa_restatement_sanity():
    a = torch.rand(2, 3, 40, 40)
    assert torch.all(orc.psnr_y(a, a) > 90)
    assert torch.allclose(orc.ssim_y(a, a), torch.ones(2))
    b = (a + 0.05 * torch.randn_like(a)).clamp(0, 1)
    assert torch.all(orc.psnr_y(b, a) < 40) and torch.all(orc.ssim_y(b, a) < 1)


@pytest.mark.skipif(not rl.available(), reason="reference tree not present (GPU box)")
def test_iqa_matches_reference():
    iqa = rl.load_module("esrgan", "image_quality_assessment")
    a, b = torch.rand(2, 3, 48, 40), torch.rand(2, 3, 48, 40)
    assert torch.allclose(iqa.PSNR(4, True)(a, b), orc.psnr_y(a, b), rtol=0, atol=1e-9)
    assert torch.allclose(iqa.SSIM(4, True)(a, b), orc.ssim_y(a, b), rtol=0, atol=1e-6)
