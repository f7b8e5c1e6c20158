"""CPU: what a deterministic plan (torch.use_deterministic_algorithms) changes, counted on the plan.  Same packing, a larger
workspace (the partial-sum lanes) and one ordered-sum launch behind every weight- and bias-gradient launch.  The GPU side
(bit-identical repeats, accuracy against the default mode) is in test_deterministic_gpu.py."""
import ctypes as C

import pytest
import torch

import sr_gan_fd_b200 as b200
from sr_gan_fd_b200 import lib as _lib
from sr_gan_fd_b200.discriminator import _DiscPlan, _DiscRuntime, discriminator_unet
from sr_gan_fd_b200.function import GeneratorRuntime, _Plan
from sr_gan_fd_b200.vgg import _VggRuntime

from test_partial_grad_host import GEOMETRIES, flags

PATTERNS = ["all", "head+half", "tail", "conv4", "one_conv", "no_bias"]


@pytest.fixture(scope="module", autouse=True)
def _built():
    from sr_gan_fd_b200.build import build_native
    build_native()


def reductions(net, pattern) -> int:
    """Weight- and bias-gradient launches of a generator backward under a freeze pattern (each gets one ordered sum)."""
    names = [n for n, _ in net.named_parameters()]
    want = {n.rsplit(".", 1)[0] for n, f in zip(names, flags(net, pattern)) if f}  # conv module names with a wanted parameter
    n = 0
    for conv in dict.fromkeys(n.rsplit(".", 1)[0] for n in names):
        if conv not in want:
            continue
        if conv.startswith("trunk."):
            continue  # counted per dense block below
        # conv1, conv2, conv3, conv4: one weight- and one bias-gradient launch; an upsample conv: two weight halves and a bias launch
        n += 3 if conv.startswith("upsampling") else 2
    blocks = {c.rsplit(".", 1)[0] for c in want if c.startswith("trunk.")}  # trunk.i.rdbj: one launch for its five convs
    return n + len(blocks)


def test_version_and_descriptor_fields():
    assert _lib.load().b200sr_version() >= 101
    for desc in (_lib.NetDesc, _lib.DiscDesc, _lib.VggDesc):
        assert desc._fields_[-1] == ("deterministic", C.c_int32)
    # positional construction without the last member leaves it zero (the default mode)
    assert _lib.NetDesc(3, 3, 64, 32, 1, 2, 1, 8, 8, 1, 0).deterministic == 0


@pytest.mark.parametrize("factory,nb,geo", GEOMETRIES, ids=[f"{f}-{nb}-{'x'.join(map(str, g))}" for f, nb, g in GEOMETRIES])
def test_generator_plan_shares_packing_and_counts_the_ordered_sums(factory, nb, geo):
    net = getattr(b200, factory)(num_blocks=nb)
    ref = _Plan(net.net_desc(), *geo, True, 0, False)
    det = _Plan(net.net_desc(), *geo, True, 0, True)
    assert det.pack_layout == ref.pack_layout
    assert det.packed_bytes == ref.packed_bytes
    assert det.param_numel == ref.param_numel and det.num_params == ref.num_params
    assert det.workspace_bytes > ref.workspace_bytes
    assert det.launches_fwd == ref.launches_fwd
    full = reductions(net, "all")
    assert det.launches_bwd == ref.launches_bwd + full
    assert det.launches_bwd_bucketed == ref.launches_bwd_bucketed + full
    for pattern in PATTERNS:
        fl = flags(net, pattern)
        for dx in (False, True):
            assert det.backward_launches(fl, with_dx=dx) == ref.backward_launches(fl, with_dx=dx) + reductions(net, pattern), (pattern, dx)
    frozen = flags(net, "frozen")
    assert det.backward_launches(frozen) == 0
    assert det.backward_launches(frozen, with_dx=True) == ref.backward_launches(frozen, with_dx=True)


def test_generator_inference_plan_is_unchanged():
    net = b200.rrdbnet_x4(num_blocks=2)
    ref = _Plan(net.net_desc(), 2, 24, 20, False, 0, False)
    det = _Plan(net.net_desc(), 2, 24, 20, False, 0, True)
    assert (det.workspace_bytes, det.packed_bytes, det.pack_layout, det.launches_fwd) == \
        (ref.workspace_bytes, ref.packed_bytes, ref.pack_layout, ref.launches_fwd)


@pytest.mark.parametrize("fp16,geo", [(True, (16, 256, 256)), (False, (2, 64, 64))])
def test_discriminator_plan_counts_the_ordered_sums(fp16, geo):
    lib = _lib.load()
    ref = _DiscPlan(3, 1, 64, *geo, True, fp16, False)
    det = _DiscPlan(3, 1, 64, *geo, True, fp16, True)
    assert det.packed_bytes == ref.packed_bytes and det.param_numel == ref.param_numel
    assert lib.b200sr_pack_layout_id(det.handle) == lib.b200sr_pack_layout_id(ref.handle)
    assert det.workspace_bytes > ref.workspace_bytes
    assert lib.b200sr_num_launches(det.handle, 0) == lib.b200sr_num_launches(ref.handle, 0)
    # weight-gradient launches of the 64-channel U-Net (four 128 x 128 problems per launch): 1 each for conv4, conv3, conv2,
    # up3, up2, conv1, 2 for up1, 8 for down3, 2 for down2, 1 for down1 = 19; bias gradients of conv1 and conv4 = 2
    assert lib.b200sr_num_launches(det.handle, 1) == lib.b200sr_num_launches(ref.handle, 1) + 21


def test_vgg_plan_has_a_partial_sum_area_and_the_same_packing():
    lib = _lib.load()
    rt = _VggRuntime()
    mean, std = [0.485, 0.456, 0.406], [0.229, 0.224, 0.225]
    ref = rt.plan(4, 32, 32, 15, (1 << 15) | (1 << 8), 15, 2, mean, std, False)
    det = rt.plan(4, 32, 32, 15, (1 << 15) | (1 << 8), 15, 2, mean, std, True)
    assert det is not ref
    assert det["layout"] == ref["layout"] and det["packed_bytes"] == ref["packed_bytes"]
    assert det["ws_bytes"] > ref["ws_bytes"]
    assert lib.b200sr_num_launches(det["handle"], 1) == lib.b200sr_num_launches(ref["handle"], 1)


def test_iqa_scratch_covers_every_crop():
    lib = _lib.load()
    n, h, w = 3, 96, 80
    full = int(lib.b200sr_iqa_det_scratch_bytes(n, h, w))
    assert full > 0
    for crop in (0, 4, 20):
        assert int(lib.b200sr_iqa_det_scratch_bytes(n, h - 2 * crop, w - 2 * crop)) <= full


def test_python_plan_keys_tell_the_modes_apart():
    net = b200.rrdbnet_x4(num_blocks=1)
    rt = GeneratorRuntime()
    dev = torch.device("cuda", 0)
    a = rt.plan(net.net_desc(), dev, 1, 16, 16, True, False)
    b = rt.plan(net.net_desc(), dev, 1, 16, 16, True, True)
    assert a is not b and b.deterministic and not a.deterministic
    assert rt.plan(net.net_desc(), dev, 1, 16, 16, True, False) is a
    assert rt.plan(net.net_desc(), dev, 1, 16, 16, True, True) is b
    # the discriminator reads the torch flag (with or without warn_only) when it picks its plan
    disc = discriminator_unet(in_channels=3, out_channels=1, channels=64)
    drt = _DiscRuntime()
    prev = torch.are_deterministic_algorithms_enabled(), torch.is_deterministic_algorithms_warn_only_enabled()
    try:
        torch.use_deterministic_algorithms(False)
        p0 = drt.plan(disc, dev, 1, 16, 16, True)
        torch.use_deterministic_algorithms(True, warn_only=True)
        p1 = drt.plan(disc, dev, 1, 16, 16, True)
        torch.use_deterministic_algorithms(True)
        assert drt.plan(disc, dev, 1, 16, 16, True) is p1
    finally:
        torch.use_deterministic_algorithms(prev[0], warn_only=prev[1])
    assert p0 is not p1 and p1.deterministic and not p0.deterministic
