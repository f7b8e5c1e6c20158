"""CPU: what a selective generator backward (b200sr_backward_select) launches for a freeze pattern, counted on the plan.
The GPU side (gradients, profiler launch list) is in test_partial_grad_gpu.py."""
import pytest

import sr_gan_fd_b200 as b200
from sr_gan_fd_b200.function import _Plan


def trainable(name: str, pattern: str, num_blocks: int) -> bool:
    """Whether parameter `name` (state_dict name) is trained under a freeze pattern."""
    if pattern == "all":
        return True
    if pattern == "frozen":
        return False
    if pattern == "tail":  # conv2, upsampling*, conv3, conv4
        return not (name.startswith("conv1.") or name.startswith("trunk."))
    if pattern == "conv4":
        return name.startswith("conv4.")
    if pattern.startswith("head+"):  # conv1 and the first k RRDBs frozen ("head+half": k = num_blocks // 2)
        k = num_blocks // 2 if pattern == "head+half" else int(pattern[5:])
        if name.startswith("conv1."):
            return False
        return not (name.startswith("trunk.") and int(name.split(".")[1]) < k)
    if pattern == "one_conv":  # one conv frozen inside an otherwise trainable dense block
        return not name.startswith(f"trunk.{num_blocks - 1}.rdb2.conv3.")
    if pattern == "no_bias":
        return not name.endswith(".bias")
    raise ValueError(pattern)


def flags(net, pattern):
    nb = len(net.trunk)
    return [trainable(n, pattern, nb) for n, _ in net.named_parameters()]


def _plan(net, batch, h, w, bucket_rrdbs=0):
    return _Plan(net.net_desc(), batch, h, w, True, bucket_rrdbs)


GEOMETRIES = [
    ("rrdbnet_x4", 2, (2, 24, 20)),    # re-associated dense blocks, two image groups
    ("rrdbnet_x1", 2, (2, 16, 16)),    # no tail upsampling
    ("rrdbnet_x8", 1, (1, 16, 12)),    # three upsample stages
    ("rrdbnet_x4", 1, (1, 160, 264)),  # per-conv schedule: one chain for tail and trunk
    ("rrdbnet_x4", 23, (16, 64, 64)),  # config 2
    ("rrdbnet_x4", 23, (64, 64, 64)),  # long trunk chain cut in pieces
]


@pytest.fixture(scope="module", autouse=True)
def _built():
    from sr_gan_fd_b200.build import build_native
    build_native()


@pytest.mark.parametrize("factory,nb,geo", GEOMETRIES, ids=[f"{f}-{nb}-{'x'.join(map(str, g))}" for f, nb, g in GEOMETRIES])
def test_launch_counts_follow_the_freeze_pattern(factory, nb, geo):
    net = getattr(b200, factory)(num_blocks=nb)
    plan = _plan(net, *geo)
    # no mask: exactly the full backward's count; a mask of all ones is the same thing
    assert plan.backward_launches() == plan.launches_bwd
    assert plan.backward_launches(with_cb=True) == plan.launches_bwd_bucketed
    assert plan.backward_launches(flags(net, "all")) == plan.launches_bwd
    assert plan.backward_launches(flags(net, "no_bias")) == plan.launches_bwd  # weights still need every launch
    full = plan.launches_bwd
    head = plan.backward_launches(flags(net, "head+half"))
    tail = plan.backward_launches(flags(net, "tail"))
    conv4 = plan.backward_launches(flags(net, "conv4"))
    assert full > head > tail > conv4 > 0, (full, head, tail, conv4)
    # the input gradient forces the whole walk and the carrier sum, but no weight gradient
    frozen_dx = plan.backward_launches(flags(net, "frozen"), with_dx=True)
    assert 0 < frozen_dx < plan.backward_launches(with_dx=True)
    assert plan.backward_launches(flags(net, "head+half"), with_dx=True) > head
    assert plan.backward_launches(flags(net, "frozen")) == 0
    # one frozen conv inside a trainable dense block: that block's one weight-gradient launch still runs
    assert plan.backward_launches(flags(net, "one_conv")) == full


def test_frozen_generator_with_dx_skips_every_parameter_kernel():
    """config 2 frozen + dx: ingest + the data-gradient chains + the carrier sum + the dx chain, nothing else."""
    net = b200.rrdbnet_x4(num_blocks=23)
    plan = _plan(net, 16, 64, 64)
    assert plan.backward_launches(flags(net, "frozen"), with_dx=True) == 1 + 2 + 1 + 1


def test_buckets_without_wanted_convs_are_not_unpacked():
    """With a bucket callback, every bucket is one unpack launch; a frozen prefix drops the buckets that hold only frozen convs."""
    net = b200.rrdbnet_x4(num_blocks=23)
    plan = _plan(net, 16, 64, 64, bucket_rrdbs=6)
    full_cb, full = plan.backward_launches(with_cb=True), plan.backward_launches()
    head_cb, head = plan.backward_launches(flags(net, "head+12"), with_cb=True), plan.backward_launches(flags(net, "head+12"))
    # the tail, RRDBs 18-22, 12-17, 6-11, 2-5, 0-1 and conv1 are buckets; with conv1 and RRDBs 0-11 frozen three of them are left
    assert full_cb - full == 7 - 1
    assert head_cb - head == 3 - 1
