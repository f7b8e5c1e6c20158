"""CPU: the RRDB trunk as a module of its own (RRDBTrunk / native_trunk) -- trunk plans' sizes, descriptor checks, launch counts per
freeze pattern, adoption of an existing Sequential, and the CPU forward / backward against the oracle restatement.  The GPU side
(bit-identity with the generator's own trunk, oracle bars, freeze patterns, determinism, composed models) is test_trunk_gpu.py."""
import copy
import ctypes as C
import pickle
from collections import OrderedDict

import pytest
import torch
from torch import nn

import sr_gan_fd_b200 as b200
from oracle import rrdbnet_oracle as orc
from sr_gan_fd_b200 import lib as _lib
from sr_gan_fd_b200.function import _Plan

RRDB_PARAMS = 30            # 3 dense blocks x 5 convs x (weight, bias)
RRDB_NUMEL = 719_424        # 3 x (18464 + 27680 + 36896 + 46112 + 110656)


@pytest.fixture(scope="module", autouse=True)
def _built():
    from sr_gan_fd_b200.build import build_native
    build_native()


def _desc(num_blocks, **over):
    d = dict(in_channels=64, out_channels=64, channels=64, growth=32, num_blocks=num_blocks, n_up=0, trunk_only=1)
    d.update(over)
    return d


def _lookup(plan, name):
    off, nbytes = C.c_int64(-1), C.c_int64(-1)
    return _lib.load().b200sr_debug_buffer(plan.handle, name.encode(), C.byref(off), C.byref(nbytes))


def trainable(name: str, pattern: str, num_blocks: int) -> bool:
    """Whether trunk parameter `name` (Sequential state_dict name) is trained under a freeze pattern."""
    if pattern == "all":
        return True
    if pattern == "frozen":
        return False
    if pattern == "head+half":  # the first half of the RRDBs frozen
        return int(name.split(".")[0]) >= num_blocks // 2
    if pattern == "last":       # only the last RRDB trained
        return int(name.split(".")[0]) == num_blocks - 1
    if pattern == "one_conv":   # one conv frozen inside an otherwise trainable dense block
        return not name.startswith(f"{num_blocks - 1}.rdb2.conv3.")
    if pattern == "no_bias":
        return not name.endswith(".bias")
    raise ValueError(pattern)


def flags(trunk, pattern):
    return [trainable(n, pattern, len(trunk)) for n, _ in trunk.named_parameters()]


@pytest.mark.parametrize("num_blocks", [1, 2, 23])
@pytest.mark.parametrize("training", [True, False])
def test_trunk_plan_sizes(num_blocks, training):
    plan = _Plan(_desc(num_blocks), 2, 24, 40, training)
    assert plan.num_params == RRDB_PARAMS * num_blocks
    assert plan.param_numel == RRDB_NUMEL * num_blocks
    assert plan.scale == 1 and plan.out_channels == 64
    gen = _Plan(b200.rrdbnet_x1(num_blocks=num_blocks).net_desc(), 2, 24, 40, training)
    assert gen.num_params == plan.num_params + 8 and plan.workspace_bytes < gen.workspace_bytes
    assert plan.pack_layout != gen.pack_layout
    # every trunk conv has a data gradient: the backward is twice the forward
    assert plan.flops_bwd == 2 * plan.flops_fwd
    assert plan.flops_fwd == 2 * (RRDB_NUMEL - 3 * 192) * num_blocks * 2 * 24 * 40  # 2 x MACs: weight elements x pixels


def test_trunk_module_state_dict_keys_match_a_plain_sequential():
    torch.manual_seed(0)
    t = b200.RRDBTrunk(num_blocks=3)
    ref = nn.Sequential(*[b200.rrdbnet._ResidualResidualDenseBlock(64, 32) for _ in range(3)])
    assert list(t.state_dict()) == list(ref.state_dict())
    assert sum(p.numel() for p in t.parameters()) == 3 * RRDB_NUMEL
    assert list(t.net_desc().items()) == list(_desc(3).items())


@pytest.mark.parametrize("bad", [dict(n_up=1), dict(in_channels=3), dict(out_channels=3), dict(out_channels=16), dict(channels=32),
                                 dict(growth=16), dict(num_blocks=0)])
def test_invalid_trunk_descriptors_are_rejected(bad):
    with pytest.raises(RuntimeError, match="libb200sr error -1"):
        _Plan({**_desc(2), **bad}, 1, 16, 16, True)


@pytest.mark.parametrize("training", [True, False])
def test_trunk_plan_names_only_the_trunk_buffers(training):
    plan = _Plan(_desc(2), 3, 40, 72, training)
    R = 6
    have = ["TR", "C1", "C2", "D0", "D1"] + ([f"D{r}" for r in range(R)] + ["GR", "GC1", "GC2"] + [f"DYB{r}" for r in range(R)]
                                               if training else [])
    for name in have:
        assert _lookup(plan, name) == 0, name
    gone = ["xin", "T0", "SPLT", "SPL0", "SPLC", "CMASK", "DYP", "G3", "GT", "GTB", "GO1", f"D{R}", f"DYB{R}"]
    if not training:
        gone += ["D2", "GR", "DYB0"]
    for name in gone:
        assert _lookup(plan, name) == -1, name


GEOMETRIES = [(2, 2, 24, 20), (2, 1, 160, 264), (23, 16, 64, 64), (23, 64, 64, 64)]


@pytest.mark.parametrize("nb,n,h,w", GEOMETRIES, ids=[f"{nb}-{n}x{h}x{w}" for nb, n, h, w in GEOMETRIES])
def test_trunk_launch_counts_follow_the_freeze_pattern(nb, n, h, w):
    trunk = b200.RRDBTrunk(num_blocks=nb)
    plan = _Plan(trunk.net_desc(), n, h, w, True)
    chains = plan.launches_fwd - 2                      # forward: ingest + chains + export
    assert chains >= 1
    # backward: dy ingest + the data-gradient chains + one weight-gradient launch per dense block + one unpack; dx adds its export
    assert plan.launches_bwd == 1 + chains + 3 * nb + 1
    assert plan.backward_launches() == plan.launches_bwd
    assert plan.backward_launches(flags(trunk, "all")) == plan.launches_bwd
    assert plan.backward_launches(flags(trunk, "no_bias")) == plan.launches_bwd
    assert plan.backward_launches(flags(trunk, "one_conv")) == plan.launches_bwd
    assert plan.backward_launches(with_dx=True) == plan.launches_bwd + 1
    assert plan.backward_launches(flags(trunk, "frozen"), with_dx=True) == 1 + chains + 1
    assert plan.backward_launches(flags(trunk, "frozen")) == 0
    half = plan.backward_launches(flags(trunk, "head+half"))
    last = plan.backward_launches(flags(trunk, "last"))
    assert plan.launches_bwd > half >= last > 0
    assert last == 1 + 1 + 3 + 1                        # the walk stops after the last RRDB: one chain launch
    assert plan.backward_launches(flags(trunk, "last"), with_dx=True) == 1 + chains + 3 + 1 + 1


def test_trunk_buckets():
    trunk = b200.RRDBTrunk(num_blocks=23)
    plan = _Plan(trunk.net_desc(), 16, 64, 64, True, grad_bucket_rrdbs=6)
    # RRDBs 18-22, 12-17, 6-11, 2-5, 0-1 are buckets (no conv1 / tail buckets in a trunk plan)
    assert plan.launches_bwd_bucketed - plan.launches_bwd == 5 - 1


def _ref_rrdb():
    """an RRDB as other code bases write it: its own forward, a LeakyReLU child per dense block"""
    class RDB(nn.Module):
        def __init__(self):
            super().__init__()
            for k in range(1, 6):
                setattr(self, f"conv{k}", nn.Conv2d(64 + 32 * (k - 1), 32 if k < 5 else 64, 3, 1, 1))
            self.lrelu = nn.LeakyReLU(0.2, True)

    class RRDB(nn.Module):
        def __init__(self):
            super().__init__()
            self.rdb1, self.rdb2, self.rdb3 = RDB(), RDB(), RDB()
    return RRDB()


class _Model(nn.Module):
    def __init__(self, nb):
        super().__init__()
        self.conv_first = nn.Conv2d(3, 64, 3, 1, 1)
        self.body = nn.Sequential(*[_ref_rrdb() for _ in range(nb)])
        self.conv_body = nn.Conv2d(64, 64, 3, 1, 1)


def test_native_trunk_adopts_the_children():
    torch.manual_seed(1)
    model = _Model(3)
    before = OrderedDict((k, v.clone()) for k, v in model.state_dict().items())
    params = [id(p) for p in model.parameters()]
    children = [id(m) for m in model.body]
    model.body = b200.native_trunk(model.body)
    assert isinstance(model.body, b200.RRDBTrunk) and isinstance(model.body, nn.Sequential)
    assert [id(m) for m in model.body] == children
    assert [id(p) for p in model.parameters()] == params
    after = model.state_dict()
    assert list(after) == list(before)
    assert all(torch.equal(after[k], v) for k, v in before.items())
    assert b200.native_trunk(model.body) is model.body
    # a slice is a trunk of the same modules
    part = model.body[1:]
    assert isinstance(part, b200.RRDBTrunk) and [id(m) for m in part] == children[1:]
    # the generator's own Sequential converts too
    net = b200.rrdbnet_x4(num_blocks=2)
    t = b200.native_trunk(net.trunk)
    assert [n for n, _ in t.named_parameters()] == [n[len("trunk."):] for n, _ in net.named_parameters() if n.startswith("trunk.")]


def _broken(kind):
    seq = nn.Sequential(*[_ref_rrdb() for _ in range(2)])
    rdb = seq[1].rdb2
    if kind == "not_sequential":
        return nn.ModuleList(list(seq))
    if kind == "empty":
        return nn.Sequential()
    if kind == "extra_child":
        seq[0].rdb4 = copy.deepcopy(seq[0].rdb1)
    elif kind == "missing_rdb":
        del seq[0].rdb3
    elif kind == "extra_param":
        seq[0].scale = nn.Parameter(torch.ones(1))
    elif kind == "rdb_extra_param":
        rdb.gain = nn.Parameter(torch.ones(1))
    elif kind == "rdb_buffer":
        rdb.register_buffer("running", torch.zeros(1))
    elif kind == "no_bias":
        rdb.conv3 = nn.Conv2d(128, 32, 3, 1, 1, bias=False)
    elif kind == "stride":
        rdb.conv3 = nn.Conv2d(128, 32, 3, 2, 1)
    elif kind == "kernel":
        rdb.conv3 = nn.Conv2d(128, 32, 5, 1, 2)
    elif kind == "width":
        rdb.conv1 = nn.Conv2d(64, 16, 3, 1, 1)
    elif kind == "dilation":
        rdb.conv5 = nn.Conv2d(192, 64, 3, 1, 2, dilation=2)
    elif kind == "reflect":
        rdb.conv2 = nn.Conv2d(96, 32, 3, 1, 1, padding_mode="reflect")
    elif kind == "not_conv":
        rdb.conv4 = nn.Linear(160, 32)
    return seq


@pytest.mark.parametrize("kind", ["not_sequential", "empty", "extra_child", "missing_rdb", "extra_param", "rdb_extra_param", "rdb_buffer",
                                  "no_bias", "stride", "kernel", "width", "dilation", "reflect", "not_conv"])
def test_native_trunk_rejects_other_structures(kind):
    with pytest.raises(ValueError):
        b200.native_trunk(_broken(kind))


def _oracle_params(trunk):
    return OrderedDict(("trunk." + k, v.detach().clone().requires_grad_(True)) for k, v in trunk.state_dict().items())


def test_cpu_forward_backward_equal_the_oracle_bit_for_bit():
    torch.manual_seed(2)
    trunk = b200.RRDBTrunk(num_blocks=2)
    for p in trunk.parameters():  # biases away from zero, larger trunk weights: every term of the contract shows
        p.data.add_(torch.randn_like(p) * 0.05)
    x = torch.randn(2, 64, 11, 13)
    dy = torch.randn(2, 64, 11, 13)
    xa = x.clone().requires_grad_(True)
    y = trunk(xa)
    y.backward(dy)
    p = _oracle_params(trunk)
    xb = x.clone().requires_grad_(True)
    ref = xb
    for b in range(2):
        ref = orc.rrdb_forward(ref, p, f"trunk.{b}")
    ref.backward(dy)
    assert torch.equal(y.detach(), ref.detach())
    assert torch.equal(xa.grad, xb.grad)
    for (n, q), g in zip(trunk.named_parameters(), p.values()):
        assert torch.equal(q.grad, g.grad), n


def test_trunk_module_round_trips():
    torch.manual_seed(3)
    trunk = b200.RRDBTrunk(num_blocks=2)
    x = torch.randn(1, 64, 8, 8)
    y = trunk(x)
    trunk._runtime()  # native state must not travel
    for other in (copy.deepcopy(trunk), pickle.loads(pickle.dumps(trunk))):
        assert isinstance(other, b200.RRDBTrunk) and "_b200_runtime" not in other.__dict__
        assert torch.equal(other(x), y)
    fresh = b200.RRDBTrunk(num_blocks=2)
    fresh.load_state_dict(trunk.state_dict())
    assert torch.equal(fresh(x), y)
    with torch.no_grad():
        assert torch.equal(trunk.eval()(x), y)
