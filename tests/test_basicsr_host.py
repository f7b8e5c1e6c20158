"""CPU: BasicSR's RRDBNet layout (BasicSRRRDBNet / native_generator) and the unclamped generator plans behind it -- plan sizes, launch
counts and buffer names against the clamped plan of the same descriptor, the module against a restatement of BasicSR's class (keys,
init, load_state_dict, CPU forward / backward), adoption and its rejections.  The GPU side is test_basicsr_gpu.py."""
import copy
import ctypes as C
import pickle

import pytest
import torch
import torch.nn.functional as F
from torch import nn
from torch.nn import init as nn_init

import sr_gan_fd_b200 as b200
from sr_gan_fd_b200 import lib as _lib
from sr_gan_fd_b200.function import _Plan


@pytest.fixture(scope="module", autouse=True)
def _built():
    from sr_gan_fd_b200.build import build_native
    build_native()


# --- a restatement of basicsr/archs/rrdbnet_arch.py and the helpers it imports (basicsr/archs/arch_util.py) ----------------------
@torch.no_grad()
def default_init_weights(module_list, scale=1, bias_fill=0, **kwargs):
    if not isinstance(module_list, list):
        module_list = [module_list]
    for module in module_list:
        for m in module.modules():
            if isinstance(m, nn.Conv2d):
                nn_init.kaiming_normal_(m.weight, **kwargs)
                m.weight.data *= scale
                if m.bias is not None:
                    m.bias.data.fill_(bias_fill)
            elif isinstance(m, nn.Linear):
                nn_init.kaiming_normal_(m.weight, **kwargs)
                m.weight.data *= scale
                if m.bias is not None:
                    m.bias.data.fill_(bias_fill)


def make_layer(basic_block, num_basic_block, **kwarg):
    return nn.Sequential(*[basic_block(**kwarg) for _ in range(num_basic_block)])


def pixel_unshuffle(x, scale):
    b, c, hh, hw = x.size()
    out_channel = c * (scale ** 2)
    assert hh % scale == 0 and hw % scale == 0
    h = hh // scale
    w = hw // scale
    x_view = x.view(b, c, h, scale, w, scale)
    return x_view.permute(0, 1, 3, 5, 2, 4).reshape(b, out_channel, h, w)


class ResidualDenseBlock(nn.Module):
    def __init__(self, num_feat=64, num_grow_ch=32):
        super().__init__()
        self.conv1 = nn.Conv2d(num_feat, num_grow_ch, 3, 1, 1)
        self.conv2 = nn.Conv2d(num_feat + num_grow_ch, num_grow_ch, 3, 1, 1)
        self.conv3 = nn.Conv2d(num_feat + 2 * num_grow_ch, num_grow_ch, 3, 1, 1)
        self.conv4 = nn.Conv2d(num_feat + 3 * num_grow_ch, num_grow_ch, 3, 1, 1)
        self.conv5 = nn.Conv2d(num_feat + 4 * num_grow_ch, num_feat, 3, 1, 1)
        self.lrelu = nn.LeakyReLU(negative_slope=0.2, inplace=True)
        default_init_weights([self.conv1, self.conv2, self.conv3, self.conv4, self.conv5], 0.1)

    def forward(self, x):
        x1 = self.lrelu(self.conv1(x))
        x2 = self.lrelu(self.conv2(torch.cat((x, x1), 1)))
        x3 = self.lrelu(self.conv3(torch.cat((x, x1, x2), 1)))
        x4 = self.lrelu(self.conv4(torch.cat((x, x1, x2, x3), 1)))
        x5 = self.conv5(torch.cat((x, x1, x2, x3, x4), 1))
        return x5 * 0.2 + x


class RRDB(nn.Module):
    def __init__(self, num_feat, num_grow_ch=32):
        super().__init__()
        self.rdb1 = ResidualDenseBlock(num_feat, num_grow_ch)
        self.rdb2 = ResidualDenseBlock(num_feat, num_grow_ch)
        self.rdb3 = ResidualDenseBlock(num_feat, num_grow_ch)

    def forward(self, x):
        out = self.rdb1(x)
        out = self.rdb2(out)
        out = self.rdb3(out)
        return out * 0.2 + x


class RRDBNet(nn.Module):
    def __init__(self, num_in_ch, num_out_ch, scale=4, num_feat=64, num_block=23, num_grow_ch=32):
        super().__init__()
        self.scale = scale
        if scale == 2:
            num_in_ch = num_in_ch * 4
        elif scale == 1:
            num_in_ch = num_in_ch * 16
        self.conv_first = nn.Conv2d(num_in_ch, num_feat, 3, 1, 1)
        self.body = make_layer(RRDB, num_block, num_feat=num_feat, num_grow_ch=num_grow_ch)
        self.conv_body = nn.Conv2d(num_feat, num_feat, 3, 1, 1)
        self.conv_up1 = nn.Conv2d(num_feat, num_feat, 3, 1, 1)
        self.conv_up2 = nn.Conv2d(num_feat, num_feat, 3, 1, 1)
        self.conv_hr = nn.Conv2d(num_feat, num_feat, 3, 1, 1)
        self.conv_last = nn.Conv2d(num_feat, num_out_ch, 3, 1, 1)
        self.lrelu = nn.LeakyReLU(negative_slope=0.2, inplace=True)

    def forward(self, x):
        if self.scale == 2:
            feat = pixel_unshuffle(x, scale=2)
        elif self.scale == 1:
            feat = pixel_unshuffle(x, scale=4)
        else:
            feat = x
        feat = self.conv_first(feat)
        body_feat = self.conv_body(self.body(feat))
        feat = feat + body_feat
        feat = self.lrelu(self.conv_up1(F.interpolate(feat, scale_factor=2, mode="nearest")))
        feat = self.lrelu(self.conv_up2(F.interpolate(feat, scale_factor=2, mode="nearest")))
        out = self.conv_last(self.lrelu(self.conv_hr(feat)))
        return out
# -------------------------------------------------------------------------------------------------------------------------------------


def _clamped(desc):
    return {k: v for k, v in desc.items() if k != "clamp"}


def _lookup(plan, name):
    off, nbytes = C.c_int64(-1), C.c_int64(-1)
    return _lib.load().b200sr_debug_buffer(plan.handle, name.encode(), C.byref(off), C.byref(nbytes))


def test_version():
    assert _lib.load().b200sr_version() == 103


PLAN_CASES = [(3, 3, 1, 2, 24, 20), (12, 3, 2, 16, 64, 64), (48, 1, 23, 16, 64, 64), (3, 16, 2, 1, 256, 256), (3, 3, 2, 3, 40, 72)]


@pytest.mark.parametrize("det", [False, True])
@pytest.mark.parametrize("training", [True, False])
@pytest.mark.parametrize("in_ch,out_ch,nb,n,h,w", PLAN_CASES, ids=[f"{i}-{o}-{nb}-{n}x{h}x{w}" for i, o, nb, n, h, w in PLAN_CASES])
def test_unclamped_plan_matches_the_clamped_plan(in_ch, out_ch, nb, n, h, w, training, det):
    desc = dict(in_channels=in_ch, out_channels=out_ch, channels=64, growth=32, num_blocks=nb, n_up=2, clamp=0)
    pu = _Plan(desc, n, h, w, training, deterministic=det)
    pc = _Plan(_clamped(desc), n, h, w, training, deterministic=det)
    for attr in ("num_params", "param_numel", "pack_layout", "packed_bytes", "flops_fwd", "flops_bwd", "launches_fwd", "launches_bwd",
                 "launches_bwd_bucketed", "scale", "out_channels"):
        assert getattr(pu, attr) == getattr(pc, attr), attr
    cmask = -(-(n * out_ch * 16 * h * w) // 1024) * 1024  # N x out_ch x sH x sW bytes, rounded up to the 1024-byte granule
    assert pc.workspace_bytes - pu.workspace_bytes == (cmask if training else 0)
    assert _lookup(pu, "CMASK") == -1
    assert _lookup(pc, "CMASK") == (0 if training else -1)
    for name in ("xin", "T0", "SPLT", "SPLC") + (("DYP", "G3", "GT") if training else ()):
        assert _lookup(pu, name) == 0, name
    if training:
        nconv = pu.num_params // 2
        masks = [None, [1] * nconv, [0] * nconv, [0] + [1] * (nconv - 1), [1] * (1 + 15 * nb) + [0] * (nconv - 1 - 15 * nb),
                 [0] * (nconv - 1) + [1], [i % 3 == 0 for i in range(nconv)]]
        for mask in masks:
            flags = None if mask is None else [bool(m) for m in mask for _ in (0, 1)]
            for with_dx in (False, True):
                for with_cb in (False, True):
                    assert pu.backward_launches(flags, with_dx, with_cb) == pc.backward_launches(flags, with_dx, with_cb), (mask, with_dx)


@pytest.mark.parametrize("bad", [dict(in_channels=65), dict(out_channels=17), dict(channels=32), dict(growth=16), dict(num_blocks=0),
                                 dict(n_up=4)])
def test_unclamped_plan_rejects_what_the_clamped_plan_rejects(bad):
    desc = {**dict(in_channels=3, out_channels=3, channels=64, growth=32, num_blocks=1, n_up=2, clamp=0), **bad}
    for d in (desc, _clamped(desc)):
        with pytest.raises(RuntimeError, match="libb200sr error -1"):
            _Plan(d, 1, 16, 16, True)


@pytest.mark.parametrize("num_block", [6, 23])
@pytest.mark.parametrize("scale", [1, 2, 4])
def test_state_dict_and_init_match_basicsr(scale, num_block):
    torch.manual_seed(11)
    ref = RRDBNet(3, 3, scale=scale, num_block=num_block)
    torch.manual_seed(11)
    mine = b200.BasicSRRRDBNet(3, 3, scale=scale, num_block=num_block)
    a, b = ref.state_dict(), mine.state_dict()
    assert list(a) == list(b)
    for k in a:
        assert a[k].shape == b[k].shape, k
        assert torch.equal(a[k], b[k]), k  # same RNG draws in the same order: identical initial values
    assert [n for n, _ in mine.named_children()] == ["conv_first", "body", "conv_body", "conv_up1", "conv_up2", "conv_hr", "conv_last",
                                                     "lrelu"]
    assert mine.scale == scale
    # the library's parameter order is the state_dict order
    assert [c.weight for c in mine._conv_list()] == [p for n, p in mine.named_parameters() if n.endswith("weight")]
    d = mine.net_desc()
    assert d["clamp"] == 0 and d["n_up"] == 2 and d["num_blocks"] == num_block and d["in_channels"] == 3 * {4: 1, 2: 4, 1: 16}[scale]


def test_load_state_dict_round_trip():
    torch.manual_seed(1)
    ref = RRDBNet(3, 3, scale=2, num_block=2)
    torch.manual_seed(2)
    mine = b200.BasicSRRRDBNet(3, 3, scale=2, num_block=2)
    mine.load_state_dict(ref.state_dict())
    back = RRDBNet(3, 3, scale=2, num_block=2)
    back.load_state_dict(mine.state_dict())
    for (k, v), (k2, v2) in zip(ref.state_dict().items(), back.state_dict().items()):
        assert k == k2 and torch.equal(v, v2)


def test_unsupported_scale_is_rejected():
    with pytest.raises(ValueError):
        b200.BasicSRRRDBNet(3, 3, scale=8)


def test_native_generator_adopts_the_children():
    torch.manual_seed(3)
    ref = RRDBNet(3, 3, scale=4, num_block=3)
    before = {k: v.clone() for k, v in ref.state_dict().items()}
    params = list(ref.parameters())
    children = dict(ref.named_children())
    opt = torch.optim.Adam(ref.parameters())
    net = b200.native_generator(ref)
    assert isinstance(net, b200.BasicSRRRDBNet) and net.scale == 4
    assert all(a is b for a, b in zip(net.parameters(), params)) and len(list(net.parameters())) == len(params)
    assert all(getattr(net, n) is m for n, m in children.items())
    after = net.state_dict()
    assert list(after) == list(before) and all(torch.equal(after[k], before[k]) for k in before)
    assert opt.param_groups[0]["params"][0] is net.conv_first.weight
    assert b200.native_generator(net) is net
    # an already native trunk is accepted as the body
    ref2 = RRDBNet(3, 3, scale=1, num_block=1)
    ref2.body = b200.native_trunk(ref2.body)
    assert b200.native_generator(ref2).body is ref2.body


def _broken(kind):
    torch.manual_seed(4)
    m = RRDBNet(3, 3, scale=4, num_block=2)
    if kind == "child_name":
        m.conv_tail = m.conv_last
        del m.conv_last
    elif kind == "extra_child":
        m.extra = nn.Identity()
    elif kind == "missing_lrelu":
        del m.lrelu
    elif kind == "lrelu_slope":
        m.lrelu = nn.LeakyReLU(0.1)
    elif kind == "feat_width":
        m = RRDBNet(3, 3, scale=4, num_feat=32, num_block=1)
    elif kind == "grow_width":
        m = RRDBNet(3, 3, scale=4, num_grow_ch=16, num_block=1)
    elif kind == "no_bias":
        m.conv_hr = nn.Conv2d(64, 64, 3, 1, 1, bias=False)
    elif kind == "kernel_1x1":
        m.conv_up1 = nn.Conv2d(64, 64, 1)
    elif kind == "scale_8":
        m.scale = 8
    elif kind == "no_scale":
        del m.scale
    elif kind == "out_channels":
        m.conv_last = nn.Conv2d(64, 17, 3, 1, 1)
    elif kind == "extra_param":
        m.gain = nn.Parameter(torch.ones(1))
    elif kind == "extra_buffer":
        m.register_buffer("mean", torch.zeros(3))
    elif kind == "conv_buffer":
        m.conv_body.register_buffer("u", torch.zeros(64))
    elif kind == "rrdb_buffer":
        m.body[1].rdb2.register_buffer("u", torch.zeros(1))
    elif kind == "body_not_rrdb":
        m.body = nn.Sequential(nn.Conv2d(64, 64, 3, 1, 1))
    elif kind == "weight_norm":
        m.conv_first = torch.nn.utils.parametrizations.weight_norm(m.conv_first)
    return m


REJECTED = ["child_name", "extra_child", "missing_lrelu", "lrelu_slope", "feat_width", "grow_width", "no_bias", "kernel_1x1", "scale_8",
            "no_scale", "out_channels", "extra_param", "extra_buffer", "conv_buffer", "rrdb_buffer", "body_not_rrdb", "weight_norm"]


@pytest.mark.parametrize("kind", REJECTED)
def test_native_generator_rejects_other_structures(kind):
    with pytest.raises(ValueError):
        b200.native_generator(_broken(kind))


@pytest.mark.parametrize("scale", [1, 2, 4])
def test_cpu_forward_backward_equal_basicsr_bit_for_bit(scale):
    for nb in (1, 2):
        torch.manual_seed(5 + nb)
        ref = RRDBNet(3, 3, scale=scale, num_block=nb)
        mine = b200.BasicSRRRDBNet(3, 3, scale=scale, num_block=nb)
        mine.load_state_dict(ref.state_dict())
        g = torch.Generator().manual_seed(6)
        x = torch.rand(2, 3, 16, 12, generator=g)
        dy = torch.randn(2, 3, 16 * scale, 12 * scale, generator=g)
        outs = []
        for m in (ref, mine):
            xx = x.clone().requires_grad_(True)
            y = m(xx)
            y.backward(dy)
            outs.append([y.detach(), xx.grad] + [p.grad for p in m.parameters()])
            m.zero_grad(set_to_none=True)
        assert outs[0][0].shape == (2, 3, 16 * scale, 12 * scale)
        for a, b in zip(*outs):
            assert torch.equal(a, b)


def test_cpu_output_is_not_clamped():
    torch.manual_seed(7)
    net = b200.BasicSRRRDBNet(3, 3, scale=4, num_block=1)
    with torch.no_grad():
        net.conv_last.bias.fill_(-2.0)
        y = net(torch.rand(1, 3, 8, 8))
    assert float(y.max()) < 0


def test_round_trips():
    torch.manual_seed(8)
    net = b200.BasicSRRRDBNet(3, 3, scale=2, num_block=2)
    x = torch.rand(1, 3, 8, 8)
    with torch.no_grad():
        y = net(x)
    for other in (copy.deepcopy(net), pickle.loads(pickle.dumps(net))):
        assert isinstance(other, b200.BasicSRRRDBNet) and other.scale == 2
        assert list(other.state_dict()) == list(net.state_dict())
        with torch.no_grad():
            assert torch.equal(other(x), y)
    fresh = b200.BasicSRRRDBNet(3, 3, scale=2, num_block=2)
    fresh.load_state_dict(net.state_dict())
    with torch.no_grad():
        assert torch.equal(fresh(x), y)
    net._runtime()  # native runtime state stays out of copies
    assert "_b200_runtime" not in copy.deepcopy(net).__dict__
