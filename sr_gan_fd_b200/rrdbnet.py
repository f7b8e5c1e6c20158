"""Drop-in RRDBNet generators: same constructors, ``nn.Module`` tree and ``state_dict`` layout as the reference.

Reference interfaces mirrored here (MiNeves00/SR-GAN-FD):

* ``ESRGAN/model.py:29-86,144-243,301-322``      -> :class:`RRDBNet`, ``rrdbnet_x1/x2/x4/x8``
* ``BSRGAN/model.py:31-88,311-384,576-587``      -> :class:`BSRGAN`, ``bsrgan_x2/x4``   (A-ESRGAN/model.py:421-558 same)
* ``Real_ESRGAN/model.py:108-263,331-334``       -> :class:`RealRRDBNet` (exported as ``RRDBNet`` by the compat shim)

The submodules are real ``nn.Conv2d`` so ``torch.manual_seed(s)`` + constructor reproduces the reference's weights
bit for bit, and ``load_state_dict`` / ``utils.load_state_dict`` key+shape filtering behave identically.  Only
``forward`` differs: the whole network (forward and backward) is ONE ``torch.autograd.Function`` that calls the
C-ABI CUDA library (``include/b200sr.h``).  There is no CPU or eager-PyTorch fallback: a CPU tensor or a missing
``libb200sr.so`` raises.
"""
from __future__ import annotations

from collections import OrderedDict
from typing import Any, List

import torch
import torch.nn.functional as F
from torch import nn

from . import function as _function

__all__ = [
    "RRDBNet", "BSRGAN", "RealRRDBNet", "RRDBTrunk", "native_trunk", "BasicSRRRDBNet", "native_generator",
    "rrdbnet_x1", "rrdbnet_x2", "rrdbnet_x4", "rrdbnet_x8", "bsrgan_x2", "bsrgan_x4", "real_rrdbnet_x4",
]


class _ResidualDenseBlock(nn.Module):
    """Parameter container for one dense block (``ESRGAN/model.py:38-47``).  Never called layer by layer."""

    def __init__(self, channels: int, growth_channels: int, reinit: bool = False) -> None:
        super().__init__()
        self.conv1 = nn.Conv2d(channels + growth_channels * 0, growth_channels, (3, 3), (1, 1), (1, 1))
        self.conv2 = nn.Conv2d(channels + growth_channels * 1, growth_channels, (3, 3), (1, 1), (1, 1))
        self.conv3 = nn.Conv2d(channels + growth_channels * 2, growth_channels, (3, 3), (1, 1), (1, 1))
        self.conv4 = nn.Conv2d(channels + growth_channels * 3, growth_channels, (3, 3), (1, 1), (1, 1))
        self.conv5 = nn.Conv2d(channels + growth_channels * 4, channels, (3, 3), (1, 1), (1, 1))
        self.leaky_relu = nn.LeakyReLU(0.2, True)
        self.identity = nn.Identity()
        if reinit:
            # Real_ESRGAN/model.py:128-129,144-150 re-initialises inside every block constructor, which changes
            # the RNG draw order relative to ESRGAN/BSRGAN for the same seed.
            for module in self.modules():
                if isinstance(module, nn.Conv2d):
                    nn.init.kaiming_normal_(module.weight)
                    module.weight.data *= 0.1
                    if module.bias is not None:
                        nn.init.constant_(module.bias, 0)

    def forward(self, x):  # pragma: no cover - guarded on purpose
        raise RuntimeError("dense blocks are executed by the fused B200 generator kernel, not layer by layer")


class _ResidualResidualDenseBlock(nn.Module):
    """``ESRGAN/model.py:72-75``."""

    def __init__(self, channels: int, growth_channels: int, reinit: bool = False) -> None:
        super().__init__()
        self.rdb1 = _ResidualDenseBlock(channels, growth_channels, reinit)
        self.rdb2 = _ResidualDenseBlock(channels, growth_channels, reinit)
        self.rdb3 = _ResidualDenseBlock(channels, growth_channels, reinit)

    def forward(self, x):  # pragma: no cover
        raise RuntimeError("RRDBs are executed by the fused B200 generator kernel, not layer by layer")


def _up_stage(channels: int) -> nn.Sequential:
    return nn.Sequential(nn.Conv2d(channels, channels, (3, 3), (1, 1), (1, 1)), nn.LeakyReLU(0.2, True))


class _NativeState:
    """Mixin of the modules whose forward runs in libb200sr.so: ESRGAN init, and native runtime state that is never part of
    the module's persistent state."""

    def _finish_init(self) -> None:
        for module in self.modules():
            if isinstance(module, nn.Conv2d):
                nn.init.kaiming_normal_(module.weight)
                module.weight.data *= 0.1
                if module.bias is not None:
                    nn.init.constant_(module.bias, 0)

    # --- native runtime state is never part of the module's persistent state --------------------------------
    def _runtime(self) -> "_function.GeneratorRuntime":
        rt = self.__dict__.get("_b200_runtime")
        if rt is None:
            rt = _function.GeneratorRuntime()
            self.__dict__["_b200_runtime"] = rt
        return rt

    def __getstate__(self):
        state = self.__dict__.copy()
        state.pop("_b200_runtime", None)
        return state

    def __deepcopy__(self, memo):
        import copy
        cls = self.__class__
        new = cls.__new__(cls)
        memo[id(self)] = new
        for k, v in self.__dict__.items():
            if k == "_b200_runtime":
                continue
            new.__dict__[k] = copy.deepcopy(v, memo)
        return new


class _GeneratorBase(_NativeState, nn.Module):
    """Shared forward: collects the convs in ``state_dict`` order and hands them to the native path."""

    upscale_factor: int
    _n_up: int
    _pixel_unshuffle: int = 1

    def zero_grad(self, set_to_none: bool = True) -> None:
        """Same contract as ``nn.Module.zero_grad``; the ``set_to_none`` path skips the generic per-parameter work (the
        training loop calls this every step, ESRGAN/train_rrdbnet.py:255, and the gradients are views of one flat buffer)."""
        if not set_to_none:
            return super().zero_grad(set_to_none=False)
        rt = self._runtime()
        if rt.convs is None:
            rt.convs = self._conv_list()  # every parameter of the generator belongs to one of these convs
        for conv in rt.convs:
            pd = conv._parameters
            pd["weight"].grad = None
            if pd["bias"] is not None:
                pd["bias"].grad = None

    def _conv_list(self) -> List[nn.Conv2d]:
        convs = [self.conv1]
        for rrdb in self.trunk:
            for rdb in (rrdb.rdb1, rrdb.rdb2, rrdb.rdb3):
                convs += [rdb.conv1, rdb.conv2, rdb.conv3, rdb.conv4, rdb.conv5]
        convs.append(self.conv2)
        for u in range(1, self._n_up + 1):
            convs.append(getattr(self, f"upsampling{u}")[0])
        convs += [self.conv3[0], self.conv4]
        return convs

    def net_desc(self) -> dict:
        first_rdb = self.trunk[0].rdb1
        return dict(
            in_channels=self.conv1.in_channels, out_channels=self.conv4.out_channels,
            channels=self.conv1.out_channels, growth=first_rdb.conv1.out_channels,
            num_blocks=len(self.trunk), n_up=self._n_up, pixel_unshuffle=self._pixel_unshuffle,
        )

    def _forward_impl(self, x: torch.Tensor) -> torch.Tensor:
        return _function.generator_forward(self, x)

    def forward(self, x: torch.Tensor) -> torch.Tensor:
        return self._forward_impl(x)


class RRDBNet(_GeneratorBase):
    """``ESRGAN/model.py:144-243`` -- same signature, same children, same init."""

    def __init__(self, in_channels: int = 3, out_channels: int = 3, channels: int = 64, growth_channels: int = 32,
                 num_blocks: int = 23, upscale_factor: int = 4) -> None:
        super().__init__()
        self.upscale_factor = upscale_factor
        self.conv1 = nn.Conv2d(in_channels, channels, (3, 3), (1, 1), (1, 1))
        self.trunk = nn.Sequential(*[_ResidualResidualDenseBlock(channels, growth_channels)
                                     for _ in range(num_blocks)])
        self.conv2 = nn.Conv2d(channels, channels, (3, 3), (1, 1), (1, 1))
        self._n_up = {1: 0, 2: 1, 4: 2, 8: 3}.get(upscale_factor, 0)
        for u in range(1, self._n_up + 1):
            setattr(self, f"upsampling{u}", _up_stage(channels))
        self.conv3 = nn.Sequential(nn.Conv2d(channels, channels, (3, 3), (1, 1), (1, 1)), nn.LeakyReLU(0.2, True))
        self.conv4 = nn.Conv2d(channels, out_channels, (3, 3), (1, 1), (1, 1))
        self._initialize_weights()

    def _initialize_weights(self) -> None:
        self._finish_init()


class BSRGAN(_GeneratorBase):
    """``BSRGAN/model.py:311-384`` (and its copy ``A-ESRGAN/model.py:489-552``): ctor kw ``num_rrdb``; always
    ``upsampling1``, ``upsampling2`` only for x4."""

    def __init__(self, in_channels: int = 3, out_channels: int = 3, channels: int = 64, growth_channels: int = 32,
                 num_rrdb: int = 23, upscale_factor: int = 4) -> None:
        super().__init__()
        self.upscale_factor = upscale_factor
        self.conv1 = nn.Conv2d(in_channels, channels, (3, 3), (1, 1), (1, 1))
        self.trunk = nn.Sequential(*[_ResidualResidualDenseBlock(channels, growth_channels)
                                     for _ in range(num_rrdb)])
        self.conv2 = nn.Conv2d(channels, channels, (3, 3), (1, 1), (1, 1))
        self.upsampling1 = _up_stage(channels)
        self._n_up = 1
        if upscale_factor == 4:
            self.upsampling2 = _up_stage(channels)
            self._n_up = 2
        self.conv3 = nn.Sequential(nn.Conv2d(channels, channels, (3, 3), (1, 1), (1, 1)), nn.LeakyReLU(0.2, True))
        self.conv4 = nn.Conv2d(channels, out_channels, (3, 3), (1, 1), (1, 1))
        self._finish_init()


class RealRRDBNet(_GeneratorBase):
    """``Real_ESRGAN/model.py:179-263``: positional ctor, always two upsamplings, pixel-unshuffle front for x2/x1."""

    def __init__(self, in_channels: int, out_channels: int, channels: int, growth_channels: int, num_rrdb: int,
                 upscale_factor: int) -> None:
        super().__init__()
        if upscale_factor == 2:
            in_channels *= 4
            downscale_factor = 2
        elif upscale_factor == 1:
            in_channels *= 16
            downscale_factor = 4
        else:
            downscale_factor = 1
        self.downsampling = nn.PixelUnshuffle(downscale_factor)
        self._pixel_unshuffle = downscale_factor
        self.conv1 = nn.Conv2d(in_channels, channels, (3, 3), (1, 1), (1, 1))
        self.trunk = nn.Sequential(*[_ResidualResidualDenseBlock(channels, growth_channels, reinit=True)
                                     for _ in range(num_rrdb)])
        self.conv2 = nn.Conv2d(channels, channels, (3, 3), (1, 1), (1, 1))
        self.upsampling1 = _up_stage(channels)
        self.upsampling2 = _up_stage(channels)
        self._n_up = 2
        self.conv3 = nn.Sequential(nn.Conv2d(channels, channels, (3, 3), (1, 1), (1, 1)), nn.LeakyReLU(0.2, True))
        self.conv4 = nn.Conv2d(channels, out_channels, (3, 3), (1, 1), (1, 1))
        self._finish_init()

    def _forward_impl(self, x: torch.Tensor) -> torch.Tensor:
        # nn.PixelUnshuffle is pure data movement on the 3-channel input (identity for x4); kept as the torch op.
        return _function.generator_forward(self, self.downsampling(x))


class RRDBTrunk(_NativeState, nn.Sequential):
    """The RRDB stack alone, as a drop-in for ``nn.Sequential(*RRDBs)`` in any generator built around it (BasicSR /
    Real-ESRGAN ``RRDBNet``, A-ESRGAN's ``bsrgantrans_x2`` / ``gen_rrdb2x``, models with their own head, tail or
    conditioning).  ``state_dict`` keys are those of the Sequential (``0.rdb1.conv1.weight`` ...).

    Math contract (ESRGAN / BasicSR RRDB), for ``x`` of shape ``[N, 64, H, W]``::

        dense block:  o_k = LeakyReLU_0.2(conv_k(cat(x, o_1 .. o_{k-1})))  for k = 1..4
                      rdb(x) = 0.2 * conv5(cat(x, o_1 .. o_4)) + x
        RRDB:         rrdb(x) = 0.2 * rdb3(rdb2(rdb1(x))) + x
        trunk:        y = rrdb_{B-1}( ... rrdb_0(x))

    3x3 convs, stride 1, padding 1, with bias; 64 channels, growth 32.  On a CUDA device forward and backward run in the
    generator's kernels (``include/b200sr.h`` "Trunk plans"): ``x`` may be fp32, fp16 or bf16, NCHW or channels_last; ``y``
    and the input gradient are fp32, ``y`` is not clamped.  On the CPU the children run through stock torch ops.
    Build one with the constructor, or adopt an existing Sequential with :func:`native_trunk`."""

    def __init__(self, channels: int = 64, growth_channels: int = 32, num_blocks: int = 23) -> None:
        nn.Sequential.__init__(self, *[_ResidualResidualDenseBlock(channels, growth_channels) for _ in range(num_blocks)])
        self._finish_init()

    def __getitem__(self, idx):
        if isinstance(idx, slice):  # nn.Sequential would call the constructor with the children
            return _adopt(OrderedDict(list(self._modules.items())[idx]))
        return nn.Sequential.__getitem__(self, idx)

    def _conv_list(self) -> List[nn.Conv2d]:
        return [getattr(getattr(rrdb, r), c) for rrdb in self for r in ("rdb1", "rdb2", "rdb3")
                for c in ("conv1", "conv2", "conv3", "conv4", "conv5")]

    def net_desc(self) -> dict:
        conv1 = self[0].rdb1.conv1
        return dict(in_channels=conv1.in_channels, out_channels=conv1.in_channels, channels=conv1.in_channels,
                    growth=conv1.out_channels, num_blocks=len(self), n_up=0, trunk_only=1)

    def forward(self, x: torch.Tensor) -> torch.Tensor:
        if not x.is_cuda:
            return _function.eager_trunk(self, x)
        return _function.generator_forward(self, x)


def _adopt(children: "OrderedDict[str, nn.Module]") -> RRDBTrunk:
    trunk = RRDBTrunk.__new__(RRDBTrunk)
    nn.Sequential.__init__(trunk, children)
    return trunk


def native_trunk(seq: nn.Sequential) -> RRDBTrunk:
    """An :class:`RRDBTrunk` that adopts the children of ``seq`` (the same module objects: Parameter identity, optimizer state and
    the parent model's ``state_dict`` are unchanged).  Usage: ``model.trunk = native_trunk(model.trunk)``.

    Every child must hold exactly ``rdb1``, ``rdb2``, ``rdb3``, each with ``conv1`` .. ``conv5``: 3x3 ``nn.Conv2d`` with bias,
    stride 1, padding 1, of the RRDB shapes for 64 channels and growth 32, and no other parameters or buffers
    (parameter-free children such as a LeakyReLU module are fine).  Anything else raises ``ValueError``: the native path computes
    the contract in :class:`RRDBTrunk`'s docstring and nothing else."""
    if isinstance(seq, RRDBTrunk):
        return seq
    _check_rrdb_stack(seq)
    return _adopt(OrderedDict(seq.named_children()))


def _check_rrdb_stack(seq: nn.Module) -> None:
    """Raise ``ValueError`` unless ``seq`` is what :func:`native_trunk` accepts (an :class:`RRDBTrunk` always is)."""
    if isinstance(seq, RRDBTrunk):
        return
    if not isinstance(seq, nn.Sequential) or len(seq) == 0:
        raise ValueError("native_trunk expects a non-empty nn.Sequential of RRDBs")
    for name, rrdb in seq.named_children():
        if [n for n, _ in rrdb.named_children()] != ["rdb1", "rdb2", "rdb3"] or \
                any(True for _ in rrdb.named_parameters(recurse=False)) or any(True for _ in rrdb.named_buffers(recurse=False)):
            raise ValueError(f"trunk child {name!r} is not an RRDB of exactly rdb1, rdb2, rdb3")
        for r in ("rdb1", "rdb2", "rdb3"):
            rdb = getattr(rrdb, r)
            expect = {f"conv{k}.{p}" for k in range(1, 6) for p in ("weight", "bias")}
            params = {n for n, _ in rdb.named_parameters()}
            if params != expect or any(True for _ in rdb.named_buffers()):
                raise ValueError(f"{name}.{r}: expected the parameters of conv1..conv5 and nothing else, got {sorted(params)}")
            for k in range(1, 6):
                _check_conv3x3(getattr(rdb, f"conv{k}"), f"{name}.{r}.conv{k}", 64 + 32 * (k - 1), 32 if k < 5 else 64)


def _check_conv3x3(conv: nn.Module, name: str, cin: int, cout: int) -> None:
    """Raise ``ValueError`` unless ``conv`` is a 3x3 ``nn.Conv2d(cin, cout)``, stride 1, padding 1, with bias: the only conv the native
    kernels compute."""
    if not (type(conv) is nn.Conv2d and conv.in_channels == cin and conv.out_channels == cout and
            conv.kernel_size == (3, 3) and conv.stride == (1, 1) and conv.padding == (1, 1) and
            conv.dilation == (1, 1) and conv.groups == 1 and conv.padding_mode == "zeros" and conv.bias is not None):
        raise ValueError(f"{name}: expected a 3x3 Conv2d({cin}, {cout}), stride 1, padding 1, with bias; got {conv!r}")


class BasicSRRRDBNet(_GeneratorBase):
    """BasicSR's ``RRDBNet`` (``basicsr/archs/rrdbnet_arch.py``), the generator of the Real-ESRGAN release checkpoints: same
    constructor, children (``conv_first``, ``body``, ``conv_body``, ``conv_up1``, ``conv_up2``, ``conv_hr``, ``conv_last``,
    ``lrelu``), init and ``state_dict``, so a Real-ESRGAN ``params_ema`` dict loads unchanged.  ``scale`` 2 and 1 pixel-unshuffle
    the input by 2 and 4 first (``conv_first`` takes ``num_in_ch * 4`` / ``* 16`` channels).  Math::

        feat = conv_first(unshuffle(x));  feat = feat + conv_body(body(feat))        (body: the RRDBs of RRDBTrunk)
        feat = lrelu(conv_up1(nearest_x2(feat)));  feat = lrelu(conv_up2(nearest_x2(feat)))
        out  = conv_last(lrelu(conv_hr(feat)))                                        -- NOT clamped

    On a CUDA device forward and backward run in the generator's kernels through an unclamped plan (``include/b200sr.h``
    "Unclamped plans"); on the CPU the children run through stock torch ops.  Adopt an existing module of this layout with
    :func:`native_generator`."""

    _n_up = 2

    def __init__(self, num_in_ch: int, num_out_ch: int, scale: int = 4, num_feat: int = 64, num_block: int = 23,
                 num_grow_ch: int = 32) -> None:
        super().__init__()
        if scale not in (1, 2, 4):
            raise ValueError(f"BasicSRRRDBNet supports scale 1, 2 and 4, got {scale}")
        self._set_scale(scale)
        self.conv_first = nn.Conv2d(num_in_ch * self._pixel_unshuffle ** 2, num_feat, 3, 1, 1)
        # BasicSR's ResidualDenseBlock runs default_init_weights(..., 0.1) in its constructor: the reinit=True dense block
        self.body = nn.Sequential(*[_ResidualResidualDenseBlock(num_feat, num_grow_ch, reinit=True) for _ in range(num_block)])
        self.conv_body = nn.Conv2d(num_feat, num_feat, 3, 1, 1)
        self.conv_up1 = nn.Conv2d(num_feat, num_feat, 3, 1, 1)
        self.conv_up2 = nn.Conv2d(num_feat, num_feat, 3, 1, 1)
        self.conv_hr = nn.Conv2d(num_feat, num_feat, 3, 1, 1)
        self.conv_last = nn.Conv2d(num_feat, num_out_ch, 3, 1, 1)
        self.lrelu = nn.LeakyReLU(negative_slope=0.2, inplace=True)

    def _set_scale(self, scale: int) -> None:
        self.scale = self.upscale_factor = scale
        self._pixel_unshuffle = {4: 1, 2: 2, 1: 4}[scale]

    def _conv_list(self) -> List[nn.Conv2d]:
        convs = [self.conv_first]
        for rrdb in self.body:
            for rdb in (rrdb.rdb1, rrdb.rdb2, rrdb.rdb3):
                convs += [rdb.conv1, rdb.conv2, rdb.conv3, rdb.conv4, rdb.conv5]
        return convs + [self.conv_body, self.conv_up1, self.conv_up2, self.conv_hr, self.conv_last]

    def net_desc(self) -> dict:
        return dict(in_channels=self.conv_first.in_channels, out_channels=self.conv_last.out_channels,
                    channels=self.conv_first.out_channels, growth=self.body[0].rdb1.conv1.out_channels, num_blocks=len(self.body),
                    n_up=2, pixel_unshuffle=self._pixel_unshuffle, clamp=0)

    def _forward_impl(self, x: torch.Tensor) -> torch.Tensor:
        if self._pixel_unshuffle > 1:  # pure data movement on the few input channels; kept as the torch op
            x = F.pixel_unshuffle(x, self._pixel_unshuffle)
        if x.dim() == 4 and not x.is_cuda:
            return self._eager_forward(x)
        return _function.generator_forward(self, x)

    def _eager_forward(self, x: torch.Tensor) -> torch.Tensor:
        feat = self.conv_first(x)
        feat = feat + self.conv_body(_function.eager_trunk(self.body, feat))
        feat = self.lrelu(self.conv_up1(F.interpolate(feat, scale_factor=2, mode="nearest")))
        feat = self.lrelu(self.conv_up2(F.interpolate(feat, scale_factor=2, mode="nearest")))
        return self.conv_last(self.lrelu(self.conv_hr(feat)))


_BASICSR_CHILDREN = ["conv_first", "body", "conv_body", "conv_up1", "conv_up2", "conv_hr", "conv_last", "lrelu"]


def native_generator(model: nn.Module) -> BasicSRRRDBNet:
    """A :class:`BasicSRRRDBNet` that adopts the children of ``model``, a module of BasicSR's ``RRDBNet`` layout (for example an
    instance of BasicSR's own class).  The same module objects are kept: Parameter identity, optimizer state and the ``state_dict``
    (keys, order and values) are unchanged.  Usage: ``net = native_generator(net)``.

    ``model`` must have exactly the children ``conv_first``, ``body``, ``conv_body``, ``conv_up1``, ``conv_up2``, ``conv_hr``,
    ``conv_last``, ``lrelu`` in that order, a ``scale`` of 1, 2 or 4, 64 features, a ``body`` that :func:`native_trunk` accepts,
    3x3 convs with bias, a LeakyReLU(0.2) and no other parameters or buffers.  Anything else raises ``ValueError``."""
    if isinstance(model, BasicSRRRDBNet):
        return model
    names = [n for n, _ in model.named_children()]
    if names != _BASICSR_CHILDREN:
        raise ValueError(f"expected the children {_BASICSR_CHILDREN} of BasicSR's RRDBNet, got {names}")
    if any(True for _ in model.named_parameters(recurse=False)) or any(True for _ in model.named_buffers(recurse=False)):
        raise ValueError("the model holds parameters or buffers of its own besides its children's")
    scale = getattr(model, "scale", None)
    if scale not in (1, 2, 4):
        raise ValueError(f"the BasicSR layout runs natively at scale 1, 2 and 4, got {scale!r}")
    unshuffle = {4: 1, 2: 2, 1: 4}[scale]
    cin, cout = model.conv_first.in_channels, model.conv_last.out_channels
    if cin % (unshuffle * unshuffle) or not 1 <= cin <= 64:
        raise ValueError(f"conv_first takes {cin} channels: not a multiple of {unshuffle * unshuffle} in [1, 64] (scale {scale})")
    if not 1 <= cout <= 16:
        raise ValueError(f"conv_last gives {cout} channels, the native tail supports 1..16")
    for name, ci, co in (("conv_first", cin, 64), ("conv_body", 64, 64), ("conv_up1", 64, 64), ("conv_up2", 64, 64),
                         ("conv_hr", 64, 64), ("conv_last", 64, cout)):
        conv = getattr(model, name)
        _check_conv3x3(conv, name, ci, co)
        if [n for n, _ in conv.named_parameters()] != ["weight", "bias"] or any(True for _ in conv.named_buffers()):
            raise ValueError(f"{name}: expected the parameters weight and bias and nothing else")
    if not (type(model.lrelu) is nn.LeakyReLU and model.lrelu.negative_slope == 0.2):
        raise ValueError(f"lrelu: expected LeakyReLU(negative_slope=0.2), got {model.lrelu!r}")
    _check_rrdb_stack(model.body)
    net = BasicSRRRDBNet.__new__(BasicSRRRDBNet)
    nn.Module.__init__(net)
    net._set_scale(scale)
    for name, child in model.named_children():
        net.add_module(name, child)
    net.train(model.training)
    return net


# --- factories (names the reference scripts look up with model.__dict__[arch]) ------------------------------------
def rrdbnet_x1(**kwargs: Any) -> RRDBNet:
    return RRDBNet(upscale_factor=1, **kwargs)


def rrdbnet_x2(**kwargs: Any) -> RRDBNet:
    return RRDBNet(upscale_factor=2, **kwargs)


def rrdbnet_x4(**kwargs: Any) -> RRDBNet:
    return RRDBNet(upscale_factor=4, **kwargs)


def rrdbnet_x8(**kwargs: Any) -> RRDBNet:
    return RRDBNet(upscale_factor=8, **kwargs)


def bsrgan_x2(**kwargs: Any) -> BSRGAN:
    print("* BSRGAN 2x")  # BSRGAN/model.py:577
    return BSRGAN(upscale_factor=2, **kwargs)


def bsrgan_x4(**kwargs: Any) -> BSRGAN:
    print("* BSRGAN 4x")  # BSRGAN/model.py:584
    return BSRGAN(upscale_factor=4, **kwargs)


def real_rrdbnet_x4(**kwargs: Any) -> RealRRDBNet:
    return RealRRDBNet(upscale_factor=4, **kwargs)
