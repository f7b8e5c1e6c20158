"""U-Net discriminator next to the generator path (SURVEY.md section 8f, rank 2).

Drop-in for ``DiscriminatorUNet`` (``BSRGAN/model.py:91-167`` = ``Real_ESRGAN/model.py:29-105``) and its factory
``discriminator_unet`` (``BSRGAN/model.py:557-560``): same constructor, same children (real ``nn.Conv2d`` modules wrapped
by ``torch.nn.utils.spectral_norm`` in the reference's order, so ``state_dict`` keys -- ``*.weight_orig / weight_u / weight_v`` --
shapes and the RNG draw order of the initialisation are the reference's).

CUDA inputs run forward and backward inside libb200sr.so (``b200sr_disc_*`` in ``include/b200sr.h``): the ten convs on the tcgen05
chain / weight-gradient kernels (bf16 operands, fp32 accumulation; the 4x4 stride-2 convs as 3x3 convs over the pixel-unshuffled
input), bilinear upsampling + skip additions and their transposes as small fused kernels.  The spectral normalisation stays what it is
in the reference -- torch's own forward pre-hooks (power iteration on ``weight_u / weight_v`` in training mode, ``weight_orig / sigma``)
-- so the native path receives the EFFECTIVE weights and hands back their gradients; autograd carries them on to ``weight_orig``
through torch's graph of ``W / sigma``, exactly as in the reference.  A frozen discriminator (``requires_grad = False`` on its
parameters, the generator update of ``BSRGAN/train_bsrgan.py:441-463``) only runs the data-gradient kernels; an input without gradient
(the discriminator update, ``:414-436``) skips the input gradient.

CPU tensors, other channel widths, ``upsample_method != "bilinear"`` or sizes that are not multiples of 8 take the reference's op
sequence on the module's own children (stock torch ops).  A CUDA tensor that qualifies NEVER falls back: a missing library raises.
"""
from __future__ import annotations

import ctypes as C
from collections import OrderedDict
from typing import Any, List

import torch
import torch.nn.functional as F_torch
from torch import Tensor, nn
from torch.nn.utils import spectral_norm
from torch.nn.utils.spectral_norm import SpectralNorm

from . import lib as _lib

__all__ = ["DiscriminatorUNet", "discriminator_unet"]

_DTYPES = {torch.float32: _lib.F32, torch.float16: _lib.F16, torch.bfloat16: _lib.BF16}
_MAX_PLANS = 6


class _DiscPlan:
    def __init__(self, in_channels: int, out_channels: int, channels: int, batch: int, height: int, width: int, training: bool,
                 fp16: bool = True, deterministic: bool = False) -> None:
        lib = _lib.load()
        d = _lib.DiscDesc(in_channels, out_channels, channels, batch, height, width, 1 if training else 0, 1 if fp16 else 0,
                          1 if deterministic else 0)
        handle = C.c_void_p()
        _lib.check(lib.b200sr_disc_plan_create(C.byref(d), C.byref(handle)))
        self.handle = handle
        self.training = training
        self.deterministic = deterministic
        self.out_channels = out_channels
        self.workspace_bytes = int(lib.b200sr_workspace_bytes(handle))
        self.packed_bytes = int(lib.b200sr_packed_bytes(handle))
        self.param_numel = int(lib.b200sr_param_numel(handle))
        self.flops_fwd = float(lib.b200sr_flops(handle, 0))
        self.flops_bwd_d = float(lib.b200sr_flops(handle, 1))  # discriminator update: weight + data gradients
        self.flops_bwd_g = float(lib.b200sr_flops(handle, 2))  # generator update: data gradients only

    def __del__(self):
        try:
            if self.handle:
                _lib.load().b200sr_plan_destroy(self.handle)
                self.handle = None
        except Exception:
            pass


class _DiscRuntime:
    """Native state of one module (plans per geometry).  Lives in ``module.__dict__``; never pickled or deep-copied."""

    def __init__(self) -> None:
        self.plans: "OrderedDict[tuple, _DiscPlan]" = OrderedDict()
        self.last_plan = None

    def plan(self, module, device, batch, height, width, training) -> _DiscPlan:
        fp16 = module.operand_dtype == "fp16"
        det = _lib.deterministic()  # the backward runs in the forward's mode
        key = (device.index, batch, height, width, training, fp16, det)
        p = self.plans.get(key)
        if p is None:
            p = _DiscPlan(module._in_channels, module._out_channels, module._channels, batch, height, width, training, fp16, det)
            self.plans[key] = p
            while len(self.plans) > _MAX_PLANS:
                self.plans.popitem(last=False)
        else:
            self.plans.move_to_end(key)
        self.last_plan = p
        return p


class _DiscFn(torch.autograd.Function):
    """Whole-network autograd node: forward enqueues b200sr_disc_forward, backward b200sr_disc_backward."""

    @staticmethod
    def forward(ctx, module, x, *weights):
        lib = _lib.load()
        rt = module._runtime()
        n, _, h, w = x.shape
        # slots: weight, bias of conv1, down1..3, up1..3, conv2, conv3, conv4 (biases only for conv1 / conv4)
        w1, b1, d1, d2, d3, u1, u2, u3, c2, c3, w4, b4 = weights
        slots = [w1, b1, d1, None, d2, None, d3, None, u1, None, u2, None, u3, None, c2, None, c3, None, w4, b4]
        training = any(ctx.needs_input_grad[1:])
        with torch.cuda.device(x.device):
            stream = torch.cuda.current_stream().cuda_stream
            plan = rt.plan(module, x.device, n, h, w, training)
            # ONE allocation for the activations and this forward's packed weights (the spectral norm changes them on every call):
            # the library caches its TMA descriptors per (workspace, packed) address pair, and one large block is what the caching
            # allocator hands back at the same address call after call
            ws_bytes = (plan.workspace_bytes + 1023) // 1024 * 1024
            buf = torch.empty(ws_bytes + plan.packed_bytes, dtype=torch.uint8, device=x.device)
            workspace, packed = buf[:ws_bytes], buf[ws_bytes:]
            ptrs = (C.c_void_p * 20)(*[t.data_ptr() if t is not None else None for t in slots])
            _lib.check(lib.b200sr_pack_weights(plan.handle, ptrs, C.c_void_p(packed.data_ptr()), C.c_void_p(stream)))
            y = torch.empty((n, plan.out_channels, h, w), dtype=torch.float32, device=x.device)
            strides = (C.c_int64 * 4)(*x.stride())
            _lib.check(lib.b200sr_disc_forward(plan.handle, C.c_void_p(x.data_ptr()), _DTYPES[x.dtype], strides,
                                               C.c_void_p(packed.data_ptr()), C.c_void_p(workspace.data_ptr()),
                                               C.c_void_p(y.data_ptr()), C.c_void_p(stream)))
        if training:
            ctx.plan, ctx.workspace, ctx.packed = plan, workspace, packed
            ctx.x_meta = (tuple(x.shape), x.dtype)
            ctx.w_shapes = [tuple(t.shape) for t in weights]
        return y

    @staticmethod
    def backward(ctx, dy):
        lib = _lib.load()
        plan = ctx.plan
        if ctx.workspace is None:
            raise RuntimeError("the B200 discriminator supports one backward per forward (activations already released)")
        need = ctx.needs_input_grad
        want_w = any(need[2:])
        dy = dy.contiguous().float()
        with torch.cuda.device(dy.device):
            stream = torch.cuda.current_stream().cuda_stream
            flat = torch.empty(plan.param_numel, dtype=torch.float32, device=dy.device) if want_w else None
            dx = torch.empty(ctx.x_meta[0], dtype=torch.float32, device=dy.device) if need[1] else None
            _lib.check(lib.b200sr_disc_backward(plan.handle, C.c_void_p(dy.data_ptr()), C.c_void_p(ctx.packed.data_ptr()),
                                                C.c_void_p(ctx.workspace.data_ptr()),
                                                C.c_void_p(flat.data_ptr()) if flat is not None else None,
                                                C.c_void_p(dx.data_ptr()) if dx is not None else None, C.c_void_p(stream)))
        ctx.workspace = None
        if dx is not None and ctx.x_meta[1] != torch.float32:
            dx = dx.to(ctx.x_meta[1])
        grads: List[Any] = [None] * len(ctx.w_shapes)
        if flat is not None:
            numels = [int(torch.Size(s).numel()) for s in ctx.w_shapes]
            for i, (piece, shp) in enumerate(zip(flat.split(numels), ctx.w_shapes)):
                if need[2 + i]:
                    grads[i] = piece.view(shp)
        return (None, dx, *grads)


class DiscriminatorUNet(nn.Module):
    """``BSRGAN/model.py:91-167``.  Same constructor arguments, children and ``state_dict`` as the reference class."""

    use_native = True  # A/B switch (benchmarks): False sends CUDA tensors through the stock torch ops as well
    # 16-bit format of the native path's activations, packed weights and gradients (fp32 accumulation either way): "fp16" is what the
    # reference's scripts run this module in (torch.autocast's CUDA default, BSRGAN/train_bsrgan.py:415,425,447) and, with an 11-bit
    # mantissa, six times closer to fp32 than "bf16", which in turn cannot overflow under an aggressive GradScaler scale
    operand_dtype = "fp16"

    def __init__(
            self,
            in_channels: int,
            out_channels: int,
            channels: int,
            upsample_method: str = "bilinear",
    ) -> None:
        super(DiscriminatorUNet, self).__init__()
        self.upsample_method = upsample_method
        self._in_channels, self._out_channels, self._channels = int(in_channels), int(out_channels), int(channels)

        # construction order = the reference's (BSRGAN/model.py:102-135): every spectral_norm draws weight_u / weight_v right after
        # its conv's own initialisation, so a seeded construction reproduces the reference's tensors
        def sn_block(cin: int, cout: int, k: int, stride: int) -> nn.Sequential:
            return nn.Sequential(spectral_norm(nn.Conv2d(cin, cout, (k, k), (stride, stride), (1, 1), bias=False)), nn.LeakyReLU(0.2, True))

        c = channels
        self.conv1 = nn.Conv2d(in_channels, 64, (3, 3), (1, 1), (1, 1))
        self.down_block1 = sn_block(c, int(c * 2), 4, 2)
        self.down_block2 = sn_block(int(c * 2), int(c * 4), 4, 2)
        self.down_block3 = sn_block(int(c * 4), int(c * 8), 4, 2)
        self.up_block1 = sn_block(int(c * 8), int(c * 4), 3, 1)
        self.up_block2 = sn_block(int(c * 4), int(c * 2), 3, 1)
        self.up_block3 = sn_block(int(c * 2), c, 3, 1)
        self.conv2 = sn_block(c, c, 3, 1)
        self.conv3 = sn_block(c, c, 3, 1)
        self.conv4 = nn.Conv2d(c, out_channels, (3, 3), (1, 1), (1, 1))

    # ------------------------------------------------------------------------------------------------------------------
    def _runtime(self) -> _DiscRuntime:
        rt = self.__dict__.get("_b200_disc")
        if rt is None:
            rt = _DiscRuntime()
            self.__dict__["_b200_disc"] = rt
        return rt

    def __getstate__(self):
        state = self.__dict__.copy()
        state.pop("_b200_disc", None)
        return state

    def __deepcopy__(self, memo):
        import copy
        cls = self.__class__
        new = cls.__new__(cls)
        memo[id(self)] = new
        for k, v in self.__dict__.items():
            if k != "_b200_disc":
                new.__dict__[k] = copy.deepcopy(v, memo)
        return new

    def _sn_convs(self) -> List[nn.Conv2d]:
        return [self.down_block1[0], self.down_block2[0], self.down_block3[0], self.up_block1[0], self.up_block2[0],
                self.up_block3[0], self.conv2[0], self.conv3[0]]

    def _native_ok(self, x: Tensor) -> bool:
        return (self.use_native and x.is_cuda and x.dim() == 4 and self._channels == 64 and self.upsample_method == "bilinear"
                and 1 <= self._in_channels <= 16 and 1 <= self._out_channels <= 16 and x.shape[1] == self._in_channels
                and x.shape[2] >= 8 and x.shape[3] >= 8 and x.shape[2] % 8 == 0 and x.shape[3] % 8 == 0
                and self.conv1.weight.is_cuda)

    @staticmethod
    def _effective_weight(conv: nn.Conv2d) -> Tensor:
        """Run the conv's spectral-norm forward pre-hook (what ``conv(x)`` would do first: one power iteration in training mode,
        then ``weight = weight_orig / sigma``, ``torch/nn/utils/spectral_norm.py``) and return the weight it leaves on the module."""
        for hook in conv._forward_pre_hooks.values():
            if isinstance(hook, SpectralNorm):
                hook(conv, (None,))
        return conv.weight

    def forward(self, x: Tensor) -> Tensor:
        return self._forward_impl(x)

    # Support torch.script function
    def _forward_impl(self, x: Tensor) -> Tensor:
        if not self._native_ok(x):
            return self._torch_forward(x)
        if x.dtype not in _DTYPES:
            x = x.float()
        weights = [self.conv1.weight, self.conv1.bias] + [self._effective_weight(c) for c in self._sn_convs()] + \
                  [self.conv4.weight, self.conv4.bias]
        with torch.autocast("cuda", enabled=False):
            weights = [t.float().contiguous() for t in weights]
            return _DiscFn.apply(self, x, *weights)

    def _torch_forward(self, x: Tensor) -> Tensor:
        """The reference's graph (BSRGAN/model.py:143-167) on this module's own children, stock torch ops."""
        def up(t: Tensor) -> Tensor:
            return F_torch.interpolate(t, scale_factor=2, mode="bilinear", align_corners=False)

        out1 = self.conv1(x)
        down1 = self.down_block1(out1)
        down2 = self.down_block2(down1)
        down3 = self.down_block3(down2)
        t = self.up_block1(up(down3)) + down2
        t = self.up_block2(up(t)) + down1
        t = self.up_block3(up(t)) + out1
        return self.conv4(self.conv3(self.conv2(t)))


def discriminator_unet(**kwargs: Any) -> DiscriminatorUNet:
    """``BSRGAN/model.py:557-560``."""
    model = DiscriminatorUNet(**kwargs)
    return model
