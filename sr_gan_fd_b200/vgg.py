"""VGG19 perceptual "content" loss next to the generator path (SURVEY.md section 8f, rank 3).

Drop-ins for the reference's two ``ContentLoss`` flavours:

* :class:`ContentLoss` -- ``ESRGAN/model.py:246-292``: ``ContentLoss(feature_model_extractor_node, mean, std)(sr, gt)`` -> scalar
  ``l1_loss(f(sr), f(gt))`` at ONE node, differentiable w.r.t. ``sr`` (``train_esrgan.py`` back-propagates it into the generator);
* :class:`ContentLossMulti` -- ``BSRGAN/model.py:501-554`` (= Real_ESRGAN, A-ESRGAN): a LIST of nodes, returns
  ``torch.Tensor([losses])`` of shape [1, n] which -- exactly as in the reference -- carries no gradient.

Both build torchvision's VGG19 the way the reference does (``models.vgg19(weights=IMAGENET1K_V1)`` +
``create_feature_extractor``; frozen, eval), so the module tree / ``state_dict`` are the reference's.  CUDA fp32 inputs run the
sixteen 3x3 convs on the tcgen05 chain kernel of libb200sr.so (bf16 operands, fp32 accumulation; sr and gt as ONE batch; the
feature nodes are kept in fp32 -- the LAST requested node before its ReLU, every earlier node AFTER it, because that is what
torchvision hands the reference: its in-place ReLUs overwrite each extracted conv output except the one that ends the graph),
max-pools / normalisation / the L1 reduction and, for the ESRGAN flavour, the data-gradient chain back to ``sr`` as small fused
kernels (ReLU + max-pool backward in one pass).  Anything else (CPU tensors, nodes that are not
conv outputs, other dtypes) takes the reference's op sequence through ``self.feature_extractor``.
"""
from __future__ import annotations

import ctypes as C
from typing import List, Optional, Sequence

import torch
import torch.nn.functional as F
import torchvision.models as models
from torch import nn
from torchvision import transforms
from torchvision.models.feature_extraction import create_feature_extractor

from . import lib as _lib

__all__ = ["ContentLoss", "ContentLossMulti", "VGG_CONV_NODES"]

# torchvision vgg19().features indices of the sixteen convs (conv1_1 ... conv5_4); a node "features.<i>" with i in this list is
# that conv's output
VGG_CONV_NODES = [0, 2, 5, 7, 10, 12, 14, 16, 19, 21, 23, 25, 28, 30, 32, 34]
_COUT = [64, 64, 128, 128, 256, 256, 256, 256, 512, 512, 512, 512, 512, 512, 512, 512]
_POOL_AFTER = [False, True, False, True, False, False, False, True, False, False, False, True, False, False, False, False]


def _conv_index(node: str) -> Optional[int]:
    if node.startswith("features."):
        try:
            i = int(node.split(".")[1])
        except ValueError:
            return None
        return VGG_CONV_NODES.index(i) if i in VGG_CONV_NODES else None
    return None


class _VggRuntime:
    """Native state of one loss module: packed weights and plans per (geometry, gradient request)."""

    def __init__(self) -> None:
        self.plans = {}
        self.packed = {}

    def plan(self, batch, h, w, last_conv, feat_mask, grad_conv, grad_images, mean, std, deterministic=False):
        key = (batch, h, w, last_conv, feat_mask, grad_conv, grad_images, deterministic)
        p = self.plans.get(key)
        if p is None:
            d = _lib.VggDesc(batch, h, w, last_conv, feat_mask, grad_conv, grad_images, (C.c_float * 3)(*mean), (C.c_float * 3)(*std),
                             1 if deterministic else 0)
            handle = C.c_void_p()
            lib = _lib.load()
            _lib.check(lib.b200sr_vgg_plan_create(C.byref(d), C.byref(handle)))
            p = dict(handle=handle, ws_bytes=int(lib.b200sr_workspace_bytes(handle)), packed_bytes=int(lib.b200sr_packed_bytes(handle)),
                     layout=int(lib.b200sr_pack_layout_id(handle)))
            if len(self.plans) >= 6:
                old = self.plans.pop(next(iter(self.plans)))
                lib.b200sr_plan_destroy(old["handle"])
            self.plans[key] = p
        return p

    def packed_for(self, plan, params: List[torch.Tensor], stream: int) -> torch.Tensor:
        key = (plan["layout"], tuple(p.data_ptr() for p in params), tuple(p._version for p in params))
        ent = self.packed.get(plan["layout"])
        if ent is not None and ent[0] == key:
            return ent[1]
        buf = torch.empty(plan["packed_bytes"], dtype=torch.uint8, device=params[0].device)
        ptrs = (C.c_void_p * len(params))(*[p.data_ptr() for p in params])
        _lib.check(_lib.load().b200sr_pack_weights(plan["handle"], ptrs, C.c_void_p(buf.data_ptr()), C.c_void_p(stream)))
        self.packed[plan["layout"]] = (key, buf)
        return buf


def _feature_numel(conv: int, pairs: int, h: int, w: int) -> int:
    for l in range(conv):
        if _POOL_AFTER[l]:
            h //= 2
            w //= 2
    return pairs * h * w * _COUT[conv]


class _VggL1Fn(torch.autograd.Function):
    """mean |f(sr) - f(gt)| at one conv node, with the gradient w.r.t. sr from the native data-gradient chain."""

    @staticmethod
    def forward(ctx, sr, gt, owner, conv):
        loss, plan, ws, packed = owner._native_losses(sr, gt, [conv], grad_conv=conv)
        ctx.owner, ctx.plan, ctx.ws, ctx.packed = owner, plan, ws, packed
        ctx.shape = tuple(sr.shape)
        return loss[0].float()

    @staticmethod
    def backward(ctx, g):
        owner = ctx.owner
        dx = torch.empty(ctx.shape, dtype=torch.float32, device=g.device)
        up = g.detach().reshape(1).float().contiguous()
        with torch.cuda.device(g.device):
            _lib.check(_lib.load().b200sr_vgg_backward(ctx.plan["handle"], C.c_void_p(up.data_ptr()), C.c_void_p(ctx.packed.data_ptr()),
                                                       C.c_void_p(ctx.ws.data_ptr()), C.c_void_p(dx.data_ptr()),
                                                       C.c_void_p(torch.cuda.current_stream().cuda_stream)))
        ctx.ws = None
        std = torch.tensor(owner._std, dtype=torch.float32, device=g.device).view(1, 3, 1, 1)
        return dx / std, None, None, None  # the chain differentiates w.r.t. the NORMALISED image


class _ContentLossBase(nn.Module):
    use_native = True  # A/B switch (benchmarks): False sends CUDA tensors through the stock torch ops as well

    def _setup(self, nodes: Sequence[str], mean, std) -> None:
        # exactly the reference's construction (ESRGAN/model.py:266-281): torchvision VGG19, frozen, eval
        model = models.vgg19(weights=models.VGG19_Weights.IMAGENET1K_V1)
        self.feature_extractor = create_feature_extractor(model, list(nodes))
        self.feature_extractor.eval()
        self.normalize = transforms.Normalize(mean, std)
        for p in self.feature_extractor.parameters():
            p.requires_grad = False
        self._mean, self._std = [float(v) for v in mean], [float(v) for v in std]
        self._convs = [_conv_index(n) for n in nodes]

    def _vgg_params(self) -> List[torch.Tensor]:
        feats = self.feature_extractor.features
        last = max(self._convs)
        out = []
        for l in range(last + 1):
            conv = getattr(feats, str(VGG_CONV_NODES[l]))
            out += [conv.weight, conv.bias]
        return out

    def _native_ok(self, sr: torch.Tensor, gt: torch.Tensor) -> bool:
        return (self.use_native and all(c is not None for c in self._convs) and sr.is_cuda and gt.is_cuda and sr.dtype == torch.float32 and gt.dtype == torch.float32
                and sr.dim() == 4 and sr.shape[1] == 3 and sr.shape == gt.shape and len(self._mean) == 3)

    def _native_losses(self, sr, gt, convs, grad_conv=-1):
        rt = self.__dict__.setdefault("_b200_vgg", _VggRuntime())
        pairs, _, h, w = sr.shape
        x = torch.cat([sr.detach(), gt.detach()], 0).contiguous()
        mask = 0
        for c in convs:
            mask |= 1 << c
        params = self._vgg_params()
        lib = _lib.load()
        with torch.cuda.device(sr.device):
            stream = torch.cuda.current_stream().cuda_stream
            plan = rt.plan(2 * pairs, h, w, max(convs), mask, grad_conv, pairs if grad_conv >= 0 else 0, self._mean, self._std,
                           _lib.deterministic())
            packed = rt.packed_for(plan, params, stream)
            ws = torch.empty(plan["ws_bytes"], dtype=torch.uint8, device=sr.device)
            strides = (C.c_int64 * 4)(*x.stride())
            _lib.check(lib.b200sr_vgg_forward(plan["handle"], C.c_void_p(x.data_ptr()), strides, C.c_void_p(packed.data_ptr()),
                                              C.c_void_p(ws.data_ptr()), C.c_void_p(stream)))
            sums = torch.empty(len(convs), dtype=torch.float64, device=sr.device)
            for i, c in enumerate(convs):
                _lib.check(lib.b200sr_vgg_feature_l1(plan["handle"], C.c_void_p(ws.data_ptr()), c, pairs, C.c_void_p(sums[i:].data_ptr()), C.c_void_p(stream)))
        counts = torch.tensor([_feature_numel(c, pairs, h, w) for c in convs], dtype=torch.float64, device=sr.device)
        return sums / counts, plan, ws, packed

    def __getstate__(self):
        state = self.__dict__.copy()
        state.pop("_b200_vgg", None)
        return state


class ContentLoss(_ContentLossBase):
    """``ESRGAN/model.py:246-292``: one node, scalar loss, gradient flows to ``sr_tensor``."""

    def __init__(self, feature_model_extractor_node: str, feature_model_normalize_mean: list, feature_model_normalize_std: list) -> None:
        super().__init__()
        self.feature_model_extractor_node = feature_model_extractor_node
        self._setup([feature_model_extractor_node], feature_model_normalize_mean, feature_model_normalize_std)

    def forward(self, sr_tensor: torch.Tensor, gt_tensor: torch.Tensor) -> torch.Tensor:
        if self._native_ok(sr_tensor, gt_tensor):
            if torch.is_grad_enabled() and sr_tensor.requires_grad:
                return _VggL1Fn.apply(sr_tensor, gt_tensor, self, self._convs[0])
            return self._native_losses(sr_tensor, gt_tensor, [self._convs[0]])[0][0].float()
        return self._torch_forward(sr_tensor, gt_tensor)

    def _torch_forward(self, sr_tensor: torch.Tensor, gt_tensor: torch.Tensor) -> torch.Tensor:
        """The reference's op sequence (ESRGAN/model.py:283-292)."""
        sr_tensor, gt_tensor = self.normalize(sr_tensor), self.normalize(gt_tensor)
        node = self.feature_model_extractor_node
        return F.l1_loss(self.feature_extractor(sr_tensor)[node], self.feature_extractor(gt_tensor)[node])


class ContentLossMulti(_ContentLossBase):
    """``BSRGAN/model.py:501-554``: several nodes, returns ``torch.Tensor([losses])`` ([1, n], no gradient -- as the reference)."""

    def __init__(self, feature_model_extractor_nodes: list, feature_model_normalize_mean: list, feature_model_normalize_std: list) -> None:
        super().__init__()
        self.feature_model_extractor_nodes = feature_model_extractor_nodes
        self._setup(feature_model_extractor_nodes, feature_model_normalize_mean, feature_model_normalize_std)

    def forward(self, sr_tensor: torch.Tensor, gt_tensor: torch.Tensor) -> torch.Tensor:
        assert sr_tensor.size() == gt_tensor.size(), "Two tensor must have the same size"
        if self._native_ok(sr_tensor, gt_tensor):
            losses = self._native_losses(sr_tensor, gt_tensor, list(self._convs))[0]
            return losses.float().view(1, -1)
        device = sr_tensor.device
        sr_tensor, gt_tensor = self.normalize(sr_tensor), self.normalize(gt_tensor)
        sr_feature, gt_feature = self.feature_extractor(sr_tensor), self.feature_extractor(gt_tensor)
        losses = [F.l1_loss(sr_feature[n], gt_feature[n]) for n in self.feature_model_extractor_nodes]
        return torch.Tensor([losses]).to(device=device)
