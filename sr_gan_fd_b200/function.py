"""The one ``torch.autograd.Function`` behind the drop-in generators: forward and backward of the whole RRDBNet
run inside libb200sr.so (C ABI, ``include/b200sr.h``).  PyTorch is used only for device memory, streams and autograd
bookkeeping.

Replaces, in the reference, the eager module calls ``ESRGAN/model.py:211-232`` (forward) and the autograd graph that
``scaler.scale(loss).backward()`` walks (``ESRGAN/train_rrdbnet.py:261``, ``BSRGAN/train_bsrgan.py:463``).
"""
from __future__ import annotations

import ctypes as C
from collections import OrderedDict
from typing import Callable, List, Optional

import torch

from . import lib as _lib

_DTYPES = {torch.float32: _lib.F32, torch.float16: _lib.F16, torch.bfloat16: _lib.BF16}
_MAX_PLANS = 8
_MAX_PACKED = 4  # packed-weight buffers kept per module ((training, pack layout) pairs; ~40 MB each for the x4 net)


class _Plan:
    def __init__(self, desc: dict, batch: int, height: int, width: int, training: bool, grad_bucket_rrdbs: int = 0,
                 deterministic: bool = False) -> None:
        lib = _lib.load()
        nd = _lib.NetDesc(desc["in_channels"], desc["out_channels"], desc["channels"], desc["growth"],
                          desc["num_blocks"], desc["n_up"], batch, height, width, 1 if training else 0, grad_bucket_rrdbs,
                          1 if deterministic else 0)
        handle = C.c_void_p()
        if desc.get("trunk_only"):
            create = lib.b200sr_trunk_plan_create
        elif desc.get("clamp", 1) == 0:  # generators whose output is conv4's (BasicSR layout)
            create = lib.b200sr_unclamped_plan_create
        else:
            create = lib.b200sr_plan_create
        _lib.check(create(C.byref(nd), C.byref(handle)))
        self.handle = handle
        self.training = training
        self.deterministic = deterministic
        self.geometry = (batch, height, width)
        self.scale = 1 << desc["n_up"]
        self.out_channels = desc["out_channels"]
        self.workspace_bytes = int(lib.b200sr_workspace_bytes(handle))
        self.packed_bytes = int(lib.b200sr_packed_bytes(handle))
        self.pack_layout = int(lib.b200sr_pack_layout_id(handle))
        self.num_params = int(lib.b200sr_num_params(handle))
        self.param_numel = int(lib.b200sr_param_numel(handle))
        self.flops_fwd = float(lib.b200sr_flops(handle, 0))
        self.flops_bwd = float(lib.b200sr_flops(handle, 1))
        self.launches_fwd = int(lib.b200sr_num_launches(handle, 0))
        self.launches_bwd = int(lib.b200sr_num_launches(handle, 1)) if training else 0
        self.launches_bwd_bucketed = int(lib.b200sr_num_launches(handle, 2)) if training else 0

    def backward_launches(self, need_params=None, with_dx: bool = False, with_cb: bool = False) -> int:
        """Kernel launches of one backward that computes the gradients of the parameters flagged in ``need_params``
        (state_dict order; None: all of them), the input gradient if ``with_dx``, with a bucket callback if ``with_cb``."""
        mask = conv_mask(need_params) if need_params is not None else None
        return int(_lib.load().b200sr_backward_launches(self.handle, mask, int(with_dx), int(with_cb)))

    def __del__(self):
        try:
            if self.handle:
                _lib.load().b200sr_plan_destroy(self.handle)
                self.handle = None
        except Exception:
            pass


class GeneratorRuntime:
    """Per-module native state (plans, packed weights).  Lives in ``module.__dict__['_b200_runtime']`` and is never
    pickled, deep-copied or registered as a buffer (``AveragedModel`` zips buffers with strict=True)."""

    def __init__(self) -> None:
        self.plans: "OrderedDict[tuple, _Plan]" = OrderedDict()
        self.packed = OrderedDict()  # (training, pack layout) -> uint8 tensor
        self.packed_key = {}    # (training, pack layout) -> (versions, ptrs)
        self.pack_serial = {}
        # optional hook(flat_grads: Tensor, offset: int, count: int) called as gradient buckets are enqueued
        self.grad_bucket_hook: Optional[Callable[[torch.Tensor, int, int], None]] = None
        # optional hook(flat_grads) called once backward has enqueued all of its kernels
        self.grad_done_hook: Optional[Callable[[torch.Tensor], None]] = None
        self.grad_bucket_rrdbs = 0  # RRDBs per announced gradient bucket (0: one)
        self.last_plan: Optional[_Plan] = None
        # host fast path: the conv modules in state_dict order, and what was already validated about their parameters
        self.convs = None
        self.checked_ptrs = None
        self.param_shapes = None
        self.param_numels = None
        self.cur_key = None

    def plan(self, desc: dict, device: torch.device, batch: int, height: int, width: int, training: bool,
             deterministic: bool = False) -> _Plan:
        key = (device.index, batch, height, width, training, self.grad_bucket_rrdbs, deterministic)
        p = self.plans.get(key)
        if p is None:
            p = _Plan(desc, batch, height, width, training, self.grad_bucket_rrdbs, deterministic)
            self.plans[key] = p
            while len(self.plans) > _MAX_PLANS:
                self.plans.popitem(last=False)
        else:
            self.plans.move_to_end(key)
        self.last_plan = p
        return p

    def packed_weights(self, plan: _Plan, params: List[torch.Tensor], stream: int, key=None) -> torch.Tensor:
        # one packed buffer per (training, pack layout): the dense-block schedule -- and with it the packing -- depends on
        # the geometry (windowed re-association for small batches, per-conv for large frames)
        slot = (plan.training, plan.pack_layout)
        if key is None:
            key = (tuple([p._version for p in params]), tuple([p.data_ptr() for p in params]))
        buf = self.packed.get(slot)
        if buf is not None and buf.device == params[0].device and self.packed_key.get(slot) == key:
            self.packed.move_to_end(slot)
            return buf
        if buf is None or buf.device != params[0].device or buf.numel() != plan.packed_bytes:
            buf = torch.empty(plan.packed_bytes, dtype=torch.uint8, device=params[0].device)
            self.packed[slot] = buf
            while len(self.packed) > _MAX_PACKED:
                old, _ = self.packed.popitem(last=False)
                self.packed_key.pop(old, None)
        self.packed.move_to_end(slot)
        ptrs = (C.c_void_p * len(params))(*key[1])
        _lib.check(_lib.load().b200sr_pack_weights(plan.handle, ptrs, C.c_void_p(buf.data_ptr()), C.c_void_p(stream)))
        self.packed_key[slot] = key
        self.pack_serial[slot] = self.pack_serial.get(slot, 0) + 1
        return buf


class _Launched:
    """What one enqueued native forward leaves behind (handed to the autograd Function as a non-tensor argument)."""
    __slots__ = ("y", "plan", "rt", "workspace", "packed", "pack_slot", "pack_serial")


def _launch_forward(module, rt: "GeneratorRuntime", x: torch.Tensor, training: bool, params) -> _Launched:
    """Enqueue the whole native forward NOW.  It runs before the autograd bookkeeping of the 702-input Function, so the GPU
    is already working while the host builds the graph (the host path in front of the first kernel is what an end-to-end
    step with a per-step ``loss.item()`` pays in full)."""
    lib = _lib.load()
    desc = module.net_desc()
    n, c, h, w = x.shape
    if c != desc["in_channels"]:
        raise RuntimeError(f"expected {desc['in_channels']} input channels, got {c}")
    st = _Launched()
    with torch.cuda.device(x.device):
        stream = torch.cuda.current_stream().cuda_stream
        plan = rt.plan(desc, x.device, n, h, w, training, _lib.deterministic())  # the backward runs in the forward's mode
        packed = rt.packed_weights(plan, params, stream, rt.cur_key)
        workspace = torch.empty(plan.workspace_bytes, dtype=torch.uint8, device=x.device)
        y = torch.empty((n, plan.out_channels, h * plan.scale, w * plan.scale), dtype=torch.float32, device=x.device)
        strides = (C.c_int64 * 4)(*x.stride())
        _lib.check(lib.b200sr_forward(plan.handle, C.c_void_p(x.data_ptr()), _DTYPES[x.dtype], strides,
                                      C.c_void_p(packed.data_ptr()), C.c_void_p(workspace.data_ptr()),
                                      C.c_void_p(y.data_ptr()), C.c_void_p(stream)))
    st.y, st.plan, st.rt, st.workspace, st.packed = y, plan, rt, workspace, packed
    st.pack_slot = (training, plan.pack_layout)
    st.pack_serial = rt.pack_serial[st.pack_slot]
    return st


class _RRDBNetFn(torch.autograd.Function):
    """Autograd node of one (already enqueued) training forward: keeps the workspace alive and runs the native backward."""

    @staticmethod
    def forward(ctx, launched: _Launched, x, *params):
        ctx.plan = launched.plan
        ctx.rt = launched.rt
        ctx.workspace = launched.workspace
        ctx.packed = launched.packed
        ctx.pack_slot = launched.pack_slot
        ctx.pack_serial = launched.pack_serial
        ctx.x_keepalive = x
        ctx.x_meta = (tuple(x.shape), x.dtype)
        return launched.y

    @staticmethod
    def backward(ctx, dy):
        lib = _lib.load()
        plan: _Plan = ctx.plan
        rt: GeneratorRuntime = ctx.rt
        if ctx.workspace is None:
            raise RuntimeError("the B200 generator supports one backward per forward (activations already released)")
        if rt.pack_serial.get(ctx.pack_slot) != ctx.pack_serial:
            raise RuntimeError("generator weights were re-packed between this forward and its backward")
        dy = dy.contiguous().float()
        need = ctx.needs_input_grad
        need_params = need[2:]
        all_params = all(need_params)
        any_params = all_params or any(need_params)
        with torch.cuda.device(dy.device):
            stream = torch.cuda.current_stream().cuda_stream
            flat = None
            if any_params:
                flat = torch.empty(plan.param_numel, dtype=torch.float32, device=dy.device)  # fresh per backward
            hook = rt.grad_bucket_hook
            if hook is not None and flat is not None:
                cb = _lib.BUCKET_CB(lambda user, off, cnt: hook(flat, int(off), int(cnt)))
            else:
                cb = _lib.BUCKET_CB()
            dx = None
            if need[1]:  # gradient w.r.t. the LR input: conv1's data gradient, fp32 NCHW (only when x.requires_grad)
                dx = torch.empty(ctx.x_meta[0], dtype=torch.float32, device=dy.device)
            args = (plan.handle, C.c_void_p(dy.data_ptr()), C.c_void_p(ctx.packed.data_ptr()), C.c_void_p(ctx.workspace.data_ptr()),
                    C.c_void_p(flat.data_ptr()) if flat is not None else None, C.c_void_p(dx.data_ptr()) if dx is not None else None)
            if all_params:
                _lib.check(lib.b200sr_backward(*args, cb, None, C.c_void_p(stream)))
            else:  # frozen or partially frozen generator: only what autograd asks for is computed
                mask = conv_mask(need_params) if any_params else None
                _lib.check(lib.b200sr_backward_select(*args, mask, cb, None, C.c_void_p(stream)))
            if rt.grad_done_hook is not None and flat is not None:
                rt.grad_done_hook(flat)
        ctx.workspace = None
        ctx.x_keepalive = None
        if dx is not None and ctx.x_meta[1] != torch.float32:
            dx = dx.to(ctx.x_meta[1])
        if flat is None:
            return (None, dx, *([None] * len(need_params)))
        pieces = flat.split(rt.param_numels)  # one call: 702 views of the flat gradient buffer, state_dict order
        grads = [t.view(shp) if need_params[i] else None for i, (t, shp) in enumerate(zip(pieces, rt.param_shapes))]
        return (None, dx, *grads)


def conv_mask(need_params) -> "C.Array":
    """Per-conv byte mask of ``b200sr_backward_select`` from per-parameter flags (weight, bias pairs in state_dict order):
    a conv is wanted when its weight or its bias is."""
    flags = [bool(need_params[i] or need_params[i + 1]) for i in range(0, len(need_params), 2)]
    return (C.c_uint8 * len(flags))(*flags)


def generator_forward(module, x: torch.Tensor) -> torch.Tensor:
    """Entry used by the drop-in modules' ``forward`` (generators and :class:`~sr_gan_fd_b200.rrdbnet.RRDBTrunk`: the module's
    ``net_desc()`` says which plan it runs, its ``_conv_list()`` which parameters)."""
    if x.dim() != 4:
        raise RuntimeError(f"expected NCHW input, got shape {tuple(x.shape)}")
    if not x.is_cuda:
        # CPU tensors (the reference scripts' default ``--device_type cpu``, ESRGAN/inference.py:92-99) take the module's own
        # nn.Conv2d children through plain torch ops.  This is NOT a fallback for the CUDA path: a CUDA tensor always goes to
        # libb200sr.so and raises if the library is missing.
        return eager_forward(module, x)
    if x.dtype not in _DTYPES:
        x = x.float()
    rt = module._runtime()
    if rt.convs is None:
        rt.convs = module._conv_list()
    params = []
    add = params.append
    for conv in rt.convs:  # read through _parameters so that re-assigned Parameters are picked up
        pd = conv._parameters
        add(pd["weight"])
        add(pd["bias"])
    ptrs = tuple([p.data_ptr() for p in params])
    if ptrs != rt.checked_ptrs:  # dtype / layout can only change together with the storage
        for p in params:
            if p.dtype != torch.float32 or not p.is_contiguous() or p.device != x.device:
                raise RuntimeError("generator parameters must be contiguous fp32 tensors on the input's device")
        rt.checked_ptrs = ptrs
        rt.param_shapes = [tuple(p.shape) for p in params]
        rt.param_numels = [p.numel() for p in params]
    elif params[0].device != x.device:
        raise RuntimeError("generator parameters must be contiguous fp32 tensors on the input's device")
    rt.cur_key = (tuple([p._version for p in params]), ptrs)
    training = torch.is_grad_enabled() and (x.requires_grad or any(p.requires_grad for p in params))
    launched = _launch_forward(module, rt, x, training, params)
    if not training:
        return launched.y  # nothing to differentiate: no autograd node at all
    return _RRDBNetFn.apply(launched, x, *params)


def eager_forward(module, x: torch.Tensor) -> torch.Tensor:
    """The generator graph on the module's own ``nn.Conv2d`` children with stock torch ops (autograd-capable), for
    tensors that do not live on a CUDA device.  Same wiring as ESRGAN/model.py:49-60,77-86,211-232 (BSRGAN/model.py:366-381,
    Real_ESRGAN/model.py:246-263): dense blocks with 0.2 residual scaling, long skip, nearest-x2 + conv stages, clamp."""
    import torch.nn.functional as F

    def act(t):
        return F.leaky_relu(t, 0.2)

    head = module.conv1(x)
    t = head + module.conv2(eager_trunk(module.trunk, head))
    for u in range(1, module._n_up + 1):
        t = act(getattr(module, f"upsampling{u}")[0](F.interpolate(t, scale_factor=2, mode="nearest")))
    t = module.conv4(act(module.conv3[0](t)))
    return torch.clamp(t, 0.0, 1.0)


def eager_trunk(trunk, t: torch.Tensor) -> torch.Tensor:
    """The RRDB stack on its own ``nn.Conv2d`` children with stock torch ops (ESRGAN/model.py:49-60,77-86): what
    :func:`eager_forward` runs between conv1 and conv2, and what :class:`~sr_gan_fd_b200.rrdbnet.RRDBTrunk` runs on the CPU."""
    import torch.nn.functional as F

    def act(v):
        return F.leaky_relu(v, 0.2)

    def dense_block(rdb, v):
        feats = [v]
        for conv in (rdb.conv1, rdb.conv2, rdb.conv3, rdb.conv4):
            feats.append(act(conv(torch.cat(feats, 1))))
        return rdb.conv5(torch.cat(feats, 1)) * 0.2 + v

    for rrdb in trunk:
        inner = t
        for rdb in (rrdb.rdb1, rrdb.rdb2, rrdb.rdb3):
            inner = dense_block(rdb, inner)
        t = inner * 0.2 + t
    return t


def attach_grad_bucket_hook(module, hook: Optional[Callable[[torch.Tensor, int, int], None]]) -> None:
    """Data-parallel training: ``hook(flat_grads, offset, count)`` is called from inside backward each time a
    contiguous bucket of the flat gradient buffer has been fully enqueued (see ``sr_gan_fd_b200.dist``)."""
    module._runtime().grad_bucket_hook = hook
