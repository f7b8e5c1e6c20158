"""Fused optimizer step for the drop-in generators (SURVEY.md section 8f, rank 1 -- the step right after the hot path).

``FusedAdamEMA`` is a ``torch.optim.Optimizer`` with the semantics of the reference's
``optim.Adam(model.parameters(), lr, betas, eps, weight_decay)`` (``ESRGAN/train_rrdbnet.py:195-202``) that also carries
the EMA copy the scripts maintain with ``AveragedModel(model, avg_fn=...)`` + ``update_parameters`` (``:182-183,267``):

    ema <- (1 - d) * ema + d * p          # the reference's avg_fn; the first update copies p

and cooperates with ``torch.cuda.amp.GradScaler`` (``_step_supports_amp_scaling``): unscale, non-finite skip, Adam and
EMA are ONE kernel launch over all 702 tensors (libb200sr ``b200sr_fused_adam_ema``) instead of the foreach Adam
kernels plus a 702-iteration Python EMA loop (~3k launches).  CUDA fp32 parameters only; no CPU fallback.

Frozen parameters: a parameter whose ``.grad`` is None gets no Adam update (parameter and moments untouched, as
``torch.optim.Adam`` skips it) and is still averaged into the EMA copy (``AveragedModel.update_parameters`` averages every
parameter).  One limit: the Adam step counter is shared by all parameters, so a parameter that is unfrozen later takes its
bias correction from the shared count, not from the steps it took itself.  A fixed freeze pattern matches torch exactly.
"""
from __future__ import annotations

import ctypes as C
from typing import Iterable, Optional

import numpy as np
import torch

from . import lib as _lib


class FusedAdamEMA(torch.optim.Optimizer):
    _step_supports_amp_scaling = True  # GradScaler hands us grad_scale / found_inf instead of unscaling itself

    def __init__(self, params: Iterable[torch.nn.Parameter], lr: float = 2e-4, betas=(0.9, 0.99), eps: float = 1e-8,
                 weight_decay: float = 0.0, ema_model: Optional[torch.nn.Module] = None, ema_decay: float = 0.99998) -> None:
        super().__init__(params, dict(lr=lr, betas=betas, eps=eps, weight_decay=weight_decay))
        if len(self.param_groups) != 1:
            raise ValueError("FusedAdamEMA supports a single parameter group")
        self.ema_decay = float(ema_decay)
        self._params = [p for p in self.param_groups[0]["params"]]
        for p in self._params:
            if not p.is_cuda or p.dtype != torch.float32 or not p.is_contiguous():
                raise RuntimeError("FusedAdamEMA needs contiguous fp32 CUDA parameters (no CPU fallback)")
        self._ema_params = None
        self._ema_owner = None
        if ema_model is not None:
            mod = ema_model.module if hasattr(ema_model, "module") else ema_model  # AveragedModel wraps .module
            self._ema_params = [p for p in mod.parameters()]
            if len(self._ema_params) != len(self._params):
                raise ValueError("ema_model must have the same parameter list as the optimised model")
            self._ema_owner = ema_model
        dev = self._params[0].device
        # ONE device-side step counter shared by every parameter's state entry (skipped steps do not advance it); it is
        # saved / restored through optimizer.state_dict() like torch.optim.Adam's per-parameter "step"
        step = torch.zeros(1, dtype=torch.float32, device=dev)
        for p in self._params:
            st = self.state[p]
            st["step"] = step
            st["exp_avg"] = torch.zeros_like(p)
            st["exp_avg_sq"] = torch.zeros_like(p)
        # EMA updates made so far (the first one copies): persisted in the param group so that it survives state_dict round trips
        self.param_groups[0].setdefault("ema_updates", self._ema_updates_from_owner())
        blocks = 0
        self._block0 = []
        for p in self._params:
            self._block0.append(blocks)
            blocks += (p.numel() + 1023) // 1024
        self._total_blocks = blocks
        self._block_tensor = torch.from_numpy(np.repeat(np.arange(len(self._params), dtype=np.int32),
                                                        [(p.numel() + 1023) // 1024 for p in self._params])).to(dev)
        # pointer table: two pinned host copies used alternately (the H2D copy of step k may still be in flight while the
        # host fills the table of step k + 1), each guarded by an event recorded after its copy
        self._tables_host = [torch.empty((len(self._params), 7), dtype=torch.int64).pin_memory() for _ in range(2)]
        self._table_events = [None, None]
        self._table_slot = 0
        self._table_dev = torch.empty((len(self._params), 7), dtype=torch.int64, device=dev)
        self._rebuild_table()

    def _ema_updates_from_owner(self) -> int:
        owner = self._ema_owner
        if owner is not None and hasattr(owner, "n_averaged"):
            return int(owner.n_averaged)  # AveragedModel keeps it as a buffer: a resumed EMA keeps averaging
        return 0

    def _rebuild_table(self) -> None:
        """(Re)reads every state pointer.  Called at construction and whenever ``self.state`` was replaced
        (``load_state_dict`` -- the reference's resume path, ESRGAN/utils.py:53 -- swaps in new tensors)."""
        p0 = self._params[0]
        step = self.state[p0]["step"]
        if not torch.is_tensor(step):
            step = torch.tensor([float(step)], dtype=torch.float32)
        step = step.detach().reshape(1).to(device=p0.device, dtype=torch.float32).clone()
        self._step_dev = step
        for tbl_t in self._tables_host:
            tbl = tbl_t.numpy()
            for i, p in enumerate(self._params):
                st = self.state[p]
                st["step"] = step
                for k in ("exp_avg", "exp_avg_sq"):
                    t = st[k]
                    if not t.is_cuda or t.dtype != torch.float32 or not t.is_contiguous() or t.shape != p.shape:
                        st[k] = t.to(device=p.device, dtype=torch.float32).contiguous().view_as(p).clone()
                tbl[i, 0] = p.data_ptr()
                tbl[i, 1] = 0
                tbl[i, 2] = st["exp_avg"].data_ptr()
                tbl[i, 3] = st["exp_avg_sq"].data_ptr()
                tbl[i, 4] = self._ema_params[i].data_ptr() if self._ema_params is not None else 0
                tbl[i, 5] = p.numel()
                tbl[i, 6] = self._block0[i]
        self._state_probe = (self.state[p0]["exp_avg"].data_ptr(), self.state[self._params[-1]]["exp_avg_sq"].data_ptr(),
                             p0.data_ptr(), self._ema_params[0].data_ptr() if self._ema_params is not None else 0)

    def load_state_dict(self, state_dict) -> None:
        super().load_state_dict(state_dict)
        self._params = [p for p in self.param_groups[0]["params"]]
        self.param_groups[0].setdefault("ema_updates", self._ema_updates_from_owner())
        self._rebuild_table()

    @torch.no_grad()
    def step(self, closure=None):
        if closure is not None:
            raise RuntimeError("closures are not supported")
        grp = self.param_groups[0]
        p0 = self._params[0]
        probe = (self.state[p0]["exp_avg"].data_ptr(), self.state[self._params[-1]]["exp_avg_sq"].data_ptr(), p0.data_ptr(),
                 self._ema_params[0].data_ptr() if self._ema_params is not None else 0)
        if probe != self._state_probe:  # state / parameters were re-assigned behind our back
            self._rebuild_table()
        slot = self._table_slot
        self._table_slot = 1 - slot
        ev = self._table_events[slot]
        if ev is not None:
            ev.synchronize()  # the copy that last read this pinned table (two steps ago) has finished
        tbl = self._tables_host[slot].numpy()
        for i, p in enumerate(self._params):
            g = p.grad
            if g is None:  # frozen: no Adam update (null gradient pointer), the EMA still averages it
                tbl[i, 1] = 0
                continue
            if g.dtype != torch.float32 or not g.is_contiguous():
                g = g.float().contiguous()
                p.grad = g
            tbl[i, 1] = g.data_ptr()
        dev = p0.device
        grad_scale = getattr(self, "grad_scale", None)
        found_inf = getattr(self, "found_inf", None)
        with torch.cuda.device(dev):
            cur = torch.cuda.current_stream()
            stream = cur.cuda_stream
            self._table_dev.copy_(self._tables_host[slot], non_blocking=True)
            if ev is None:
                ev = self._table_events[slot] = torch.cuda.Event()
            ev.record(cur)
            ema_copy = 1 if (self._ema_params is not None and int(grp.get("ema_updates", 0)) == 0) else 0
            _lib.check(_lib.load().b200sr_fused_adam_ema(
                C.c_void_p(self._table_dev.data_ptr()), C.c_void_p(self._block_tensor.data_ptr()), len(self._params), self._total_blocks,
                float(grp["lr"]), float(grp["betas"][0]), float(grp["betas"][1]), float(grp["eps"]), float(grp["weight_decay"]),
                C.c_void_p(self._step_dev.data_ptr()), self.ema_decay, ema_copy,
                C.c_void_p(grad_scale.data_ptr()) if grad_scale is not None else None,
                C.c_void_p(found_inf.data_ptr()) if found_inf is not None else None, C.c_void_p(stream)))
        touched = list(self._params)
        if self._ema_params is not None:
            grp["ema_updates"] = int(grp.get("ema_updates", 0)) + 1
            owner = self._ema_owner
            if owner is not None and hasattr(owner, "n_averaged"):
                owner.n_averaged += 1
            touched += self._ema_params
        # the kernel wrote the parameters (and the EMA copy) behind autograd's back: bump their version counters, which the
        # generator runtime uses to decide when the packed bf16 weights must be rebuilt
        torch._C._autograd._unsafe_set_version_counter(touched, [p._version + 1 for p in touched])
        return None
