"""ctypes binding of libb200sr.so (the C ABI declared in include/b200sr.h).  Fails loudly when the library is
missing -- there is no Python/PyTorch fallback for the generator math."""
from __future__ import annotations

import ctypes as C
import os
import threading

from .build import LIB_PATH

F32, F16, BF16 = 0, 1, 2

BUCKET_CB = C.CFUNCTYPE(None, C.c_void_p, C.c_int64, C.c_int64)


class NetDesc(C.Structure):
    _fields_ = [(n, C.c_int32) for n in (
        "in_channels", "out_channels", "channels", "growth", "num_blocks", "n_up",
        "batch", "height", "width", "training", "grad_bucket_rrdbs", "deterministic")]


class VggDesc(C.Structure):
    _fields_ = [(n, C.c_int32) for n in ("batch", "height", "width", "last_conv", "feat_mask", "grad_conv", "grad_images")] + \
               [("mean", C.c_float * 3), ("std", C.c_float * 3), ("deterministic", C.c_int32)]


class DiscDesc(C.Structure):
    _fields_ = [(n, C.c_int32) for n in ("in_channels", "out_channels", "channels", "batch", "height", "width", "training", "fp16",
                                         "deterministic")]


_lock = threading.Lock()
_lib = None

# symbol -> (restype, argtypes); every entry point declared in include/b200sr.h
SIGNATURES = {
    "b200sr_plan_create": (C.c_int, [C.POINTER(NetDesc), C.POINTER(C.c_void_p)]),
    "b200sr_trunk_plan_create": (C.c_int, [C.POINTER(NetDesc), C.POINTER(C.c_void_p)]),
    "b200sr_unclamped_plan_create": (C.c_int, [C.POINTER(NetDesc), C.POINTER(C.c_void_p)]),
    "b200sr_plan_destroy": (None, [C.c_void_p]),
    "b200sr_workspace_bytes": (C.c_size_t, [C.c_void_p]),
    "b200sr_packed_bytes": (C.c_size_t, [C.c_void_p]),
    "b200sr_pack_layout_id": (C.c_uint64, [C.c_void_p]),
    "b200sr_num_params": (C.c_int32, [C.c_void_p]),
    "b200sr_param_numel": (C.c_int64, [C.c_void_p]),
    "b200sr_flops": (C.c_double, [C.c_void_p, C.c_int]),
    "b200sr_num_launches": (C.c_int32, [C.c_void_p, C.c_int]),
    "b200sr_pack_weights": (C.c_int, [C.c_void_p, C.POINTER(C.c_void_p), C.c_void_p, C.c_void_p]),
    "b200sr_forward": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.POINTER(C.c_int64), C.c_void_p, C.c_void_p,
                                 C.c_void_p, C.c_void_p]),
    "b200sr_backward": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, BUCKET_CB,
                                  C.c_void_p, C.c_void_p]),
    "b200sr_backward_select": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                         C.POINTER(C.c_uint8), BUCKET_CB, C.c_void_p, C.c_void_p]),
    "b200sr_backward_launches": (C.c_int32, [C.c_void_p, C.POINTER(C.c_uint8), C.c_int, C.c_int]),
    "b200sr_conv3x3_scratch_bytes": (C.c_size_t, [C.c_int, C.c_int]),
    "b200sr_conv3x3_fwd": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p,
                                     C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p]),
    "b200sr_conv3x3_dgrad": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_int,
                                       C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p]),
    "b200sr_conv3x3_wgrad_scratch_bytes": (C.c_size_t, [C.c_int, C.c_int]),
    "b200sr_conv3x3_wgrad": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_int,
                                       C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]),
    "b200sr_fused_adam_ema": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int64, C.c_float, C.c_float, C.c_float, C.c_float,
                                        C.c_float, C.c_void_p, C.c_float, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]),
    "b200sr_iqa_psnr_ssim_y": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_double), C.c_void_p,
                                         C.c_void_p, C.c_void_p]),
    "b200sr_iqa_det_scratch_bytes": (C.c_size_t, [C.c_int, C.c_int, C.c_int]),
    "b200sr_iqa_psnr_ssim_y_det": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_double),
                                             C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "b200sr_tensor_to_image_u8": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p]),
    "b200sr_vgg_plan_create": (C.c_int, [C.POINTER(VggDesc), C.POINTER(C.c_void_p)]),
    "b200sr_vgg_forward": (C.c_int, [C.c_void_p, C.c_void_p, C.POINTER(C.c_int64), C.c_void_p, C.c_void_p, C.c_void_p]),
    "b200sr_vgg_feature_l1": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p]),
    "b200sr_vgg_backward": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "b200sr_disc_plan_create": (C.c_int, [C.POINTER(DiscDesc), C.POINTER(C.c_void_p)]),
    "b200sr_disc_forward": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.POINTER(C.c_int64), C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "b200sr_disc_backward": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "b200sr_last_error": (C.c_char_p, []),
    "b200sr_version": (C.c_int, []),
    "b200sr_debug_set": (None, [C.c_int]),
    "b200sr_debug_read_profile": (C.c_int, [C.c_void_p, C.c_int]),
    "b200sr_debug_buffer": (C.c_int, [C.c_void_p, C.c_char_p, C.POINTER(C.c_int64), C.POINTER(C.c_int64)]),
}


def load() -> C.CDLL:
    """dlopen the in-tree library (built by ``sr_gan_fd_b200.build.build_native`` / ``__graft_entry__.build``)."""
    global _lib
    with _lock:
        if _lib is not None:
            return _lib
        path = os.environ.get("B200SR_LIB", LIB_PATH)  # developer A/B switch: another build of the same library
        if not os.path.exists(path):
            raise RuntimeError(
                f"{path} is missing: build it with `python -m sr_gan_fd_b200.build` (needs nvcc). "
                "The B200 generator path has no PyTorch fallback.")
        lib = C.CDLL(path)
        for name, (res, args) in SIGNATURES.items():
            if "B200SR_LIB" in os.environ and not hasattr(lib, name):
                continue  # an older build loaded for a same-box A/B run may predate newer entry points; the in-tree library must have all
            fn = getattr(lib, name)
            fn.restype = res
            fn.argtypes = args
        _lib = lib
        return lib


def deterministic() -> bool:
    """Whether the native calls run in deterministic mode: ``torch.use_deterministic_algorithms(True)`` (with or without
    ``warn_only``) is in effect.  Read on every call; the plans of the two modes are cached side by side."""
    import torch
    return torch.are_deterministic_algorithms_enabled()


def check(rc: int) -> None:
    if rc != 0:
        msg = load().b200sr_last_error()
        raise RuntimeError(f"libb200sr error {rc}: {msg.decode() if msg else '?'}")
