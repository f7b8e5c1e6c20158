"""Evaluation epilogue next to the generator path (SURVEY.md section 8f, rank 4): drop-ins for the reference's ``PSNR`` / ``SSIM``
modules (``ESRGAN/image_quality_assessment.py:397-414, 507-541``; same constructors, same call, same return dtype) and for
``imgproc.tensor_to_image`` (``ESRGAN/imgproc.py:160-183``).

CUDA fp32 RGB tensors with ``only_test_y_channel=True`` and the default 11x11 window -- what every ``validate()`` /
``test_*.py`` of the reference uses (``ESRGAN/train_rrdbnet.py:93-94``) -- run as ONE fused pass per metric in libb200sr.so
(``b200sr_iqa_psnr_ssim_y``: crop + RGB->Y + fp64 error / gaussian statistics + reduction) instead of ~25 torch launches
with fp64 full-frame temporaries.  Everything else (CPU tensors, all-channel mode, other window sizes, half tensors) takes a
plain torch restatement of the same formulas below.
"""
from __future__ import annotations

import ctypes as C
from typing import Any

import numpy as np
import torch
from torch import nn
from torch.nn import functional as F

from . import lib as _lib

__all__ = ["PSNR", "SSIM", "tensor_to_image", "gaussian_window_1d"]


def gaussian_window_1d(window_size: int = 11, sigma: float = 1.5) -> np.ndarray:
    """What ``cv2.getGaussianKernel(window_size, sigma)`` returns for sigma > 0 (fp64, normalised)."""
    ax = np.arange(window_size, dtype=np.float64) - (window_size - 1) / 2.0
    k = np.exp(-(ax ** 2) / (2.0 * sigma * sigma))
    return k / k.sum()


def _rgb_to_y(t: torch.Tensor) -> torch.Tensor:
    w = torch.tensor([[65.481], [128.553], [24.966]], dtype=t.dtype, device=t.device)
    return (torch.matmul(t.permute(0, 2, 3, 1), w).permute(0, 3, 1, 2) + 16.0) / 255.0


def _rgb_to_ycbcr(t: torch.Tensor) -> torch.Tensor:
    w = torch.tensor([[65.481, -37.797, 112.0], [128.553, -74.203, -93.786], [24.966, 112.0, -18.214]], dtype=t.dtype, device=t.device)
    b = torch.tensor([16.0, 128.0, 128.0], dtype=t.dtype, device=t.device).view(1, 3, 1, 1)
    return (torch.matmul(t.permute(0, 2, 3, 1), w).permute(0, 3, 1, 2) + b) / 255.0


def _prepare(raw: torch.Tensor, dst: torch.Tensor, crop_border: int, only_y: bool):
    assert raw.shape == dst.shape, f"Supplied images have different sizes {tuple(raw.shape)} and {tuple(dst.shape)}"
    if crop_border > 0:
        raw = raw[:, :, crop_border:-crop_border, crop_border:-crop_border]
        dst = dst[:, :, crop_border:-crop_border, crop_border:-crop_border]
    if only_y:
        raw, dst = _rgb_to_y(raw), _rgb_to_y(dst)
    return raw.to(torch.float64), dst.to(torch.float64)


def _native_ok(raw: torch.Tensor, dst: torch.Tensor, only_y: bool, window_size: int, crop_border: int) -> bool:
    return (only_y and window_size == 11 and raw.is_cuda and dst.is_cuda and raw.dtype == torch.float32 and dst.dtype == torch.float32
            and raw.dim() == 4 and raw.shape[1] == 3 and raw.shape == dst.shape
            and raw.shape[2] - 2 * crop_border >= 11 and raw.shape[3] - 2 * crop_border >= 11)


def _native_sums(raw, dst, crop_border, win, want_psnr, want_ssim):
    raw, dst = raw.contiguous(), dst.contiguous()
    n, _, h, w = raw.shape
    out = torch.empty((2, n), dtype=torch.float64, device=raw.device)
    arr = (C.c_double * 11)(*[float(v) for v in win])
    lib = _lib.load()
    with torch.cuda.device(raw.device):
        stream = torch.cuda.current_stream().cuda_stream
        args = (C.c_void_p(raw.data_ptr()), C.c_void_p(dst.data_ptr()), n, h, w, crop_border, arr,
                C.c_void_p(out[0].data_ptr()) if want_psnr else None, C.c_void_p(out[1].data_ptr()) if want_ssim else None)
        if _lib.deterministic():  # per-block partials summed in block order instead of atomics
            scratch = torch.empty(int(lib.b200sr_iqa_det_scratch_bytes(n, h, w)), dtype=torch.uint8, device=raw.device)
            _lib.check(lib.b200sr_iqa_psnr_ssim_y_det(*args, C.c_void_p(scratch.data_ptr()), C.c_void_p(stream)))
        else:
            _lib.check(lib.b200sr_iqa_psnr_ssim_y(*args, C.c_void_p(stream)))
    return out


class PSNR(nn.Module):
    """``PSNR(crop_border, only_test_y_channel)(raw, dst) -> [N] float64`` (image_quality_assessment.py:361-414)."""

    def __init__(self, crop_border: int, only_test_y_channel: bool) -> None:
        super().__init__()
        self.crop_border = crop_border
        self.only_test_y_channel = only_test_y_channel
        self._win = gaussian_window_1d()

    def forward(self, raw_tensor: torch.Tensor, dst_tensor: torch.Tensor) -> torch.Tensor:
        if _native_ok(raw_tensor, dst_tensor, self.only_test_y_channel, 11, self.crop_border):
            n, _, h, w = raw_tensor.shape
            count = (h - 2 * self.crop_border) * (w - 2 * self.crop_border)
            sums = _native_sums(raw_tensor, dst_tensor, self.crop_border, self._win, True, False)[0]
            return 10 * torch.log10(255.0 ** 2 / (sums / count + 1e-8))
        raw, dst = _prepare(raw_tensor, dst_tensor, self.crop_border, self.only_test_y_channel)
        mse = torch.mean((raw * 255.0 - dst * 255.0) ** 2 + 1e-8, dim=[1, 2, 3])
        return 10 * torch.log10(255.0 ** 2 / mse)


class SSIM(nn.Module):
    """``SSIM(crop_border, only_only_test_y_channel, window_size=11, gaussian_sigma=1.5)(raw, dst) -> [N] float32``
    (image_quality_assessment.py:416-541)."""

    def __init__(self, crop_border: int, only_only_test_y_channel: bool, window_size: int = 11, gaussian_sigma: float = 1.5) -> None:
        super().__init__()
        self.crop_border = crop_border
        self.only_test_y_channel = only_only_test_y_channel
        self.window_size = window_size
        self._win = gaussian_window_1d(window_size, gaussian_sigma)
        self.gaussian_kernel_window = np.outer(self._win, self._win)

    def forward(self, raw_tensor: torch.Tensor, dst_tensor: torch.Tensor) -> torch.Tensor:
        if _native_ok(raw_tensor, dst_tensor, self.only_test_y_channel, self.window_size, self.crop_border):
            n, _, h, w = raw_tensor.shape
            count = (h - 2 * self.crop_border - 10) * (w - 2 * self.crop_border - 10)
            sums = _native_sums(raw_tensor, dst_tensor, self.crop_border, self._win, False, True)[1]
            return (sums / count).float()
        raw, dst = _prepare(raw_tensor, dst_tensor, self.crop_border, self.only_test_y_channel)
        raw, dst = raw * 255.0, dst * 255.0
        c1, c2 = (0.01 * 255.0) ** 2, (0.03 * 255.0) ** 2
        ch = raw.size(1)
        win = torch.from_numpy(self.gaussian_kernel_window).view(1, 1, self.window_size, self.window_size)
        win = win.expand(ch, 1, self.window_size, self.window_size).to(device=raw.device, dtype=raw.dtype)
        mu_r, mu_d = F.conv2d(raw, win, groups=ch), F.conv2d(dst, win, groups=ch)
        var_r = F.conv2d(raw * raw, win, groups=ch) - mu_r ** 2
        var_d = F.conv2d(dst * dst, win, groups=ch) - mu_d ** 2
        cov = F.conv2d(raw * dst, win, groups=ch) - mu_r * mu_d
        s = ((2 * mu_r * mu_d + c1) * (2 * cov + c2)) / ((mu_r ** 2 + mu_d ** 2 + c1) * (var_r + var_d + c2))
        return torch.mean(s, [1, 2, 3]).float()


def tensor_to_image(tensor: torch.Tensor, range_norm: bool, half: bool) -> Any:
    """``imgproc.tensor_to_image``: [1, C, H, W] in [0, 1] -> uint8 ndarray [H, W, C].  CUDA fp32 input: one kernel writes the
    uint8 HWC image (a quarter of the bytes cross PCIe); otherwise the reference's op sequence."""
    if tensor.is_cuda and tensor.dtype == torch.float32 and tensor.dim() == 4 and tensor.shape[0] == 1 and tensor.shape[1] <= 4:
        t = tensor.contiguous()
        _, c, h, w = t.shape
        out = torch.empty((h, w, c), dtype=torch.uint8, device=t.device)
        with torch.cuda.device(t.device):
            _lib.check(_lib.load().b200sr_tensor_to_image_u8(C.c_void_p(t.data_ptr()), c, h, w, 1 if range_norm else 0, 1 if half else 0,
                                                             C.c_void_p(out.data_ptr()), C.c_void_p(torch.cuda.current_stream().cuda_stream)))
        return out.cpu().numpy()
    if range_norm:
        tensor = tensor.add(1.0).div(2.0)
    if half:
        tensor = tensor.half()
    return tensor.squeeze(0).permute(1, 2, 0).mul(255).clamp(0, 255).cpu().numpy().astype("uint8")
