"""Image-quality metrics of evaluate() on the device (svrs_ssim, csrc/ssim.cu)."""
from __future__ import annotations

import torch

from .lib import SvrsError, lib


def ssim(a: torch.Tensor, b: torch.Tensor, win_size: int = 11, data_range: float = 1.0) -> torch.Tensor:
    """Per-image SSIM of two [N, C, H, W] batches -> float64 [N] on their device.  out[n] equals
    skimage.metrics.structural_similarity(a[n], b[n], win_size=win_size, data_range=data_range, channel_axis=0) with its
    defaults (uniform window, sample covariance, K1 = 0.01, K2 = 0.03).  The work is enqueued on the current stream; CUDA
    tensors only (there is no CPU path)."""
    if a.dim() != 4 or a.shape != b.shape:
        raise ValueError(f"ssim: expected two [N, C, H, W] tensors of the same shape, got {tuple(a.shape)} and {tuple(b.shape)}")
    if win_size % 2 == 0:
        raise ValueError("Window size must be odd.")
    if win_size > min(a.shape[2], a.shape[3]):
        raise ValueError(f"win_size exceeds image extent: {win_size} > min({a.shape[2]}, {a.shape[3]})")
    if not (a.is_cuda and b.is_cuda):
        raise SvrsError("ssim: tensors must live on a CUDA device (no CPU fallback in svrs_b200)")
    N, C, H, W = a.shape
    a = a.detach().to(torch.float32).contiguous()
    b = b.detach().to(device=a.device, dtype=torch.float32).contiguous()
    nws = lib.ssim_workspace_doubles(N, C, H, W, win_size)
    if nws < 0:
        raise SvrsError(f"svrs_ssim_workspace_doubles: {lib.last_error()}")
    ws = torch.empty(nws, device=a.device, dtype=torch.float64)
    out = torch.empty(N, device=a.device, dtype=torch.float64)
    lib.ssim(a.data_ptr(), b.data_ptr(), N, C, H, W, win_size, float(data_range), ws.data_ptr(), out.data_ptr(),
             torch.cuda.current_stream(a.device).cuda_stream)
    return out
