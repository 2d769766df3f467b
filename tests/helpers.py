"""Shared helpers for the GPU parity tests: everything calls the product through the C ABI (ctypes)."""
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "simple-vae-rs_b200")
for p in (ROOT, PKG):
    if p not in sys.path:
        sys.path.insert(0, p)

from svrs_native.lib import BF16, F32, lib  # noqa: E402


def st():
    return torch.cuda.current_stream().cuda_stream


def dt(t):
    return F32 if t == torch.float32 else BF16


def nhwc(t, dtype=torch.float32):
    return t.permute(0, 2, 3, 1).contiguous().to(dtype)


def nchw(t):
    return t.permute(0, 3, 1, 2).contiguous().float()


def pack(w, dtype, convT=False):
    """returns (pack_f, pack_b) for a conv / convT weight in torch layout (fp32, cuda)."""
    d0, d1 = w.shape[0], w.shape[1]
    kk = w.shape[2] * w.shape[3]
    p01 = torch.empty(w.numel(), device=w.device, dtype=dtype)
    p10 = torch.empty(w.numel(), device=w.device, dtype=dtype)
    lib.pack_weights(w.data_ptr(), d0, d1, kk, p01.data_ptr(), p10.data_ptr(), dt(dtype), st())
    return (p01, p10) if convT else (p10, p01)


class Guarded:
    """A device tensor `t` of `shape` inside a buffer with `pad` sentinel elements before and after it: intact() is False
    once a kernel has written outside `t`."""

    SENTINEL = 12345.0

    def __init__(self, shape, dtype, fill=float("nan"), pad=4096):
        n = 1
        for d in shape:
            n *= int(d)
        self.pad, self.n = pad, n
        self.buf = torch.full((n + 2 * pad,), self.SENTINEL, device="cuda", dtype=dtype)
        self.t = self.buf[pad:pad + n].view(shape)
        self.t.fill_(fill)

    def intact(self):
        return bool((self.buf[:self.pad] == self.SENTINEL).all() and (self.buf[self.pad + self.n:] == self.SENTINEL).all())


def task_stats(draws, target):
    """models/base.py:305-313, 341 of the reference, verbatim arithmetic on a [S,4,P,P] sample stack and a [1,4,P,P] target."""
    diff = draws - target
    return dict(mean=draws.mean(dim=0), std=draws.std(dim=0).mean(dim=0), mae=diff.abs().mean(dim=(0, 1)),
                mse=diff.pow(2).mean(dim=(0, 1)), mean_bias=(target - draws.mean(dim=0)).mean(dim=0).mean(dim=0),
                sample0=draws[0])


def report(name, got, ref, rtol, atol=0.0):
    got = got.detach().double().cpu()
    ref = ref.detach().double().cpu()
    assert got.shape == ref.shape, f"{name}: shape {tuple(got.shape)} vs {tuple(ref.shape)}"
    err = (got - ref).abs()
    scale = ref.abs().max().item() + 1e-30
    mx = err.max().item() if err.numel() else 0.0
    rel = mx / scale
    print(f"[parity] {name}: max|err|={mx:.3e} rel-to-max={rel:.3e} (ref max {scale:.3e})")
    assert torch.isfinite(got).all(), f"{name}: non-finite values"
    assert mx <= atol + rtol * scale, f"{name}: max|err| {mx:.3e} > {atol} + {rtol}*{scale:.3e}"
    return rel
