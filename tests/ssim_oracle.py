"""fp64 numpy oracle of the SSIM metric that evaluate() logs (scikit-image's structural_similarity with its defaults).

Test infrastructure: plain numpy, so it runs wherever the tests do.  tests/test_cpu_ssim.py pins it to explicit-window loops
and to scipy's uniform_filter; tests/test_ssim_gpu.py and tools/ssim_bench.py compare the device kernel with it."""
import numpy as np


def ssim(a, b, win_size=11, data_range=1.0):
    """skimage.metrics.structural_similarity(a[n], b[n], win_size, data_range=data_range, channel_axis=0) with its defaults
    (uniform window, use_sample_covariance=True, K1=0.01, K2=0.03) for [N][C][H][W] arrays -> float64 [N]: per plane the mean of
    S = (2 ux uy + C1)(2 vxy + C2) / ((ux^2 + uy^2 + C1)(vx + vy + C2)) over the interior positions (windows fully inside the
    plane; skimage crops (win-1)/2 from every edge), then the mean over the C planes.  Window means from summed-area tables
    (numpy only, so the oracle runs wherever the tests do)."""
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    assert a.shape == b.shape and a.ndim == 4 and win_size % 2 == 1 and win_size <= min(a.shape[2:])
    w = win_size
    npix = w * w

    def wmean(t):
        s = np.zeros(t.shape[:2] + (t.shape[2] + 1, t.shape[3] + 1))
        s[:, :, 1:, 1:] = t.cumsum(axis=2).cumsum(axis=3)
        return (s[:, :, w:, w:] - s[:, :, :-w, w:] - s[:, :, w:, :-w] + s[:, :, :-w, :-w]) / npix

    # (co)variances are shift-invariant: take them of the planes minus their means, so the table sums stay small
    ma, mb = a.mean(axis=(2, 3), keepdims=True), b.mean(axis=(2, 3), keepdims=True)
    a0, b0 = a - ma, b - mb
    ux0, uy0 = wmean(a0), wmean(b0)
    cov_norm = npix / (npix - 1.0)
    vx = cov_norm * (wmean(a0 * a0) - ux0 * ux0)
    vy = cov_norm * (wmean(b0 * b0) - uy0 * uy0)
    vxy = cov_norm * (wmean(a0 * b0) - ux0 * uy0)
    ux, uy = ux0 + ma, uy0 + mb
    c1, c2 = (0.01 * data_range) ** 2, (0.03 * data_range) ** 2
    s = (2 * ux * uy + c1) * (2 * vxy + c2) / ((ux * ux + uy * uy + c1) * (vx + vy + c2))
    return s.mean(axis=(2, 3)).mean(axis=1)
