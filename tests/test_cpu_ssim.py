"""CPU tests (-m "not gpu") of the SSIM metric: the fp64 oracle (tests/ssim_oracle.py) against independent restatements
and known answers, and the argument checks of svrs_native.metrics.ssim, which happen before any device work."""
import numpy as np
import pytest
import torch

import ssim_oracle
from svrs_native import metrics
from svrs_native.lib import SvrsError


def _direct(a, b, win, R=1.0):
    """scikit-image's formulas with an explicit win x win window at every interior position."""
    N, C, H, W = a.shape
    npix = win * win
    c1, c2 = (0.01 * R) ** 2, (0.03 * R) ** 2
    out = np.zeros(N)
    for n in range(N):
        for c in range(C):
            tot = 0.0
            for y in range(H - win + 1):
                for x in range(W - win + 1):
                    wa, wb = a[n, c, y:y + win, x:x + win], b[n, c, y:y + win, x:x + win]
                    ux, uy = wa.mean(), wb.mean()
                    vx = ((wa - ux) ** 2).sum() / (npix - 1)
                    vy = ((wb - uy) ** 2).sum() / (npix - 1)
                    vxy = ((wa - ux) * (wb - uy)).sum() / (npix - 1)
                    tot += (2 * ux * uy + c1) * (2 * vxy + c2) / ((ux * ux + uy * uy + c1) * (vx + vy + c2))
            out[n] += tot / ((H - win + 1) * (W - win + 1)) / C
    return out


def _pair(shape, seed):
    rng = np.random.default_rng(seed)
    a = rng.random(shape)
    return a, np.clip(a + 0.2 * rng.standard_normal(shape), 0, 1)


@pytest.mark.parametrize("shape,win,R", [((1, 1, 24, 31), 11, 1.0), ((2, 4, 32, 32), 11, 1.0), ((2, 4, 32, 32), 7, 2.0)])
def test_oracle_equals_direct_windows(shape, win, R):
    a, b = _pair(shape, 1)
    np.testing.assert_allclose(ssim_oracle.ssim(a, b, win, R), _direct(a, b, win, R), rtol=0, atol=1e-12)


def test_oracle_equals_uniform_filter_restatement():
    """scikit-image's own path: scipy.ndimage.uniform_filter window means, cropped by (win-1)/2."""
    ndi = pytest.importorskip("scipy.ndimage")
    a, b = _pair((2, 4, 32, 40), 2)
    win, npix = 11, 121
    pad = (win - 1) // 2
    ref = np.zeros(2)
    for n in range(2):
        for c in range(4):
            f = lambda t: ndi.uniform_filter(t, size=win)
            x, y = a[n, c], b[n, c]
            ux, uy = f(x), f(y)
            cn = npix / (npix - 1)
            vx, vy, vxy = cn * (f(x * x) - ux * ux), cn * (f(y * y) - uy * uy), cn * (f(x * y) - ux * uy)
            c1, c2 = 0.01 ** 2, 0.03 ** 2
            s = (2 * ux * uy + c1) * (2 * vxy + c2) / ((ux * ux + uy * uy + c1) * (vx + vy + c2))
            ref[n] += s[pad:-pad, pad:-pad].mean() / 4
    np.testing.assert_allclose(ssim_oracle.ssim(a, b), ref, rtol=0, atol=1e-12)


def test_oracle_known_answers():
    a, _ = _pair((3, 4, 20, 20), 3)
    np.testing.assert_allclose(ssim_oracle.ssim(a, a), 1.0, rtol=0, atol=1e-12)
    c1v, c2v = 0.3, 0.7
    ca, cb = np.full((1, 2, 16, 16), c1v), np.full((1, 2, 16, 16), c2v)
    C1 = 0.01 ** 2
    np.testing.assert_allclose(ssim_oracle.ssim(ca, cb), (2 * c1v * c2v + C1) / (c1v ** 2 + c2v ** 2 + C1), rtol=0, atol=1e-12)
    # data_range enters only through C1 and C2: scaling images and range together leaves SSIM unchanged
    a, b = _pair((2, 3, 18, 21), 4)
    np.testing.assert_allclose(ssim_oracle.ssim(3 * a, 3 * b, 11, 3.0), ssim_oracle.ssim(a, b, 11, 1.0), rtol=0, atol=1e-12)
    assert abs(ssim_oracle.ssim(a, b, 11, 2.0) - ssim_oracle.ssim(a, b, 11, 1.0)).max() > 1e-3


def test_metrics_ssim_argument_checks_before_device():
    a = torch.rand(2, 4, 16, 16)
    with pytest.raises(ValueError, match="same shape"):
        metrics.ssim(a, torch.rand(2, 4, 16, 15))
    with pytest.raises(ValueError, match="same shape"):
        metrics.ssim(a[0], a[0])
    with pytest.raises(ValueError, match="odd"):
        metrics.ssim(a, a, win_size=10)
    with pytest.raises(ValueError, match="exceeds image extent"):
        metrics.ssim(a, a, win_size=17)
    with pytest.raises(SvrsError, match="CUDA"):
        metrics.ssim(a, a)


def test_workspace_query_is_host_callable():
    """One fp64 partial per band of 16 output rows of every plane; -1 for what svrs_ssim rejects (no device needed)."""
    from svrs_native.lib import lib
    assert lib.ssim_workspace_doubles(128, 4, 64, 64, 11) == 128 * 4 * 4        # 54 interior rows -> 4 bands
    assert lib.ssim_workspace_doubles(5, 1, 11, 11, 11) == 5
    assert lib.ssim_workspace_doubles(16, 4, 256, 256, 11) == 16 * 4 * 16
    assert lib.ssim_workspace_doubles(0, 4, 64, 64, 11) == 0
    assert lib.ssim_workspace_doubles(1, 4, 512, 409, 11) > 0                  # widest plane at win 11
    for bad in [(1, 4, 64, 64, 1), (1, 4, 64, 64, 10), (1, 4, 64, 10, 11), (1, 0, 64, 64, 11), (-1, 4, 64, 64, 11),
                (1, 4, 64, 410, 11)]:
        assert lib.ssim_workspace_doubles(*bad) == -1, bad
    assert "shared memory" in lib.last_error()
