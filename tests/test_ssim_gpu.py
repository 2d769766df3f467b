"""SSIM on the device (-m gpu): svrs_ssim / svrs_native.metrics.ssim against the fp64 oracle (tests/ssim_oracle.py, which
tests/test_cpu_ssim.py pins to scikit-image's formulas), its determinism and graph capture, its argument errors, and the
Metrics/SSIM* values evaluate() logs.

Tolerance: 6e-7 absolute per image, about twice the worst error measured on a B200 (1000 W power limit): 2.7e-7 at
(128, 4, 64, 64) (fp32 window sums over shifted planes, double SSIM formula)."""
import numpy as np
import pytest
import torch

from helpers import report, st
import ssim_oracle
from svrs_native import metrics
from svrs_native.lib import SvrsError, lib

pytestmark = pytest.mark.gpu
DEV = "cuda"
TOL = 6e-7


def _inputs(kind, shape, seed):
    """numpy PCG64 image pairs in [0, 1]."""
    rng = np.random.default_rng(seed)
    N, C, H, W = shape
    yy, xx = np.meshgrid(np.linspace(0, 1, H), np.linspace(0, 1, W), indexing="ij")
    ph = rng.uniform(0, 6, (N, C, 1, 1))
    smooth = 0.5 + 0.3 * np.sin(6 * xx + ph) * np.cos(5 * yy - ph)
    if kind == "textured":
        a, b = smooth, smooth + 0.05 * np.sin(11 * xx + 3 * yy + ph)
    elif kind == "noisy":
        a, b = smooth, smooth + 0.1 * rng.standard_normal(shape)
    elif kind == "unrelated":
        a, b = rng.random(shape), rng.random(shape)
    elif kind == "saturated":      # flat sigmoid outputs near 0.98: E[a^2] - E[a]^2 cancels in fp32 without the shift
        a = 1 / (1 + np.exp(-(3.9 + 0.05 * rng.standard_normal(shape))))
        b = 1 / (1 + np.exp(-(3.9 + 0.05 * rng.standard_normal(shape))))
    else:                          # identical
        a = np.clip(smooth + 0.05 * rng.standard_normal(shape), 0, 1)
        b = a
    return np.clip(a, 0, 1).astype(np.float32), np.clip(b, 0, 1).astype(np.float32)


KINDS = ["textured", "noisy", "unrelated", "saturated", "identical"]


@pytest.mark.parametrize("shape", [(8, 4, 32, 32), (128, 4, 64, 64), (2, 4, 256, 256), (3, 4, 37, 50), (5, 1, 11, 11)])
def test_ssim_matches_oracle(shape):
    worst = 0.0
    for win in (11, 7):
        for R in (1.0, 2.0):
            for i, kind in enumerate(KINDS):
                a, b = _inputs(kind, shape, 100 * win + 10 * int(R) + i)
                got = metrics.ssim(torch.from_numpy(a).to(DEV), torch.from_numpy(b).to(DEV), win, R)
                assert got.dtype == torch.float64 and got.shape == (shape[0],) and got.device.type == "cuda"
                ref = torch.from_numpy(ssim_oracle.ssim(a, b, win, R))
                worst = max(worst, report(f"ssim {shape} win {win} R {R} {kind}", got, ref, 0.0, atol=TOL) * float(ref.abs().max()))
                if kind == "identical":
                    assert float((got - 1).abs().max()) <= 1e-6
    print(f"[parity] ssim {shape}: worst |err| {worst:.3e}")


def test_ssim_unaligned_rows_take_the_scalar_path():
    """A contiguous tensor whose storage starts 4 bytes past a 16-byte boundary (and a 16-byte-aligned one as reference)."""
    a, b = _inputs("noisy", (4, 4, 64, 64), 7)
    n = a.size
    buf_a, buf_b = torch.empty(n + 1, device=DEV), torch.empty(n + 1, device=DEV)
    ua, ub = buf_a[1:].view(a.shape), buf_b[1:].view(b.shape)
    ua.copy_(torch.from_numpy(a))
    ub.copy_(torch.from_numpy(b))
    assert ua.is_contiguous() and ua.data_ptr() % 16 == 4
    got = metrics.ssim(ua, ub)
    report("ssim unaligned", got, torch.from_numpy(ssim_oracle.ssim(a, b)), 0.0, atol=TOL)
    assert torch.equal(got, metrics.ssim(torch.from_numpy(a).to(DEV), torch.from_numpy(b).to(DEV)))


def test_ssim_deterministic_and_graph_capturable():
    a, b = (torch.from_numpy(t).to(DEV) for t in _inputs("noisy", (128, 4, 64, 64), 3))
    r1, r2 = metrics.ssim(a, b), metrics.ssim(a, b)
    assert torch.equal(r1, r2), "two calls differ"
    ws = torch.empty(lib.ssim_workspace_doubles(128, 4, 64, 64, 11), device=DEV, dtype=torch.float64)
    out = torch.full((128,), float("nan"), device=DEV, dtype=torch.float64)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    g = torch.cuda.CUDAGraph()
    with torch.cuda.stream(s):
        with torch.cuda.graph(g, stream=s):
            lib.ssim(a.data_ptr(), b.data_ptr(), 128, 4, 64, 64, 11, 1.0, ws.data_ptr(), out.data_ptr(), s.cuda_stream)
    torch.cuda.current_stream().wait_stream(s)
    g.replay()
    torch.cuda.synchronize()
    assert torch.equal(out, r1), "graph replay differs from the eager call"


def test_ssim_writes_nothing_outside_out_and_workspace():
    N, C, H, W, win = 6, 4, 37, 50, 7
    a, b = (torch.from_numpy(t).to(DEV) for t in _inputs("textured", (N, C, H, W), 5))
    nws = lib.ssim_workspace_doubles(N, C, H, W, win)
    G = 1024
    wsb = torch.full((nws + 2 * G,), 12345.0, device=DEV, dtype=torch.float64)
    outb = torch.full((N + 2 * G,), -777.0, device=DEV, dtype=torch.float64)
    lib.ssim(a.data_ptr(), b.data_ptr(), N, C, H, W, win, 1.0, wsb[G:].data_ptr(), outb[G:].data_ptr(), st())
    torch.cuda.synchronize()
    assert bool((wsb[:G] == 12345.0).all()) and bool((wsb[G + nws:] == 12345.0).all()), "workspace guard band written"
    assert bool((outb[:G] == -777.0).all()) and bool((outb[G + N:] == -777.0).all()), "out guard band written"
    report("ssim via raw ABI", outb[G:G + N], torch.from_numpy(ssim_oracle.ssim(a.cpu().numpy(), b.cpu().numpy(), win)), 0.0, atol=TOL)


def test_ssim_library_limits_raise():
    a = torch.rand(2, 4, 16, 16, device=DEV)
    with pytest.raises(SvrsError, match="odd and >= 3"):
        metrics.ssim(a, a, win_size=1)
    wide = torch.rand(1, 1, 11, 410, device=DEV)
    with pytest.raises(SvrsError, match="shared memory"):
        metrics.ssim(wide, wide)
    out = torch.empty(2, device=DEV, dtype=torch.float64)
    with pytest.raises(SvrsError, match="C > 0"):
        lib.ssim(a.data_ptr(), a.data_ptr(), 2, 0, 16, 16, 11, 1.0, out.data_ptr(), out.data_ptr(), st())
    with pytest.raises(SvrsError, match="null pointer"):
        lib.ssim(a.data_ptr(), None, 2, 4, 16, 16, 11, 1.0, out.data_ptr(), out.data_ptr(), st())
    empty = torch.empty(0, 4, 16, 16, device=DEV)
    assert metrics.ssim(empty, empty).shape == (0,)


class _RecordingRun:
    def __init__(self):
        self.logs = []

    def log(self, d, step=None):
        self.logs.append((dict(d), step))

    def finish(self):
        pass


def _spy(model, name, store):
    orig = getattr(model, name)

    def wrapped(*a, **k):
        out = orig(*a, **k)
        store.append((a, out))
        return out
    setattr(model, name, wrapped)


def _oracle_mean(pairs):
    vals = np.concatenate([ssim_oracle.ssim(a.cpu().numpy(), b.cpu().numpy()) for a, b in pairs])
    return float(vals.mean())


def test_evaluate_logs_reference_ssim_metrics():
    """evaluate(full_val=True) on Cond_SRVAE(2, 64) and VAE(2, 32), eval mode: the logged Metrics/SSIM* equal the oracle's mean over
    the pairs evaluate() formed (spies keep the tensors forward / conditional_generation returned: both draw Philox noise),
    and exactly the reference's keys are logged (epoch 3: no image logging)."""
    import models
    from torch.utils.data import DataLoader, TensorDataset

    g = torch.Generator().manual_seed(0)
    hr = torch.rand(7, 4, 64, 64, generator=g)
    loader = DataLoader(TensorDataset(torch.nn.functional.avg_pool2d(hr, 2), hr), batch_size=3)
    torch.manual_seed(0)
    model = models.Cond_SRVAE(2, 64).to(DEV).eval()
    fw, gen = [], []
    _spy(model, "forward", fw)
    _spy(model, "conditional_generation", gen)
    run = _RecordingRun()
    model.evaluate(loader, run, 3, full_val=True)
    assert len(fw) == len(gen) == 1 + 3            # the image batch, then every validation batch
    assert [set(d) for d, _ in run.logs] == [{"Metrics/SSIM_LR", "Metrics/SSIM_HR", "Metrics/SSIM_SR"}] and run.logs[0][1] == 3
    logged = run.logs[0][0]
    want = {"Metrics/SSIM_LR": _oracle_mean([(a[1], out[1]) for a, out in fw[1:]]),
            "Metrics/SSIM_HR": _oracle_mean([(a[0], out[0]) for a, out in fw[1:]]),
            "Metrics/SSIM_SR": _oracle_mean([(fa[0], g_out) for (fa, _), (_, g_out) in zip(fw[1:], gen[1:])])}
    for k, v in want.items():
        print(f"[parity] {k}: logged {logged[k]:.9f} oracle {v:.9f}")
        assert isinstance(logged[k], float) and abs(logged[k] - v) <= TOL, k
    run2 = _RecordingRun()
    model.evaluate(loader, run2, 3, full_val=False)
    assert run2.logs == []

    x = torch.rand(5, 4, 32, 32, generator=g)
    vloader = DataLoader(TensorDataset(x, x), batch_size=2)
    vae = models.VAE(2, 32).to(DEV).eval()
    fw = []
    _spy(vae, "forward", fw)
    run = _RecordingRun()
    vae.evaluate(vloader, run, 3, full_val=True)
    assert len(fw) == 1 + 3
    assert [set(d) for d, _ in run.logs] == [{"Metrics/SSIM"}]
    v = _oracle_mean([(a[0], out[0]) for a, out in fw[1:]])
    print(f"[parity] Metrics/SSIM: logged {run.logs[0][0]['Metrics/SSIM']:.9f} oracle {v:.9f}")
    assert abs(run.logs[0][0]["Metrics/SSIM"] - v) <= TOL
