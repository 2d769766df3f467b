"""CPU tests of the host-side argument checks of the ELBO and sampling entry points (csrc/elbo.cu, csrc/sample_stats.cu):
strides shorter than a row, zero latent widths and pointers that are not 16-byte aligned for the kernels' vector
accesses are rejected with SVRS_E_ARG before anything is enqueued.

The pointers are fake integers, and the tests run only without a CUDA device.  A library without one of these checks can
then never reach memory: the call gets as far as the launch and fails with a CUDA error, which the message match tells
apart from the argument error."""
import pytest
import torch

from svrs_native.lib import ACT_SIGMOID, F32, SvrsError, lib

pytestmark = pytest.mark.skipif(torch.cuda.is_available(), reason="passes fake device pointers; host-only")

A, M = 0x10000, 0x10004        # a 16-byte aligned and a 4-byte aligned (misaligned) fake device address


def _latents(**kw):
    a = dict(mu3=A, lv3=A, ld3=16, yflat=A, ldy=16, eps=A, stack=A, B=2, S=4, Wz=16)
    a.update(kw)
    lib.sample_latents(a["mu3"], a["lv3"], a["ld3"], a["yflat"], a["ldy"], a["eps"], a["stack"], a["B"], a["S"], a["Wz"],
                       1, 2, 0, None, None)


@pytest.mark.parametrize("arg", ["mu3", "lv3", "yflat", "eps", "stack"])
def test_sample_latents_rejects_misaligned_pointers(arg):
    with pytest.raises(SvrsError, match="aligned"):
        _latents(**{arg: M})


@pytest.mark.parametrize("arg", ["ld3", "ldy"])
def test_sample_latents_rejects_rows_shorter_than_wz(arg):
    with pytest.raises(SvrsError, match=r"must be >= Wz \(16\)"):
        _latents(**{arg: 12})


def _tail(**kw):
    a = dict(x=A, target=A)
    a.update(kw)
    lib.sample_tail_stats(a["x"], F32, A, A, a["target"], 1, 8, 8, 8, 16, 4, 1, A, A, A, A, A, A, A, None)


@pytest.mark.parametrize("arg", ["x", "target"])
def test_sample_tail_stats_rejects_misaligned_pointers(arg):
    with pytest.raises(SvrsError, match="aligned"):
        _tail(**{arg: M})


def _elbo_args(**kw):
    a = dict(nx=16, ny=16, mu1=A, ld1=8, W1=8, mu2=A, ld2=8, ld3=8, W2=8, B=2)
    a.update(kw)
    return a


def _elbo_fwd(**kw):
    a = _elbo_args(**kw)
    lib.elbo_fwd(A, A, F32, F32, a["nx"], A, A, F32, F32, a["ny"], a["mu1"], A, a["ld1"], a["W1"], a["mu2"], A, a["ld2"],
                 A, A, a["ld3"], a["W2"], a["B"], A, None)


def _elbo_bwd(dld1=8, dld2=8, dld3=8, **kw):
    a = _elbo_args(**kw)
    lib.elbo_bwd(A, A, F32, F32, a["nx"], A, F32, A, A, F32, F32, a["ny"], A, F32,
                 a["mu1"], A, a["ld1"], a["W1"], A, A, dld1,
                 a["mu2"], A, a["ld2"], A, A, dld2,
                 A, A, a["ld3"], a["W2"], A, A, dld3,
                 a["B"], A, A, A, A, ACT_SIGMOID, None)


@pytest.mark.parametrize("call", [_elbo_fwd, _elbo_bwd], ids=["fwd", "bwd"])
@pytest.mark.parametrize("kw,msg", [(dict(ld1=4), r"ld1 \(4\) < W1 \(8\)"),
                                    (dict(ld2=4), r"ld2 \(4\) / ld3 \(8\) < W2 \(8\)"),
                                    (dict(ld3=4), r"ld2 \(8\) / ld3 \(4\) < W2 \(8\)"),
                                    (dict(W1=0), r"W1 > 0"),
                                    (dict(W2=0), r"W2 > 0")],
                         ids=["ld1", "ld2", "ld3", "W1", "W2"])
def test_elbo_rejects_short_rows_and_zero_widths(call, kw, msg):
    with pytest.raises(SvrsError, match=msg):
        call(**kw)


@pytest.mark.parametrize("kw,msg", [(dict(dld1=4), r"dld1 \(4\) < W1 \(8\)"),
                                    (dict(dld2=4), r"dld2 \(4\) < W2 \(8\)"),
                                    (dict(dld3=4), r"dld3 \(4\) < W2 \(8\)")],
                         ids=["dld1", "dld2", "dld3"])
def test_elbo_bwd_rejects_gradient_rows_shorter_than_width(kw, msg):
    with pytest.raises(SvrsError, match=msg):
        _elbo_bwd(**kw)
