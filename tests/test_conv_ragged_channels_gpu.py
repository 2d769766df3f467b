"""tcgen05 convolutions with channel counts that are multiples of 8 but not of 16 / 64 (-m gpu), through the C ABI.

conv_tc (fprop, dgrad) reads the reduction channels in ceil(K / cw) chunks whose last box TMA zero-fills; wgrad_tc
zero-fills the last G box (columns past Ca) and the last X box (rows past Cb) and clips them in its epilogues.  Each case
runs one conv form (c3 = k3 s1, c4 = k4 s2, ct = transposed k4 s2) on tcgen05 and on the CUDA-core kernels
(svrs_set_tc_enabled(0)) and compares both with float64 torch on the same bf16-rounded inputs.  Bounds as
tests/test_kernels_gpu.py: 7e-3 relative to the maximum for bf16 conv outputs, 2e-5 for weight and bias gradients.

Every output sits inside a sentinel guard band; the per-tap packed gradient [tap][Cb][Ca] has at least one tap's worth
of guard rows after the last tap, so a ragged box that spilled past Cb or Ca would show."""
import pytest
import torch
import torch.nn.functional as F

from helpers import BF16, Guarded, lib, nchw, nhwc, pack, report, st

pytestmark = pytest.mark.gpu
DEV = "cuda"

# Layers of Cond_SRVAE(1.5, 64) and Cond_SRVAE(1.2, 64) that leave the CUDA-core kernels, at their own map and 128
# patches (tests/test_cpu_ragged_dispatch.py derives the list from the models): N, H, W, Cin, Cout, form
MOVED = [
    (128, 8, 8, 128, 336, "c3"),      # encoder_x, cr 1.5
    (128, 8, 8, 336, 336, "c3"),      # decoder_x conv
    (128, 8, 8, 336, 256, "ct"),      # decoder_x upsample
    (128, 4, 4, 128, 672, "c3"),      # y_to_z
    (128, 4, 4, 168, 168, "c3"),      # u_to_z
    (128, 4, 4, 168, 672, "c3"),
    (128, 4, 4, 1344, 672, "c3"),     # mu / logvar heads
    (128, 4, 4, 672, 672, "c3"),
    (128, 8, 8, 128, 424, "c3"),      # encoder_x, cr 1.2
    (128, 8, 8, 424, 424, "c3"),
    (128, 8, 8, 424, 256, "ct"),
    (128, 4, 4, 128, 848, "c3"),
    (128, 4, 4, 1696, 848, "c3"),
    (128, 4, 4, 848, 848, "c3"),
]

# Small cases for every chunk width of a ragged reduction (24 -> one 32-channel box, 40 / 56 -> one 64-channel box,
# 72 / 168 / 424 -> 64-channel chunks with a ragged last one), output channels ragged and not, and image counts that
# leave the last TMA box part-empty (4x4 maps: 8 images a box, 8x8: 2, 2x2: 32).
SMALL = [
    (3, 8, 8, 24, 64),
    (2, 8, 8, 40, 24),
    (5, 4, 4, 56, 40),
    (2, 8, 8, 72, 128),
    (3, 4, 4, 168, 72),
    (2, 8, 8, 424, 56),
    (2, 16, 16, 24, 40),
    (1, 4, 4, 104, 168),
]
CASES = MOVED + [c + (f,) for c in SMALL for f in ("c3", "c4", "ct")]


def _rand(shape, gen):
    return torch.randn(shape, generator=gen).to(torch.bfloat16).float()


def _ids(c):
    return "x".join(str(v) for v in c)


@pytest.mark.parametrize("case", CASES, ids=_ids)
def test_ragged_conv_fprop_dgrad_wgrad(case):
    N, H, W, Cin, Cout, form = case
    dtype = torch.bfloat16
    g = torch.Generator().manual_seed(N * 7 + H + Cin * 3 + Cout + len(form))
    ks = 3 if form == "c3" else 4
    x = _rand((N, Cin, H, W), g)
    b = torch.randn(Cout, generator=g)
    if form == "ct":
        w = _rand((Cin, Cout, 4, 4), g) * 0.1
        w = w.to(dtype).float()
        fwd = lambda xx, ww, bb: F.conv_transpose2d(xx, ww, bb, stride=2, padding=1)
        gh, gw = H, W                      # conv_tc's grid: the coarse input grid (one problem per output parity)
    else:
        w = (_rand((Cout, Cin, ks, ks), g) * 0.1).to(dtype).float()
        s = 1 if form == "c3" else 2
        fwd = lambda xx, ww, bb: F.conv2d(xx, ww, bb, stride=s, padding=1)
        gh, gw = H // s, W // s
    # float64 truth (on the device: the moved layers are tens of GFLOP)
    xr = x.to(DEV).double().requires_grad_(True)
    wr = w.to(DEV).double().requires_grad_(True)
    br = b.to(DEV).double().requires_grad_(True)
    yr = fwd(xr, wr, br)
    gy = _rand(tuple(yr.shape), g)
    yr.backward(gy.to(DEV).double())
    OH, OW = yr.shape[2], yr.shape[3]

    # the new rule takes every GEMM of the layer on tcgen05 (the parent sent at least one of them to the CUDA cores)
    assert lib.tc_would_run(BF16, Cin, Cout, gh, gw) == 1, "fprop not on tcgen05"
    assert lib.tc_would_run(BF16, Cout, Cin, gh, gw) == 1, "dgrad not on tcgen05"
    if form == "ct":
        layout = lib.convT2d_wgrad_layout(BF16, N, H, W, Cin, Cout)
    else:
        layout = lib.conv2d_wgrad_layout(BF16, N, H, W, Cin, Cout, ks)
    assert layout == 1, "wgrad not on tcgen05"

    xd, wd, bd, gyd = nhwc(x.to(DEV), dtype), w.to(DEV), b.to(DEV), nhwc(gy.to(DEV), dtype)
    pf, pb = pack(wd, dtype, convT=(form == "ct"))
    wshape = tuple(w.shape)
    kk = wshape[2] * wshape[3]
    Ca, Cb = (Cin, Cout) if form == "ct" else (Cout, Cin)     # packed gradient [tap][Cb][Ca]
    dw0 = torch.randn(wshape, generator=g).to(DEV)            # non-zero starting gradients: the kernels accumulate
    db0 = torch.randn(Cout, generator=g).to(DEV)

    def wgrad(dw, dwp, db):
        if form == "ct":
            lib.convT2d_wgrad(xd.data_ptr(), gyd.data_ptr(), dw, dwp, db, BF16, N, H, W, Cin, Cout, 0, st())
        else:
            lib.conv2d_wgrad(xd.data_ptr(), gyd.data_ptr(), dw, dwp, db, BF16, N, H, W, Cin, Cout, ks, 0, st())

    res = {}
    try:
        for tc in (1, 0):
            lib.set_tc_enabled(tc)
            y = Guarded((N, OH, OW, Cout), dtype)
            dx = Guarded(tuple(xd.shape), dtype)
            if form == "ct":
                lib.convT2d_fprop(xd.data_ptr(), pf.data_ptr(), pb.data_ptr(), bd.data_ptr(), y.t.data_ptr(), BF16, N, H, W, Cin, Cout, 0, st())
                lib.convT2d_dgrad(gyd.data_ptr(), pb.data_ptr(), pf.data_ptr(), dx.t.data_ptr(), BF16, N, H, W, Cin, Cout, st())
            else:
                lib.conv2d_fprop(xd.data_ptr(), pf.data_ptr(), pb.data_ptr(), bd.data_ptr(), y.t.data_ptr(), BF16, N, H, W, Cin, Cout, ks, 0, st())
                lib.conv2d_dgrad(gyd.data_ptr(), pb.data_ptr(), pf.data_ptr(), dx.t.data_ptr(), BF16, N, H, W, Cin, Cout, ks, st())
            # torch layout, accumulating into non-zero dw / db
            dw = Guarded(wshape, torch.float32)
            dw.t.copy_(dw0)
            db = Guarded((Cout,), torch.float32)
            db.t.copy_(db0)
            wgrad(dw.t.data_ptr(), None, db.t.data_ptr())
            # torch layout without a bias gradient
            dw_nb = Guarded(wshape, torch.float32, fill=0.0)
            wgrad(dw_nb.t.data_ptr(), None, None)
            torch.cuda.synchronize()
            for name, gb in (("y", y), ("dx", dx), ("dw", dw), ("db", db), ("dw (no db)", dw_nb)):
                assert gb.intact(), f"tc={tc}: {name} written outside its buffer"
            res[tc] = (nchw(y.t), nchw(dx.t), dw.t - dw0, db.t - db0, dw_nb.t.clone())

        # per-tap packed scratch (what the fused optimiser reads), accumulating into a non-zero scratch; dw must stay untouched
        lib.set_tc_enabled(1)
        guard_rows = max(4096, Ca * Cb)
        pk = Guarded((kk, Cb, Ca), torch.float32, pad=guard_rows)
        pk0 = torch.randn((kk, Cb, Ca), generator=g).to(DEV)
        pk.t.copy_(pk0)
        untouched = Guarded(wshape, torch.float32, fill=0.0)
        dbp = Guarded((Cout,), torch.float32, fill=0.0)
        wgrad(untouched.t.data_ptr(), pk.t.data_ptr(), dbp.t.data_ptr())
        pk_nb = Guarded((kk, Cb, Ca), torch.float32, fill=0.0, pad=guard_rows)
        wgrad(untouched.t.data_ptr(), pk_nb.t.data_ptr(), None)
        torch.cuda.synchronize()
    finally:
        lib.set_tc_enabled(1)
    assert pk.intact() and pk_nb.intact(), "packed gradient written past its taps"
    assert dbp.intact() and untouched.intact()
    assert float(untouched.t.abs().max()) == 0.0, "packed mode wrote the torch-layout buffer"
    to_torch = lambda p: p.permute(2, 1, 0).reshape(wshape)      # [tap][b][a] -> [a][b][tap]

    tag = f"{form} {N}x{H}x{W} {Cin}->{Cout}"
    y1, dx1, dw1, db1, dwnb1 = res[1]
    y0, dx0, dw0s, db0s, dwnb0 = res[0]
    report(f"{tag} fprop tc vs fp64", y1, yr.detach(), 7e-3)
    report(f"{tag} dgrad tc vs fp64", dx1, xr.grad, 7e-3)
    report(f"{tag} fprop tc vs simt", y1, y0, 8e-3)
    report(f"{tag} dgrad tc vs simt", dx1, dx0, 8e-3)
    report(f"{tag} wgrad tc vs fp64", dw1, wr.grad, 2e-5)
    report(f"{tag} wgrad tc vs simt", dw1, dw0s, 2e-5)
    report(f"{tag} wgrad simt vs fp64", dw0s, wr.grad, 2e-5)
    report(f"{tag} wgrad (no db) tc vs fp64", dwnb1, wr.grad, 2e-5)
    report(f"{tag} wgrad (no db) simt vs fp64", dwnb0, wr.grad, 2e-5)
    report(f"{tag} bgrad tc vs fp64", db1, br.grad, 2e-5)
    report(f"{tag} bgrad simt vs fp64", db0s, br.grad, 2e-5)
    report(f"{tag} packed wgrad vs fp64", to_torch(pk.t - pk0), wr.grad, 2e-5)
    report(f"{tag} packed wgrad (no db) vs fp64", to_torch(pk_nb.t), wr.grad, 2e-5)
    report(f"{tag} packed-mode bgrad vs fp64", dbp.t, br.grad, 2e-5)
