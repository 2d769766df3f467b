"""Kernel-level parity (-m gpu): every C-ABI entry point against a float64 CPU evaluation of the torch op the
reference calls at that site (and against oracle/np_primitives for first-principles definitions).

Tolerances: fp32 kernels 1e-5 relative to the tensor's max magnitude (north star: 1e-5 in fp32);
bf16 kernels 7e-3 relative-to-max per element (<= 2x the measured 3.6e-3: bf16 has 8 mantissa bits; inputs are pre-rounded to
bf16 so the only error is the bf16 rounding of the OUTPUT plus fp32 accumulation order)."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from helpers import BF16, F32, Guarded, dt, lib, nchw, nhwc, pack, report, st

pytestmark = pytest.mark.gpu
DEV = "cuda"

TOL = {torch.float32: 1e-5, torch.bfloat16: 7e-3}      # bf16: <= 2x the measured 3.6e-3 (output rounding to bf16 = 2^-9 relative)

CONV_CASES = [
    # N, H, W, Cin, Cout
    (2, 8, 8, 16, 32),
    (3, 6, 10, 5, 7),        # odd channel counts + non-square: scalar load paths
    (1, 4, 4, 128, 64),
    (2, 16, 16, 4, 4),       # first layers of every encoder
    (3, 16, 16, 16, 4),      # image-side ends: narrow wgrad kernel (one warp per tap)
    (2, 16, 32, 4, 16),
    (2, 8, 8, 64, 16),
    (1, 4, 4, 42, 84),       # cr = 1.5 channel counts (SURVEY 8.2)
    (5, 2, 2, 8, 130),
]


def _rand(shape, gen, dtype):
    t = torch.randn(shape, generator=gen)
    return t.to(dtype).float() if dtype == torch.bfloat16 else t   # pre-round so the reference sees the same inputs


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("ksize", [3, 4])
@pytest.mark.parametrize("case", CONV_CASES)
def test_conv2d_fprop_dgrad_wgrad(case, ksize, dtype):
    N, H, W, Cin, Cout = case
    g = torch.Generator().manual_seed(hash((case, ksize)) % 2**31)
    stride = 1 if ksize == 3 else 2
    x = _rand((N, Cin, H, W), g, dtype)
    w = _rand((Cout, Cin, ksize, ksize), g, dtype) * 0.2
    w = w.to(dtype).float() if dtype == torch.bfloat16 else w
    b = torch.randn(Cout, generator=g)
    xr = x.double().requires_grad_(True)
    wr = w.double().requires_grad_(True)
    br = b.double().requires_grad_(True)
    yr = F.conv2d(xr, wr, br, stride=stride, padding=1)
    gy = _rand(tuple(yr.shape), g, dtype)
    yr.backward(gy.double())

    xd, wd, bd, gyd = nhwc(x.to(DEV), dtype), w.to(DEV), b.to(DEV), nhwc(gy.to(DEV), dtype)
    pf, pb = pack(wd, dtype)
    OH, OW = yr.shape[2], yr.shape[3]
    y = torch.empty((N, OH, OW, Cout), device=DEV, dtype=dtype)
    lib.conv2d_fprop(xd.data_ptr(), pf.data_ptr(), pb.data_ptr(), bd.data_ptr(), y.data_ptr(), dt(dtype), N, H, W, Cin, Cout, ksize, 0, st())
    report(f"conv{ksize} fprop {case} {dtype}", nchw(y), yr, TOL[dtype])

    dx = torch.empty_like(xd)
    lib.conv2d_dgrad(gyd.data_ptr(), pb.data_ptr(), pf.data_ptr(), dx.data_ptr(), dt(dtype), N, H, W, Cin, Cout, ksize, st())
    report(f"conv{ksize} dgrad {case} {dtype}", nchw(dx), xr.grad, TOL[dtype])

    dw = torch.zeros_like(wd)
    db = torch.zeros_like(bd)
    lib.conv2d_wgrad(xd.data_ptr(), gyd.data_ptr(), dw.data_ptr(), None, db.data_ptr(), dt(dtype), N, H, W, Cin, Cout, ksize, 0, st())
    report(f"conv{ksize} wgrad {case} {dtype}", dw, wr.grad, 2e-5 if dtype == torch.float32 else 1e-5)
    report(f"conv{ksize} bgrad {case} {dtype}", db, br.grad, 2e-5 if dtype == torch.float32 else 1e-5)


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("case", CONV_CASES)
def test_convT2d_fprop_dgrad_wgrad(case, dtype):
    N, H, W, Cin, Cout = case
    g = torch.Generator().manual_seed(hash(case) % 2**31)
    x = _rand((N, Cin, H, W), g, dtype)
    w = (_rand((Cin, Cout, 4, 4), g, dtype) * 0.2)
    w = w.to(dtype).float() if dtype == torch.bfloat16 else w
    b = torch.randn(Cout, generator=g)
    xr, wr, br = x.double().requires_grad_(True), w.double().requires_grad_(True), b.double().requires_grad_(True)
    yr = F.conv_transpose2d(xr, wr, br, stride=2, padding=1)
    gy = _rand(tuple(yr.shape), g, dtype)
    yr.backward(gy.double())
    xd, wd, bd, gyd = nhwc(x.to(DEV), dtype), w.to(DEV), b.to(DEV), nhwc(gy.to(DEV), dtype)
    pf, pb = pack(wd, dtype, convT=True)
    y = torch.empty((N, 2 * H, 2 * W, Cout), device=DEV, dtype=dtype)
    lib.convT2d_fprop(xd.data_ptr(), pf.data_ptr(), pb.data_ptr(), bd.data_ptr(), y.data_ptr(), dt(dtype), N, H, W, Cin, Cout, 0, st())
    report(f"convT fprop {case} {dtype}", nchw(y), yr, TOL[dtype])
    dx = torch.empty_like(xd)
    lib.convT2d_dgrad(gyd.data_ptr(), pb.data_ptr(), pf.data_ptr(), dx.data_ptr(), dt(dtype), N, H, W, Cin, Cout, st())
    report(f"convT dgrad {case} {dtype}", nchw(dx), xr.grad, TOL[dtype])
    dw, db = torch.zeros_like(wd), torch.zeros_like(bd)
    lib.convT2d_wgrad(xd.data_ptr(), gyd.data_ptr(), dw.data_ptr(), None, db.data_ptr(), dt(dtype), N, H, W, Cin, Cout, 0, st())
    report(f"convT wgrad {case} {dtype}", dw, wr.grad, 2e-5 if dtype == torch.float32 else 1e-5)
    report(f"convT bgrad {case} {dtype}", db, br.grad, 2e-5 if dtype == torch.float32 else 1e-5)


def test_conv_first_principles_numpy():
    """The kernels against oracle/np_primitives (explicit definition), not just against torch."""
    from oracle import np_primitives as npp
    g = torch.Generator().manual_seed(3)
    x = torch.randn(2, 3, 6, 6, generator=g)
    w3 = torch.randn(5, 3, 3, 3, generator=g)
    w4 = torch.randn(5, 3, 4, 4, generator=g)
    wt = torch.randn(3, 5, 4, 4, generator=g)
    b = torch.randn(5, generator=g)
    xd = nhwc(x.to(DEV))
    bd = b.to(DEV)          # keep device tensors alive: a temporary's storage is recycled as soon as data_ptr() returns
    for ks, w in ((3, w3), (4, w4)):
        ref = npp.conv2d(x.numpy(), w.numpy(), b.numpy(), 1 if ks == 3 else 2, 1)
        pf, pb = pack(w.to(DEV), torch.float32)
        y = torch.empty((2, ref.shape[2], ref.shape[3], 5), device=DEV)
        lib.conv2d_fprop(xd.data_ptr(), pf.data_ptr(), pb.data_ptr(), bd.data_ptr(), y.data_ptr(), F32, 2, 6, 6, 3, 5, ks, 0, st())
        report(f"conv{ks} vs numpy definition", nchw(y), torch.from_numpy(ref), 1e-5)
    ref = npp.conv_transpose2d_k4s2p1(x.numpy(), wt.numpy(), b.numpy())
    pf, pb = pack(wt.to(DEV), torch.float32, convT=True)
    y = torch.empty((2, 12, 12, 5), device=DEV)
    lib.convT2d_fprop(xd.data_ptr(), pf.data_ptr(), pb.data_ptr(), bd.data_ptr(), y.data_ptr(), F32, 2, 6, 6, 3, 5, 0, st())
    report("convT vs numpy definition", nchw(y), torch.from_numpy(ref), 1e-5)


@pytest.mark.parametrize("act,fn", [(1, torch.sigmoid), (2, lambda t: F.hardtanh(t, -7.0, 7.0))])
def test_conv_epilogue_activation_and_backward(act, fn):
    g = torch.Generator().manual_seed(11)
    x = torch.randn(2, 8, 4, 4, generator=g) * 3
    w = torch.randn(12, 8, 3, 3, generator=g)
    b = torch.randn(12, generator=g)
    pre = F.conv2d(x.double(), w.double(), b.double(), padding=1).requires_grad_(True)
    yr = fn(pre)
    gy = torch.randn(yr.shape, generator=g).double()
    yr.backward(gy)
    pf, pb = pack(w.to(DEV), torch.float32)
    xd = nhwc(x.to(DEV))
    bd = b.to(DEV)
    y = torch.empty((2, 4, 4, 12), device=DEV)
    lib.conv2d_fprop(xd.data_ptr(), pf.data_ptr(), pb.data_ptr(), bd.data_ptr(), y.data_ptr(), F32, 2, 4, 4, 8, 12, 3, act, st())
    report(f"conv + act {act}", nchw(y), yr, 1e-5)
    gyd = nhwc(gy.float().to(DEV))
    lib.act_bwd(y.data_ptr(), gyd.data_ptr(), gyd.data_ptr(), F32, act, gyd.numel(), st())
    report(f"act {act} backward", nchw(gyd), pre.grad, 1e-5)


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("shape", [(4, 16, 8, 8), (2, 64, 16, 16), (3, 256, 4, 4), (1, 128, 2, 2),
                                   (9, 64, 64, 61), (70, 256, 16, 15), (40, 1024, 8, 8)])   # >= 4 MB: bulk-copy streaming reduce, ragged tails
def test_batchnorm_train_fwd_bwd(shape, dtype):
    N, C, H, W = shape
    g = torch.Generator().manual_seed(C)
    x = (torch.randn(shape, generator=g) * 2 + 3)   # non-zero mean: exercises the variance cancellation
    x = x.to(dtype).float()
    gam, bet = torch.rand(C, generator=g) + 0.5, torch.randn(C, generator=g)
    bn = torch.nn.BatchNorm2d(C).double()
    with torch.no_grad():
        bn.weight.copy_(gam); bn.bias.copy_(bet)
    bn.train()
    xr = x.double().requires_grad_(True)
    yr = F.relu(bn(xr))
    gy = torch.randn(shape, generator=g).to(dtype).float()
    yr.backward(gy.double())
    M = N * H * W
    xd, gyd = nhwc(x.to(DEV), dtype), nhwc(gy.to(DEV), dtype)
    sums = torch.zeros(2 * C * 8, device=DEV, dtype=torch.float64)   # SVRS_BN_REPLICAS copies
    rm, rv = torch.zeros(C, device=DEV), torch.ones(C, device=DEV)
    nbt = torch.zeros((), device=DEV, dtype=torch.int64)
    scale, shift, mean, invstd = (torch.empty(C, device=DEV) for _ in range(4))
    gam_d, bet_d = gam.to(DEV), bet.to(DEV)
    lib.bn_stats(xd.data_ptr(), dt(dtype), M, C, sums.data_ptr(), st())
    lib.bn_finalize_train(sums.data_ptr(), M, C, gam_d.data_ptr(), bet_d.data_ptr(), 1e-5, 0.1, rm.data_ptr(),
                          rv.data_ptr(), nbt.data_ptr(), 1, scale.data_ptr(), shift.data_ptr(), mean.data_ptr(), invstd.data_ptr(), st())
    y = torch.empty_like(xd)
    lib.bn_apply(xd.data_ptr(), y.data_ptr(), dt(dtype), M, C, scale.data_ptr(), shift.data_ptr(), 1, st())
    report(f"bn fwd {shape} {dtype}", nchw(y), yr, TOL[dtype])
    report("bn running_mean", rm, bn.running_mean, 1e-6)
    report("bn running_var", rv, bn.running_var, 1e-5)
    assert int(nbt) == 1
    sums2 = torch.zeros(2 * C * 8, device=DEV, dtype=torch.float64)
    dgam, dbet = torch.zeros(C, device=DEV), torch.zeros(C, device=DEV)
    lib.bn_bwd_reduce(xd.data_ptr(), gyd.data_ptr(), dt(dtype), M, C, scale.data_ptr(), shift.data_ptr(), mean.data_ptr(),
                      invstd.data_ptr(), 1, sums2.data_ptr(), st())
    dx = torch.empty_like(xd)
    lib.bn_bwd_apply(xd.data_ptr(), gyd.data_ptr(), dx.data_ptr(), dt(dtype), M, 0, C, scale.data_ptr(), shift.data_ptr(),
                     mean.data_ptr(), invstd.data_ptr(), gam_d.data_ptr(), 1, sums2.data_ptr(), dgam.data_ptr(), dbet.data_ptr(), st())
    report(f"bn bwd dx {shape} {dtype}", nchw(dx), xr.grad, 2e-5 if dtype == torch.float32 else 2e-2)
    report("bn dgamma", dgam, bn.weight.grad, 2e-5)
    report("bn dbeta", dbet, bn.bias.grad, 2e-5)
    # second running-stat update in one call (y_to_z runs twice per forward, SURVEY Q1)
    rm2, rv2 = torch.zeros(C, device=DEV), torch.ones(C, device=DEV)
    lib.bn_finalize_train(sums.data_ptr(), M, C, gam_d.data_ptr(), bet_d.data_ptr(), 1e-5, 0.1, rm2.data_ptr(),
                          rv2.data_ptr(), nbt.data_ptr(), 2, scale.data_ptr(), shift.data_ptr(), mean.data_ptr(), invstd.data_ptr(), st())
    bn(x.double())
    report("bn running_mean after 2 updates", rm2, bn.running_mean, 1e-6)
    report("bn running_var after 2 updates", rv2, bn.running_var, 1e-5)
    assert int(nbt) == 3


def test_batchnorm_eval():
    C = 16
    g = torch.Generator().manual_seed(5)
    x = torch.randn(2, C, 4, 4, generator=g)
    bn = torch.nn.BatchNorm2d(C).double().eval()
    with torch.no_grad():
        bn.running_mean.copy_(torch.randn(C, generator=g)); bn.running_var.copy_(torch.rand(C, generator=g) + 0.5)
        bn.weight.copy_(torch.rand(C, generator=g)); bn.bias.copy_(torch.randn(C, generator=g))
    yr = F.relu(bn(x.double()))
    scale, shift = torch.empty(C, device=DEV), torch.empty(C, device=DEV)
    f = lambda t: t.float().to(DEV)
    w_, b_, rm_, rv_ = f(bn.weight.data), f(bn.bias.data), f(bn.running_mean), f(bn.running_var)
    lib.bn_finalize_eval(C, w_.data_ptr(), b_.data_ptr(), 1e-5, rm_.data_ptr(), rv_.data_ptr(), scale.data_ptr(), shift.data_ptr(), st())
    xd = nhwc(x.to(DEV))
    lib.bn_apply(xd.data_ptr(), xd.data_ptr(), F32, 32, C, scale.data_ptr(), shift.data_ptr(), 1, st())
    report("bn eval", nchw(xd), yr, 1e-5)


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("shape", [(4, 16, 8, 8), (2, 64, 16, 16), (3, 256, 4, 4), (2, 1024, 2, 2)])
def test_bn_apply_train_fused_equals_two_step(shape, dtype):
    """svrs_bn_apply_train == svrs_bn_finalize_train + svrs_bn_apply, bit for bit (outputs, saved statistics, running stats)."""
    N, C, H, W = shape
    g = torch.Generator().manual_seed(N * C + H)
    x = nhwc((torch.randn(shape, generator=g) * 1.7 + 0.6).to(DEV), dtype)
    M = N * H * W
    gamma = (torch.rand(C, generator=g) + 0.5).to(DEV)
    beta = torch.randn(C, generator=g).to(DEV)
    sums = torch.zeros(2 * C * 8, device=DEV, dtype=torch.float64)   # SVRS_BN_REPLICAS copies
    lib.bn_stats(x.data_ptr(), dt(dtype), M, C, sums.data_ptr(), st())
    outs = []
    for fused in (0, 1):
        rm, rv = torch.zeros(C, device=DEV), torch.ones(C, device=DEV)
        nbt = torch.zeros((), device=DEV, dtype=torch.int64)
        scale, shift, mean, invstd = (torch.empty(C, device=DEV) for _ in range(4))
        y = torch.empty_like(x)
        if fused:
            lib.bn_apply_train(x.data_ptr(), y.data_ptr(), dt(dtype), M, 0, C, sums.data_ptr(), gamma.data_ptr(), beta.data_ptr(), 1e-5, 0.1,
                               rm.data_ptr(), rv.data_ptr(), nbt.data_ptr(), 2, 1, scale.data_ptr(), shift.data_ptr(),
                               mean.data_ptr(), invstd.data_ptr(), st())
        else:
            lib.bn_finalize_train(sums.data_ptr(), M, C, gamma.data_ptr(), beta.data_ptr(), 1e-5, 0.1, rm.data_ptr(), rv.data_ptr(),
                                  nbt.data_ptr(), 2, scale.data_ptr(), shift.data_ptr(), mean.data_ptr(), invstd.data_ptr(), st())
            lib.bn_apply(x.data_ptr(), y.data_ptr(), dt(dtype), M, C, scale.data_ptr(), shift.data_ptr(), 1, st())
        torch.cuda.synchronize()
        outs.append((y, scale, shift, mean, invstd, rm, rv, nbt))
    for a, b in zip(*outs):
        assert torch.equal(a, b)
    assert int(outs[1][7]) == 2


def test_layout_roundtrip_and_views():
    g = torch.Generator().manual_seed(2)
    x = torch.randn(3, 6, 4, 5, generator=g).to(DEV)
    out = torch.empty((3, 4, 5, 6), device=DEV)
    lib.nchw_to_nhwc(x.data_ptr(), F32, 6 * 20, out.data_ptr(), F32, 3, 6, 4, 5, st())
    assert torch.equal(out, x.permute(0, 2, 3, 1).contiguous())
    # read the left half of wider rows (torch.chunk / torch.cat views)
    wide = torch.randn(3, 2 * 120, generator=g).to(DEV)
    lib.nchw_to_nhwc(wide.data_ptr(), F32, 240, out.data_ptr(), F32, 3, 6, 4, 5, st())
    assert torch.equal(out, wide[:, :120].reshape(3, 6, 4, 5).permute(0, 2, 3, 1).contiguous())
    back = torch.zeros(3, 240, device=DEV)
    lib.nhwc_to_nchw(out.data_ptr(), F32, back.data_ptr() + 4 * 120, F32, 240, 3, 6, 4, 5, 0, st())
    assert torch.equal(back[:, 120:], wide[:, :120]) and float(back[:, :120].abs().sum()) == 0.0
    lib.nhwc_to_nchw(out.data_ptr(), F32, back.data_ptr() + 4 * 120, F32, 240, 3, 6, 4, 5, 1, st())
    assert torch.allclose(back[:, 120:], 2 * wide[:, :120])
    # bf16 conversion
    ob = torch.empty((3, 4, 5, 6), device=DEV, dtype=torch.bfloat16)
    lib.nchw_to_nhwc(x.data_ptr(), F32, 120, ob.data_ptr(), BF16, 3, 6, 4, 5, st())
    assert torch.equal(ob, x.permute(0, 2, 3, 1).contiguous().to(torch.bfloat16))
    # flat-buffer reinterpretation (SURVEY Q4): channel 5 of the 4x4 view == rows 2-3 of channel 1 of the 8x8 view
    u = torch.arange(2 * 2048, dtype=torch.float32, device=DEV).reshape(2, 2048)
    a = torch.empty((2, 4, 4, 128), device=DEV)
    b = torch.empty((2, 8, 8, 32), device=DEV)
    lib.nchw_to_nhwc(u.data_ptr(), F32, 2048, a.data_ptr(), F32, 2, 128, 4, 4, st())
    lib.nchw_to_nhwc(u.data_ptr(), F32, 2048, b.data_ptr(), F32, 2, 32, 8, 8, st())
    assert torch.equal(a[:, :, :, 5].reshape(2, 16), b[:, 2:4, :, 1].reshape(2, 16))


def test_copy2d_and_pack():
    g = torch.Generator().manual_seed(4)
    s = torch.randn(10, 7, generator=g).to(DEV)
    d = torch.zeros(10, 20, device=DEV)
    lib.copy2d(s.data_ptr(), F32, 7, d.data_ptr() + 4 * 3, F32, 20, 10, 7, 0, st())
    assert torch.equal(d[:, 3:10], s)
    lib.copy2d(s.data_ptr(), F32, 7, d.data_ptr() + 4 * 3, F32, 20, 10, 7, 1, st())
    assert torch.equal(d[:, 3:10], 2 * s)
    lib.copy2d(s.data_ptr(), F32, 0, d.data_ptr(), F32, 20, 10, 7, 0, st())      # row broadcast
    assert torch.equal(d[:, :7], s[0:1].expand(10, 7))
    w = torch.randn(6, 5, 3, 3, generator=g).to(DEV)
    p01 = torch.empty(w.numel(), device=DEV); p10 = torch.empty(w.numel(), device=DEV)
    lib.pack_weights(w.data_ptr(), 6, 5, 9, p01.data_ptr(), p10.data_ptr(), F32, st())
    assert torch.equal(p01.view(9, 6, 5), w.reshape(6, 5, 9).permute(2, 0, 1).contiguous())
    assert torch.equal(p10.view(9, 5, 6), w.reshape(6, 5, 9).permute(2, 1, 0).contiguous())


def test_philox_matches_numpy_restatement_and_is_normal():
    from oracle import np_primitives as npp
    B, Wd, seed, sid, off = 3, 64, 0x1234_5678_9ABC, 5, 1000
    out = torch.empty(B, Wd, device=DEV)
    lib.philox_normal(out.data_ptr(), B, Wd, seed, sid, off, None, st())
    got = out.cpu().numpy().reshape(-1)
    for blk in (0, 1, 17, 47):
        ref = npp.philox_normal4(seed, sid, (off * Wd) // 4 + blk)
        np.testing.assert_allclose(got[4 * blk:4 * blk + 4], ref, rtol=0, atol=2e-5)
    stepbuf = torch.tensor([7], device=DEV, dtype=torch.int64)
    lib.philox_normal(out.data_ptr(), B, Wd, seed, sid, off, stepbuf.data_ptr(), st())
    ref = npp.philox_normal4(seed, sid, (off * Wd) // 4 + 3, step=7)
    np.testing.assert_allclose(out.cpu().numpy().reshape(-1)[12:16], ref, rtol=0, atol=2e-5)
    big = torch.empty(64, 16384, device=DEV)
    lib.philox_normal(big.data_ptr(), 64, 16384, 42, 0, 0, None, st())
    m, s = float(big.mean()), float(big.std())
    kurt = float(((big - m) ** 4).mean() / s ** 4)
    print(f"[parity] philox N(0,1): mean {m:.4e} std {s:.5f} kurtosis {kurt:.4f}")
    assert abs(m) < 5e-3 and abs(s - 1) < 5e-3 and abs(kurt - 3) < 0.05
    # partition invariance: rows [2,3) drawn alone equal row 2 of the full draw
    part = torch.empty(1, Wd, device=DEV)
    full = torch.empty(4, Wd, device=DEV)
    lib.philox_normal(full.data_ptr(), 4, Wd, 9, 1, 0, None, st())
    lib.philox_normal(part.data_ptr(), 1, Wd, 9, 1, 2, None, st())
    assert torch.equal(part[0], full[2])


def test_reparam_fwd_bwd():
    # ld_mult 2: z_ld = dz_ld = 2 Wd, z is the second half of the engine's torch.cat row; "nonzero": bwd accumulates, denc += ...
    for ld_mult in (1, 2):
        for denc0 in ("zero", "nonzero"):
            _reparam_case(ld_mult, denc0)


def _reparam_case(ld_mult, denc0):
    g = torch.Generator().manual_seed(8)
    B, Wd = 5, 256
    ld = ld_mult * Wd
    enc = torch.randn(B, 2 * Wd, generator=g)
    eps = torch.randn(B, Wd, generator=g)
    er = enc.double().requires_grad_(True)
    zr = er[:, :Wd] + eps.double() * torch.exp(0.5 * er[:, Wd:])
    gz = torch.randn(B, Wd, generator=g)
    zr.backward(gz.double())
    d0 = torch.zeros(B, 2 * Wd) if denc0 == "zero" else torch.randn(B, 2 * Wd, generator=g)
    gzbuf = torch.full((B, ld), float("nan"))      # columns past Wd must not be read
    gzbuf[:, :Wd] = gz
    encd, epsd, gzd = enc.to(DEV), eps.to(DEV), gzbuf.to(DEV)
    z = Guarded((B, ld), torch.float32)
    lib.reparam_fwd(encd.data_ptr(), epsd.data_ptr(), z.t.data_ptr(), ld, None, B, Wd, 0, 0, 0, None, st())
    report(f"reparam fwd [ld {ld}, denc {denc0}]", z.t[:, :Wd], zr, 1e-6)
    assert torch.isnan(z.t[:, Wd:]).all() and z.intact(), "reparam_fwd wrote outside the first Wd columns of its rows"
    denc = Guarded((B, 2 * Wd), torch.float32)
    denc.t.copy_(d0)
    lib.reparam_bwd(encd.data_ptr(), epsd.data_ptr(), gzd.data_ptr(), ld, denc.t.data_ptr(), B, Wd, 0, 0, 0, None, st())
    report(f"reparam bwd [ld {ld}, denc {denc0}]", denc.t, d0.double() + er.grad, 1e-6)
    assert denc.intact()
    # on-device noise with a step counter: eps_out replays exactly in backward and is svrs_philox_normal's draw
    step = torch.tensor([3], dtype=torch.int64, device=DEV)
    eo = torch.empty(B, Wd, device=DEV)
    lib.reparam_fwd(encd.data_ptr(), None, z.t.data_ptr(), ld, eo.data_ptr(), B, Wd, 77, 1, 3, step.data_ptr(), st())
    ref_eps = torch.empty(B, Wd, device=DEV)
    lib.philox_normal(ref_eps.data_ptr(), B, Wd, 77, 1, 3, step.data_ptr(), st())
    assert torch.equal(eo, ref_eps)
    d1 = torch.zeros(B, 2 * Wd, device=DEV); d2 = torch.zeros(B, 2 * Wd, device=DEV)
    lib.reparam_bwd(encd.data_ptr(), None, gzd.data_ptr(), ld, d1.data_ptr(), B, Wd, 77, 1, 3, step.data_ptr(), st())
    lib.reparam_bwd(encd.data_ptr(), eo.data_ptr(), gzd.data_ptr(), ld, d2.data_ptr(), B, Wd, 77, 1, 3, step.data_ptr(), st())
    assert torch.equal(d1, d2)
    eo4 = torch.empty(B, Wd, device=DEV)
    step4 = torch.tensor([4], dtype=torch.int64, device=DEV)
    lib.reparam_fwd(encd.data_ptr(), None, z.t.data_ptr(), ld, eo4.data_ptr(), B, Wd, 77, 1, 3, step4.data_ptr(), st())
    assert float((eo4 == eo).double().mean()) < 1e-3, "another step gave the same noise"
    # partition invariance: rows [2, 5) drawn alone at sample_offset 3 + 2 equal rows 2..4 of the full draw
    zp = Guarded((3, ld), torch.float32)
    ep = torch.empty(3, Wd, device=DEV)
    lib.reparam_fwd(encd.data_ptr() + 4 * 2 * 2 * Wd, None, zp.t.data_ptr(), ld, ep.data_ptr(), 3, Wd, 77, 1, 3 + 2, step.data_ptr(), st())
    lib.reparam_fwd(encd.data_ptr(), None, z.t.data_ptr(), ld, eo.data_ptr(), B, Wd, 77, 1, 3, step.data_ptr(), st())
    assert torch.equal(ep, eo[2:]) and torch.equal(zp.t[:, :Wd], z.t[2:, :Wd]) and zp.intact()
    # B = 0 enqueues nothing
    torch.cuda.synchronize()
    n0, before = lib.launch_count(), denc.t.clone()
    lib.reparam_fwd(encd.data_ptr(), None, z.t.data_ptr(), ld, None, 0, Wd, 77, 1, 3, step.data_ptr(), st())
    lib.reparam_bwd(encd.data_ptr(), None, gzd.data_ptr(), ld, denc.t.data_ptr(), 0, Wd, 77, 1, 3, step.data_ptr(), st())
    assert lib.launch_count() == n0 and torch.equal(denc.t, before)


def test_elbo_against_golden_vectors(golden_dir):
    """loss callables vs vectors minted from the reference's loss/ package (tests/golden/loss_vectors.pt)."""
    import os
    from loss import base_loss, cond_loss
    fx = torch.load(os.path.join(golden_dir, "loss_vectors.pt"))
    t = {k: v.to(DEV) for k, v in fx["inputs"].items()}
    leaves = {k: v.clone().requires_grad_(True) for k, v in t.items() if k not in ("x", "y")}
    gx = torch.tensor(fx["gammax"], requires_grad=True)
    gy = torch.tensor(fx["gammay"], requires_grad=True)
    terms = cond_loss(leaves["recon_x"], t["x"], leaves["recon_y"], t["y"], leaves["mu1"], leaves["lv1"], leaves["mu2"],
                      leaves["lv2"], leaves["mu3"], leaves["lv3"], gx, gy)
    for name, got, ref in zip(("mse_x", "kld_u", "mse_y", "kld_z"), terms, fx["terms"]):
        report(f"cond_loss {name}", got.reshape(1), torch.tensor([ref]), 1e-6)
    sum(terms).backward()
    for k, ref in fx["grads"].items():
        report(f"cond_loss d{k}", leaves[k].grad, ref, 1e-5)
    report("cond_loss dgammax", gx.grad.reshape(1), torch.tensor([fx["grad_gammax"]]), 1e-5)
    report("cond_loss dgammay", gy.grad.reshape(1), torch.tensor([fx["grad_gammay"]]), 1e-5)
    # chunk views (non-contiguous, row stride 2W) like the model's outputs
    enc = torch.cat((t["mu2"], t["lv2"]), dim=1)
    mu2v, lv2v = enc.chunk(2, dim=1)
    terms_v = cond_loss(t["recon_x"], t["x"], t["recon_y"], t["y"], t["mu1"], t["lv1"], mu2v, lv2v, t["mu3"], t["lv3"],
                        torch.tensor(fx["gammax"]), torch.tensor(fx["gammay"]))
    report("cond_loss kld_z on chunk views", terms_v[3].reshape(1), torch.tensor([fx["terms"][3]]), 1e-6)
    b = fx["base"]
    l2 = {k: t[k].clone().requires_grad_(True) for k in ("recon_x", "mu2", "lv2")}
    g1 = torch.tensor(b["gamma"], requires_grad=True)
    mse, kld = base_loss(l2["recon_x"], t["x"], l2["mu2"], l2["lv2"], g1)
    # d*(ssq/(2 g^2 d) + log g) with g < 1 cancels two ~3e2 numbers down to ~0.2: compare against that magnitude
    report("base_loss mse", mse.reshape(1), torch.tensor([b["terms"][0]]), 1e-6, atol=3e-7 * t["recon_x"].numel() * 0.106)
    report("base_loss kld", kld.reshape(1), torch.tensor([b["terms"][1]]), 1e-6)
    (mse + kld).backward()
    for k, ref in b["grads"].items():
        report(f"base_loss d{k}", l2[k].grad, ref, 1e-5)
    report("base_loss dgamma", g1.grad.reshape(1), torch.tensor([b["grad_gamma"]]), 1e-5)


def test_clip_adam_matches_torch():
    g = torch.Generator().manual_seed(6)
    n = 10007
    p0 = torch.randn(n, generator=g)
    ref = p0.clone().requires_grad_(True)
    opt = torch.optim.Adam([ref], lr=1e-4)
    p, m, v = p0.to(DEV), torch.zeros(n, device=DEV), torch.zeros(n, device=DEV)
    step = torch.zeros(1, device=DEV, dtype=torch.int64)
    acc = torch.zeros(1, device=DEV, dtype=torch.float64)
    for it in range(5):
        grad = torch.randn(n, generator=g) * (10.0 if it % 2 == 0 else 0.001)   # clipped and unclipped steps
        ref.grad = grad.clone()
        total = torch.nn.utils.clip_grad_norm_([ref], 1.0)
        opt.step()
        gd = grad.to(DEV)
        lib.step_increment(step.data_ptr(), st())
        lib.fill_zero(acc.data_ptr(), 8, st())
        lib.sumsq(gd.data_ptr(), n, acc.data_ptr(), st())
        lib.clip_adam(p.data_ptr(), gd.data_ptr(), m.data_ptr(), v.data_ptr(), n, acc.data_ptr(), 1.0, 1.0, 1e-4, 0.9, 0.999,
                      1e-8, step.data_ptr(), st())
        report(f"grad norm step {it}", acc.sqrt().float(), total.reshape(1), 1e-6)
        report(f"adam params step {it}", p, ref.detach(), 1e-6)
    assert int(step) == 5


def test_grid_patch_bit_exact(golden_dir):
    """Grid patching + normalisation: BIT-exact vs vectors minted from the reference's dataset.py / utils.py."""
    import os
    from dataset import grid_batch, grid_patch_normalize
    fx = torch.load(os.path.join(golden_dir, "grid_vectors.pt"))
    hr, lr = fx["hr"].to(DEV), fx["lr"].to(DEV)
    y, x = grid_batch(lr.float(), hr.float(), 64)
    assert torch.equal(y.cpu(), fx["y"]), "LR patches differ from the reference"
    assert torch.equal(x.cpu(), fx["x"]), "HR patches differ from the reference"
    y16, x16 = grid_batch(lr, hr, 64)                     # int16 source (the TIFF dtype, dataset.py:154-155)
    assert torch.equal(y16.cpu(), fx["y"]) and torch.equal(x16.cpu(), fx["x"])
    xn = grid_patch_normalize(hr, 64, torch.bfloat16, nhwc=True)
    assert torch.equal(xn.cpu(), fx["x"].permute(0, 2, 3, 1).contiguous().to(torch.bfloat16))
    # edge: single patch == whole tile (utils.normalize_image 3-D path)
    from utils import normalize_image
    one = normalize_image(hr[0].float())
    mn = hr[0].float().amin(dim=(1, 2), keepdim=True); mx = hr[0].float().amax(dim=(1, 2), keepdim=True)
    assert torch.equal(one, (hr[0].float() - mn) / (mx - mn + 1e-5))


def test_error_reporting_is_loud():
    from svrs_native.lib import SvrsError
    x = torch.zeros(4, device=DEV)
    with pytest.raises(SvrsError):
        lib.conv2d_fprop(x.data_ptr(), x.data_ptr(), None, None, x.data_ptr(), 7, 1, 2, 2, 1, 1, 3, 0, st())   # bad dtype
    with pytest.raises(SvrsError):
        lib.conv2d_fprop(x.data_ptr(), x.data_ptr(), None, None, x.data_ptr(), F32, 1, 3, 3, 1, 1, 4, 0, st())  # odd H with k4s2
    assert "conv2d_fprop" in lib.last_error()


TC_CASES = [
    # N, H, W, Cin, Cout   (bf16, reduction channels % 64 == 0 -> tcgen05 kernel)
    (2, 8, 8, 64, 64),
    (3, 16, 16, 128, 64),     # N not a multiple of the images-per-tile
    (2, 4, 4, 256, 512),      # two N tiles of 256, 8 images per 128-pixel tile, N < box
    (1, 64, 64, 64, 16),      # decoder tail 64 -> 16 at 64x64 (N tile 16)
    (2, 32, 32, 128, 128),
    (9, 4, 4, 64, 48),        # N tile 48 = 32 + 16 column loads, 9 images over two tiles
    (2, 16, 16, 16, 16),      # 16-channel chunks: SWIZZLE_32B operands, 4 (tap, chunk) pairs per stage
    (1, 64, 64, 16, 4),       # last decoder conv: N padded 4 -> 16 for the MMA, masked scalar stores
    (2, 8, 8, 32, 128),       # 32-channel chunks: SWIZZLE_64B
    (3, 8, 8, 48, 16),        # 3 chunks of 16 channels
    (2, 32, 32, 64, 16),      # decoder tail 64 -> 16
]


@pytest.mark.parametrize("case", TC_CASES)
def test_conv_tc_all_forms(case):
    """tcgen05/TMA kernel (conv_tc) for every conv form vs float64 torch, and vs the SIMT kernel on the same inputs."""
    N, H, W, Cin, Cout = case
    dtype = torch.bfloat16
    g = torch.Generator().manual_seed(sum(case))
    x = _rand((N, Cin, H, W), g, dtype)
    b = torch.randn(Cout, generator=g)
    for form in ("c3", "c4", "ct"):
        ks = 3 if form == "c3" else 4
        if form == "ct":
            w = (_rand((Cin, Cout, 4, 4), g, dtype) * 0.1).to(dtype).float()
            fwd = lambda xx, ww, bb: F.conv_transpose2d(xx, ww, bb, stride=2, padding=1)
        else:
            w = (_rand((Cout, Cin, ks, ks), g, dtype) * 0.1).to(dtype).float()
            fwd = (lambda xx, ww, bb: F.conv2d(xx, ww, bb, stride=1, padding=1)) if form == "c3" else \
                  (lambda xx, ww, bb: F.conv2d(xx, ww, bb, stride=2, padding=1))
        xr = x.double().requires_grad_(True)
        yr = fwd(xr, w.double(), b.double())
        gy = _rand(tuple(yr.shape), g, dtype)
        yr.backward(gy.double())
        xd, wd, bd, gyd = nhwc(x.to(DEV), dtype), w.to(DEV), b.to(DEV), nhwc(gy.to(DEV), dtype)
        pf, pb = pack(wd, dtype, convT=(form == "ct"))
        OH, OW = yr.shape[2], yr.shape[3]
        res = {}
        for tc in (1, 0):
            lib.set_tc_enabled(tc)
            y = torch.full((N, OH, OW, Cout), float("nan"), device=DEV, dtype=dtype)
            dx = torch.full_like(xd, float("nan"))
            if form == "ct":
                lib.convT2d_fprop(xd.data_ptr(), pf.data_ptr(), pb.data_ptr(), bd.data_ptr(), y.data_ptr(), BF16, N, H, W, Cin, Cout, 0, st())
                lib.convT2d_dgrad(gyd.data_ptr(), pb.data_ptr(), pf.data_ptr(), dx.data_ptr(), BF16, N, H, W, Cin, Cout, st())
            else:
                lib.conv2d_fprop(xd.data_ptr(), pf.data_ptr(), pb.data_ptr(), bd.data_ptr(), y.data_ptr(), BF16, N, H, W, Cin, Cout, ks, 0, st())
                lib.conv2d_dgrad(gyd.data_ptr(), pb.data_ptr(), pf.data_ptr(), dx.data_ptr(), BF16, N, H, W, Cin, Cout, ks, st())
            torch.cuda.synchronize()
            res[tc] = (y, dx)
        lib.set_tc_enabled(1)
        ran_f = lib.tc_would_run(BF16, Cin, Cout, OH if form != "ct" else H, OW if form != "ct" else W)
        print(f"[parity] {form} {case}: conv_tc taken for fprop: {bool(ran_f)}")
        report(f"conv_tc {form} fprop {case} vs fp64", nchw(res[1][0]), yr, 7e-3)
        report(f"conv_tc {form} dgrad {case} vs fp64", nchw(res[1][1]), xr.grad, 7e-3)
        report(f"conv_tc {form} fprop {case} vs simt", res[1][0].float(), res[0][0].float(), 8e-3)
        report(f"conv_tc {form} dgrad {case} vs simt", res[1][1].float(), res[0][1].float(), 8e-3)


@pytest.mark.parametrize("case", [(2, 8, 8, 64, 64), (3, 16, 16, 128, 64), (2, 4, 4, 256, 512), (2, 32, 32, 128, 128),
                                  (5, 8, 8, 64, 192), (2, 16, 16, 16, 16), (2, 32, 32, 64, 16), (2, 8, 8, 32, 128),
                                  (3, 8, 8, 48, 32), (2, 16, 16, 16, 64), (1, 64, 64, 64, 64), (3, 16, 8, 128, 64),
                                  (2, 32, 16, 64, 256)])
def test_wgrad_tc_all_forms(case):
    """tcgen05 weight-gradient kernel (MN-major operands, split-K over pixels) vs float64 torch autograd."""
    N, H, W, Cin, Cout = case
    dtype = torch.bfloat16
    g = torch.Generator().manual_seed(sum(case) + 1)
    x = _rand((N, Cin, H, W), g, dtype)
    for form in ("c3", "c4", "ct"):
        ks = 3 if form == "c3" else 4
        if form == "ct":
            w = (_rand((Cin, Cout, 4, 4), g, dtype) * 0.1).to(dtype).float()
            fwd = lambda xx, ww: F.conv_transpose2d(xx, ww, None, stride=2, padding=1)
        else:
            w = (_rand((Cout, Cin, ks, ks), g, dtype) * 0.1).to(dtype).float()
            fwd = (lambda xx, ww: F.conv2d(xx, ww, None, stride=1, padding=1)) if form == "c3" else \
                  (lambda xx, ww: F.conv2d(xx, ww, None, stride=2, padding=1))
        wr = w.double().requires_grad_(True)
        yr = fwd(x.double(), wr)
        gy = _rand(tuple(yr.shape), g, dtype)
        yr.backward(gy.double())
        xd, gyd = nhwc(x.to(DEV), dtype), nhwc(gy.to(DEV), dtype)
        res = {}
        for tc in (1, 0):
            lib.set_tc_enabled(tc)
            dw = torch.zeros(w.shape, device=DEV)
            db = torch.zeros(Cout, device=DEV)
            if form == "ct":
                lib.convT2d_wgrad(xd.data_ptr(), gyd.data_ptr(), dw.data_ptr(), None, db.data_ptr(), BF16, N, H, W, Cin, Cout, 0, st())
            else:
                lib.conv2d_wgrad(xd.data_ptr(), gyd.data_ptr(), dw.data_ptr(), None, db.data_ptr(), BF16, N, H, W, Cin, Cout, ks, 0, st())
            torch.cuda.synchronize()
            res[tc] = dw
            # bias gradient = column sums of dy (folded into the tensor-core kernels' idle epilogue warps for conv forms)
            report(f"wgrad_tc {form} {case} db (tc={tc})", db, gy.double().sum(dim=(0, 2, 3)), 2e-5)
        lib.set_tc_enabled(1)
        report(f"wgrad_tc {form} {case} vs fp64", res[1], wr.grad, 2e-5)
        report(f"wgrad_tc {form} {case} vs simt", res[1], res[0], 2e-5)


def test_pack_weights_multi_matches_single():
    """The one-launch, shared-memory-tiled pack of all layers equals the simple per-layer pack (both dtypes, conv + convT)."""
    import models
    from svrs_native.engine import ConvOp
    for dtype in (torch.float32, torch.bfloat16):
        m = models.VAE(2, 32).to(DEV)
        m.set_compute_dtype(dtype)
        eng = m._engine()
        eng.rt.ensure()
        eng.rt.pack_weights(force=True)
        torch.cuda.synchronize()
        n = 0
        for net in eng.nets.values():
            for op in net.ops:
                if not isinstance(op, ConvOp):
                    continue
                pf, pb = pack(op.mod.weight.data, dtype, convT=(op.kind == "ct"))
                assert torch.equal(op.pack_f, pf) and torch.equal(op.pack_b, pb), (net.name, op.kind, op.cin, op.cout)
                n += 1
        assert n == 16


HALO_CASES = [(2, 16, 16, 64, 64), (1, 32, 32, 128, 128), (2, 16, 8, 64, 256), (1, 64, 64, 64, 16), (3, 16, 16, 128, 64),
              (2, 32, 16, 256, 64),
              (2, 16, 16, 16, 16), (1, 64, 64, 16, 64), (2, 32, 16, 32, 32), (3, 16, 24, 32, 16)]   # 16/32-channel chunks (32B/64B swizzle)


@pytest.mark.parametrize("case", HALO_CASES)
def test_conv3_halo_kernel(case):
    """Halo-reuse kernel (one TMA load of the activation halo per tile, nine descriptor views) vs fp64 and vs the per-tap kernel."""
    N, H, W, Cin, Cout = case
    dtype = torch.bfloat16
    g = torch.Generator().manual_seed(sum(case) + 7)
    x = _rand((N, Cin, H, W), g, dtype)
    w = (_rand((Cout, Cin, 3, 3), g, dtype) * 0.1).to(dtype).float()
    b = torch.randn(Cout, generator=g)
    xr = x.double().requires_grad_(True)
    yr = F.conv2d(xr, w.double(), b.double(), stride=1, padding=1)
    gy = _rand(tuple(yr.shape), g, dtype)
    yr.backward(gy.double())
    xd, wd, bd, gyd = nhwc(x.to(DEV), dtype), w.to(DEV), b.to(DEV), nhwc(gy.to(DEV), dtype)
    pf, pb = pack(wd, dtype)
    errs = {}
    try:
        for mode in (0, 1):
            lib.set_halo_mode(mode)
            y = torch.full((N, H, W, Cout), float("nan"), device=DEV, dtype=dtype)
            dx = torch.full_like(xd, float("nan"))
            lib.conv2d_fprop(xd.data_ptr(), pf.data_ptr(), pb.data_ptr(), bd.data_ptr(), y.data_ptr(), BF16, N, H, W, Cin, Cout, 3, 0, st())
            lib.conv2d_dgrad(gyd.data_ptr(), pb.data_ptr(), pf.data_ptr(), dx.data_ptr(), BF16, N, H, W, Cin, Cout, 3, st())
            torch.cuda.synchronize()
            ef = float((nchw(y).double().cpu() - yr.detach()).abs().max() / yr.detach().abs().max())
            ed = float((nchw(dx).double().cpu() - xr.grad).abs().max() / xr.grad.abs().max())
            errs[mode] = (ef, ed)
            print(f"[parity] conv3 halo mode {mode} {case}: fprop rel err {ef:.3e}, dgrad rel err {ed:.3e}")
    finally:
        lib.set_halo_mode(1)
    assert max(errs[0]) < 7e-3, "per-tap kernel"
    assert max(errs[1]) < 7e-3, f"halo kernel: {errs}"


@pytest.mark.parametrize("case", [(2, 16, 16, 64, 64, "c3"), (2, 8, 8, 64, 128, "c4"), (3, 8, 8, 128, 64, "ct"), (2, 16, 16, 16, 32, "c3")])
def test_wgrad_packed_scratch_and_unpack(case):
    """tcgen05 wgrad into the per-tap packed scratch + one-launch unpack == wgrad straight into the torch layout."""
    import numpy as np
    N, H, W, Cin, Cout, form = case
    dtype = torch.bfloat16
    g = torch.Generator().manual_seed(sum(case[:5]))
    x = nhwc(_rand((N, Cin, H, W), g, dtype).to(DEV), dtype)
    ks = 3 if form == "c3" else 4
    if form == "ct":
        wshape, gyshape = (Cin, Cout, 4, 4), (N, 2 * H, 2 * W, Cout)
    else:
        s = 1 if form == "c3" else 2
        wshape, gyshape = (Cout, Cin, ks, ks), (N, H // s, W // s, Cout)
    gy = torch.randn(gyshape, generator=g).to(DEV).to(dtype)
    ref = torch.zeros(wshape, device=DEV)
    out = torch.zeros(wshape, device=DEV)
    scratch = torch.zeros(wshape, device=DEV)
    if form == "ct":
        lib.convT2d_wgrad(x.data_ptr(), gy.data_ptr(), ref.data_ptr(), None, None, BF16, N, H, W, Cin, Cout, 0, st())
        lib.convT2d_wgrad(x.data_ptr(), gy.data_ptr(), out.data_ptr(), scratch.data_ptr(), None, BF16, N, H, W, Cin, Cout, 0, st())
    else:
        lib.conv2d_wgrad(x.data_ptr(), gy.data_ptr(), ref.data_ptr(), None, None, BF16, N, H, W, Cin, Cout, ks, 0, st())
        lib.conv2d_wgrad(x.data_ptr(), gy.data_ptr(), out.data_ptr(), scratch.data_ptr(), None, BF16, N, H, W, Cin, Cout, ks, 0, st())
    rec = np.dtype([("w", "<u8"), ("p01", "<u8"), ("p10", "<u8"), ("d0", "<i4"), ("d1", "<i4"), ("kk", "<i4"),
                    ("tile0", "<i4"), ("tiles_b", "<i4"), ("pad", "<i4")])
    assert rec.itemsize == lib.pack_job_bytes()
    d0, d1, kk = wshape[0], wshape[1], wshape[2] * wshape[3]
    jobs = np.zeros(1, dtype=rec)
    jobs[0] = (out.data_ptr(), scratch.data_ptr(), 0, d0, d1, kk, 0, (d1 + 15) // 16, 0)
    jd = torch.from_numpy(jobs.view(np.uint8).copy()).to(DEV)
    lib.unpack_grads_multi(jd.data_ptr(), 1, ((d0 + 31) // 32) * ((d1 + 15) // 16), 16, st())
    torch.cuda.synchronize()
    assert float(scratch.abs().max()) > 0, "tensor-core wgrad did not use the packed scratch"
    report(f"packed wgrad + unpack {case}", out, ref, 2e-5)
