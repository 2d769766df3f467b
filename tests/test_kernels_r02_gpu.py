"""Kernel-level parity (-m gpu) of the round-2 C-ABI entry points: the TMA patch gather (grid mode and the reference's
random crop), the conv epilogue extras of svrs_conv2d_fprop_ex / svrs_convT2d_fprop_ex (BatchNorm statistics, fp32
NCHW-flat head output, fp32 store), the one-launch optimiser tail svrs_adam_multi, and the streaming uncertainty
statistics of the sample path.  Same conventions as test_kernels_gpu.py: float64 CPU evaluation of the torch op the
reference calls at that site is the truth; inputs are pre-rounded to bf16 so only accumulation order / output rounding
differ."""
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from helpers import BF16, F32, Guarded, dt, lib, nchw, nhwc, pack, report, st, task_stats
from oracle import ref_oracle as O
from svrs_native.lib import SvrsUnsupported

pytestmark = pytest.mark.gpu
DEV = "cuda"
R = 8   # SVRS_BN_REPLICAS


def _rand(shape, gen, dtype=torch.bfloat16):
    t = torch.randn(shape, generator=gen)
    return t.to(dtype).float() if dtype == torch.bfloat16 else t


# ------------------------------------------------------------------------------------------------ patch gather (a13, f3)
def _gather(tiles, P, origins, npatch, want_bf16=True):
    T, C, S, _ = tiles.shape
    o_nchw = torch.full((npatch, C, P, P), float("nan"), device=DEV)
    o_nhwc = torch.full((npatch, P, P, C), float("nan"), device=DEV)
    o_bf = torch.zeros((npatch, P, P, C), device=DEV, dtype=torch.bfloat16) if want_bf16 else None
    lib.patch_gather_normalize(tiles.data_ptr(), int(tiles.dtype == torch.int16), T, C, S, P,
                               None if origins is None else origins.data_ptr(), npatch, o_nchw.data_ptr(), o_nhwc.data_ptr(),
                               None if o_bf is None else o_bf.data_ptr(), st())
    torch.cuda.synchronize()
    return o_nchw, o_nhwc, o_bf


def test_patch_gather_grid_mode_bit_exact(golden_dir):
    """svrs_patch_gather_normalize, grid mode: BIT-exact vs the vectors minted from the reference's dataset.py / utils.py,
    fp32 and int16 sources, all three output layouts."""
    fx = torch.load(os.path.join(golden_dir, "grid_vectors.pt"))
    for src in (fx["hr"].to(DEV), fx["hr"].to(DEV).float()):
        a, b, c = _gather(src.contiguous(), 64, None, fx["x"].shape[0])
        assert torch.equal(a.cpu(), fx["x"])
        assert torch.equal(b.cpu(), fx["x"].permute(0, 2, 3, 1).contiguous())
        assert torch.equal(c.cpu(), fx["x"].permute(0, 2, 3, 1).contiguous().to(torch.bfloat16))
    a, b, _ = _gather(fx["lr"].to(DEV).contiguous(), 32, None, fx["y"].shape[0])
    assert torch.equal(a.cpu(), fx["y"]) and torch.equal(b.cpu(), fx["y"].permute(0, 2, 3, 1).contiguous())


@pytest.mark.parametrize("as_int16", [False, True])
def test_random_crop_same_origin_bit_exact(as_int16):
    """f3: the reference's random crop (dataset.py:205-216): LR patch at (top, left), HR patch at (2*top, 2*left), each
    min-max normalised per channel (utils.py:4-23, 3-D path).  Origins are injected so the index arithmetic is checked bit
    for bit, including the corner origins and unaligned (odd) offsets."""
    from dataset import random_crop_batch, random_crop_origins, synthetic_tiles
    normalize_image = O.normalize_image            # utils.py:4-23 restated on the CPU (oracle)
    T, S, P = 6, 256, 64
    lr, hr = synthetic_tiles(T, S, seed=5, as_int16=as_int16)
    g = torch.Generator().manual_seed(9)
    o = random_crop_origins(T, S // 2, P, g)
    mx = S // 2 - P // 2 - 1
    extra = torch.tensor([[0, 0, 0], [1, mx, mx], [2, 0, mx], [3, mx, 0], [4, 1, 3], [5, 17, 33], [0, 5, 64]], dtype=torch.int32)
    o = torch.cat([o, extra])
    assert int(o[:, 1:].max()) <= mx          # randint(0, lr_size - half) never reaches the last origin (dataset.py:207-208)
    (y_nchw, yb), (x_nchw, xb) = random_crop_batch(lr.to(DEV), hr.to(DEV), P, o, torch.bfloat16)
    torch.cuda.synchronize()
    for i, (t, top, left) in enumerate(o.tolist()):
        ry = normalize_image(lr[t].float()[:, top:top + P // 2, left:left + P // 2])
        rx = normalize_image(hr[t].float()[:, 2 * top:2 * top + P, 2 * left:2 * left + P])
        assert torch.equal(y_nchw[i].cpu(), ry), (i, t, top, left)
        assert torch.equal(x_nchw[i].cpu(), rx), (i, t, top, left)
        assert torch.equal(xb.f32[i].cpu(), rx.permute(1, 2, 0)) and torch.equal(yb.f32[i].cpu(), ry.permute(1, 2, 0))
        assert torch.equal(xb.op[i].cpu(), rx.permute(1, 2, 0).to(torch.bfloat16))


def test_patch_gather_rejects_bad_arguments():
    from svrs_native.lib import SvrsError
    t = torch.zeros(1, 4, 64, 64, device=DEV)
    out = torch.zeros(1, 4, 6, 6, device=DEV)
    with pytest.raises(SvrsError):      # P*4 bytes not a multiple of 16
        lib.patch_gather_normalize(t.data_ptr(), 0, 1, 4, 64, 6, None, 1, out.data_ptr(), None, None, st())


# ------------------------------------------------------------------------------------------------ conv epilogue extras
EX_CASES = [
    # N, H, W, Cin, Cout, ksize, kernel expected
    (4, 8, 8, 128, 64, 3),      # encoder head at 8x8 (conv_tc)
    (3, 4, 4, 256, 512, 3),     # prior head at 4x4, two N tiles
    (2, 16, 16, 64, 128, 4),    # down_block conv4s2 -> BatchNorm (conv_tc)
    (2, 16, 16, 128, 128, 3),   # halo kernel
    (2, 32, 32, 16, 64, 4),     # 16-channel chunks
    (2, 32, 32, 4, 16, 4),      # image-side down_block conv4s2 -> BatchNorm (narrow mma.sync kernel)
    (3, 16, 16, 4, 16, 4),
]


@pytest.mark.parametrize("case", EX_CASES)
def test_conv_fprop_ex_head_and_bn_sums(case):
    N, H, W, Cin, Cout, ks = case
    g = torch.Generator().manual_seed(sum(case))
    x = _rand((N, Cin, H, W), g)
    w = (_rand((Cout, Cin, ks, ks), g) * 0.1).to(torch.bfloat16).float()
    b = torch.randn(Cout, generator=g)
    stride = 1 if ks == 3 else 2
    yr = F.conv2d(x.double(), w.double(), b.double(), stride=stride, padding=1)
    OH, OW = yr.shape[2:]
    xd, wd, bd = nhwc(x.to(DEV), torch.bfloat16), w.to(DEV), b.to(DEV)
    pf, pb = pack(wd, torch.bfloat16)
    # (a) BatchNorm statistics from the fp32 accumulators
    y = torch.full((N, OH, OW, Cout), float("nan"), device=DEV, dtype=torch.bfloat16)
    sums = torch.zeros(R * 2 * Cout, device=DEV, dtype=torch.float64)
    try:
        lib.conv2d_fprop_ex(xd.data_ptr(), pf.data_ptr(), pb.data_ptr(), bd.data_ptr(), y.data_ptr(), BF16, BF16, None, 0,
                            sums.data_ptr(), N, H, W, Cin, Cout, ks, 0, st())
        torch.cuda.synchronize()
        s = sums.view(R, 2, Cout).sum(0).cpu()
        report(f"fprop_ex {case} y", nchw(y), yr, 7e-3)
        report(f"fprop_ex {case} bn sum", s[0], yr.sum(dim=(0, 2, 3)), 1e-5, atol=1e-3)
        report(f"fprop_ex {case} bn sumsq", s[1], (yr * yr).sum(dim=(0, 2, 3)), 1e-5)
    except SvrsUnsupported as ex:
        print(f"[parity] fprop_ex {case}: BatchNorm statistics not offered by this layer's kernel ({ex})")
    # (b) fp32 NCHW-flat head output (row stride > row length: the chunk / cat buffers of the engine), no NHWC output
    if ks == 3:
        ld = Cout * OH * OW + 12
        head = torch.full((N, ld), float("nan"), device=DEV)
        lib.conv2d_fprop_ex(xd.data_ptr(), pf.data_ptr(), pb.data_ptr(), bd.data_ptr(), None, BF16, BF16, head.data_ptr(), ld,
                            None, N, H, W, Cin, Cout, ks, 0, st())
        torch.cuda.synchronize()
        got = head[:, :Cout * OH * OW].reshape(N, Cout, OH, OW)
        report(f"fprop_ex {case} fp32 NCHW-flat head", got, yr, 1e-5)       # fp32 accumulators, never rounded to bf16
        assert torch.isnan(head[:, Cout * OH * OW:]).all()                  # padding of the rows untouched
        # Hardtanh(-7, 7) head (logvar_u_y_to_z, cond_vae.py:230)
        big = (b * 20).to(DEV)
        lib.conv2d_fprop_ex(xd.data_ptr(), pf.data_ptr(), pb.data_ptr(), big.data_ptr(), None, BF16, BF16, head.data_ptr(), ld,
                            None, N, H, W, Cin, Cout, ks, 2, st())
        torch.cuda.synchronize()
        yh = F.hardtanh(F.conv2d(x.double(), w.double(), (b * 20).double(), stride=1, padding=1), -7.0, 7.0)
        report(f"fprop_ex {case} hardtanh head", head[:, :Cout * OH * OW].reshape(N, Cout, OH, OW), yh, 1e-5)


@pytest.mark.parametrize("case", [(2, 8, 8, 256, 256), (2, 16, 16, 128, 64), (3, 8, 8, 32, 128), (1, 32, 32, 128, 64)])
def test_convT_fprop_ex_bn_sums(case):
    N, H, W, Cin, Cout = case
    g = torch.Generator().manual_seed(sum(case) + 3)
    x = _rand((N, Cin, H, W), g)
    w = (_rand((Cin, Cout, 4, 4), g) * 0.1).to(torch.bfloat16).float()
    b = torch.randn(Cout, generator=g)
    yr = F.conv_transpose2d(x.double(), w.double(), b.double(), stride=2, padding=1)
    xd, wd, bd = nhwc(x.to(DEV), torch.bfloat16), w.to(DEV), b.to(DEV)
    pf, pb = pack(wd, torch.bfloat16, convT=True)
    y = torch.full((N, 2 * H, 2 * W, Cout), float("nan"), device=DEV, dtype=torch.bfloat16)
    sums = torch.zeros(R * 2 * Cout, device=DEV, dtype=torch.float64)
    lib.convT2d_fprop_ex(xd.data_ptr(), pf.data_ptr(), pb.data_ptr(), bd.data_ptr(), y.data_ptr(), BF16, sums.data_ptr(),
                         N, H, W, Cin, Cout, 0, st())
    torch.cuda.synchronize()
    s = sums.view(R, 2, Cout).sum(0).cpu()
    report(f"convT fprop_ex {case} y", nchw(y), yr, 7e-3)
    report(f"convT fprop_ex {case} bn sum", s[0], yr.sum(dim=(0, 2, 3)), 1e-5, atol=1e-3)
    report(f"convT fprop_ex {case} bn sumsq", s[1], (yr * yr).sum(dim=(0, 2, 3)), 1e-5)


def test_conv_pixel_fp32_sigmoid_tail():
    """16 -> 4 + Sigmoid tail of both decoders (cond_vae.py:79-80,142-143): bf16 operands, fp32 store."""
    N, H, W, Cin, Cout = 2, 32, 32, 16, 4
    g = torch.Generator().manual_seed(4)
    x = _rand((N, Cin, H, W), g)
    w = (_rand((Cout, Cin, 3, 3), g) * 0.2).to(torch.bfloat16).float()
    b = torch.randn(Cout, generator=g)
    yr = torch.sigmoid(F.conv2d(x.double(), w.double(), b.double(), padding=1))
    xd, wd, bd = nhwc(x.to(DEV), torch.bfloat16), w.to(DEV), b.to(DEV)
    pf, pb = pack(wd, torch.bfloat16)
    y = torch.full((N, H, W, Cout), float("nan"), device=DEV)
    lib.conv2d_fprop_ex(xd.data_ptr(), pf.data_ptr(), pb.data_ptr(), bd.data_ptr(), y.data_ptr(), BF16, F32, None, 0, None,
                        N, H, W, Cin, Cout, 3, 1, st())
    torch.cuda.synchronize()
    report("conv_pixel bf16 -> fp32 sigmoid", nchw(y), yr, 2e-6)


# ------------------------------------------------------------------------------------------------ one-launch optimiser tail
def test_fused_tail_equals_separate_kernels(golden_dir):
    """svrs_adam_multi (gradient read in the wgrad kernels' packed layout + clip + Adam + weight packs in one launch) against
    the round-1 chain (unpack_grads_multi -> sumsq -> clip_adam -> pack_weights_multi) on the same bf16 step: identical
    losses over 3 steps and identical parameters (the two chains do the same fp32 arithmetic per element)."""
    import fixtures as FX
    from svrs_native.trainer import FusedCondTrainer
    fx = FX.load(golden_dir, "cond_cr2_p64_b2")
    x, y = FX.inputs(fx)
    x, y = x.to(DEV), y.to(DEV)
    eng_w = FX.build(fx, device=DEV)[0]._engine()
    r = O.PortableRng(31)
    eps = [(r.randn(2, eng_w.Wu).to(DEV), r.randn(2, eng_w.Wz).to(DEV)) for _ in range(3)]
    res, flats = [], []
    for fused in (True, False):
        model, _ = FX.build(fx, device=DEV, dtype=torch.bfloat16)
        model.train()
        tr = FusedCondTrainer(model)
        tr.fused_tail = fused
        out = [tr.step(x, y, *eps[0]).clone()]
        flats.append(tr.rt.store.flat.clone())          # parameters after the FIRST step
        out += [tr.step(x, y, eu, ez).clone() for eu, ez in eps[1:]]
        res.append(torch.stack(out).cpu())
    report("fused tail vs separate kernels: ELBO terms over 3 steps", res[0], res[1], 1e-4)
    # After one step the two chains have applied Adam to the same gradient (identical wgrad kernels; only the order of the
    # fp32 atomics differs between ANY two runs).  Adam's first step is sign-like (lr * g / (|g| + eps)), so parameters can
    # only differ where a gradient is at rounding-noise level and flips sign: a vanishing fraction, by at most 2 * lr.
    d = (flats[0] - flats[1]).abs()
    frac = float((d > 1e-6).float().mean())
    print(f"[parity] fused tail vs separate after 1 step: max |dp| {float(d.max()):.3e}, fraction > 1e-6: {frac:.3e}")
    assert float(d.max()) <= 2 * 1e-4 * 1.01 and frac < 2e-3


def _adam_ref(p, g, m, v, t, coef, lr=1e-4, b1=0.9, b2=0.999, eps=1e-8):
    """torch.optim.Adam's single-tensor update (models/base.py:106-107 of the reference: clip_grad_norm_ then Adam.step),
    float64 on the CPU."""
    g = g.double() * coef
    m = b1 * m.double() + (1 - b1) * g
    v = b2 * v.double() + (1 - b2) * g * g
    bc1, bc2 = 1 - b1 ** t, 1 - b2 ** t
    return p.double() - (lr / bc1) * m / (v.sqrt() / bc2 ** 0.5 + eps), m, v


@pytest.mark.parametrize("grad_layout", [0, 1])
def test_adam_multi_direct(grad_layout):
    """svrs_adam_multi through the C ABI on a hand-built job table: full tiles of 3x3 / 4x4 layers (the bulk-copy
    path), ragged d0 / d1 (the generic path), a 1x1-like kk, plain ranges between them; gradients in torch layout or in
    the tcgen05 weight-gradient kernels' packed [kk][d1][d0] layout.  p / m / v against float64 Adam; both bf16 packs must
    be EXACTLY the bf16 rounding of the updated fp32 master weight, permuted."""
    gen = torch.Generator().manual_seed(77 + grad_layout)
    shapes = [(64, 32, 9), (96, 48, 16), (40, 20, 9), (32, 16, 16), (4, 16, 9), (128, 64, 9), (16, 4, 16), (64, 16, 1)]
    rec = np.dtype([("off", "<i8"), ("p01", "<u8"), ("p10", "<u8"), ("d0", "<i4"), ("d1", "<i4"), ("kk", "<i4"),
                    ("layout", "<i4"), ("tile0", "<i4"), ("tiles_b", "<i4")])
    assert rec.itemsize == lib.adam_job_bytes()
    rows, off, tile0, keep = [], 0, 0, []
    tr = lib.adam_tile_rows()
    for i, (d0, d1, kk) in enumerate(shapes):
        gap = 24 + 4 * i                                   # a plain range (bias-like) before every weight; keeps off % 4 == 0
        rows.append((off, 0, 0, gap, 0, 1, 0, tile0, 0)); tile0 += (gap + 2047) // 2048; off += gap
        p01 = torch.zeros(kk * d0 * d1, dtype=torch.bfloat16, device=DEV)
        p10 = torch.zeros(kk * d0 * d1, dtype=torch.bfloat16, device=DEV)
        tc = lib.adam_tile_cols(kk)
        tiles_b = (d1 + tc - 1) // tc
        rows.append((off, p01.data_ptr(), p10.data_ptr(), d0, d1, kk, grad_layout, tile0, tiles_b))
        keep.append((off, d0, d1, kk, p01, p10))
        tile0 += ((d0 + tr - 1) // tr) * tiles_b; off += d0 * d1 * kk
    rows.append((off, 0, 0, 3000, 0, 1, 0, tile0, 0)); tile0 += 2; off += 3000      # a plain range spanning two tiles
    n = off
    p0, m0 = torch.randn(n, generator=gen), 0.1 * torch.randn(n, generator=gen)
    v0, g_t = 0.01 * torch.rand(n, generator=gen), torch.randn(n, generator=gen)
    g_buf = g_t.clone()
    if grad_layout == 1:                                   # the weights' gradients sit packed [kk][d1][d0] at the same offset
        for o, d0, d1, kk, _, _ in keep:
            g_buf[o:o + d0 * d1 * kk] = g_t[o:o + d0 * d1 * kk].view(d0, d1, kk).permute(2, 1, 0).reshape(-1)
    t_step, max_norm = 3, 1.0
    coef = min(1.0, max_norm / (float(g_t.double().pow(2).sum().sqrt()) + 1e-6))
    pr, mr, vr = _adam_ref(p0, g_t, m0, v0, t_step, coef)
    pd, md, vd, gd = p0.to(DEV), m0.to(DEV), v0.to(DEV), g_buf.to(DEV)
    acc = torch.zeros(1, dtype=torch.float64, device=DEV)
    lib.sumsq(gd.data_ptr(), n, acc.data_ptr(), st())
    step = torch.tensor([t_step], dtype=torch.int64, device=DEV)
    jobs = torch.from_numpy(np.array(rows, dtype=rec).view(np.uint8).copy()).to(DEV)
    lib.adam_multi(jobs.data_ptr(), len(rows), tile0, 16, pd.data_ptr(), gd.data_ptr(), md.data_ptr(), vd.data_ptr(), BF16,
                   acc.data_ptr(), max_norm, 1.0, 1e-4, 0.9, 0.999, 1e-8, step.data_ptr(), st())
    torch.cuda.synchronize()
    assert torch.equal(gd.cpu(), g_buf), "gradient buffer must not be modified"
    report(f"adam_multi[layout {grad_layout}] p", pd, pr, 1e-6)
    report(f"adam_multi[layout {grad_layout}] m", md, mr, 1e-6)
    report(f"adam_multi[layout {grad_layout}] v", vd, vr, 1e-6)
    for o, d0, d1, kk, p01, p10 in keep:
        w = pd[o:o + d0 * d1 * kk].view(d0, d1, kk)
        assert torch.equal(p01.view(kk, d0, d1), w.permute(2, 0, 1).to(torch.bfloat16)), (d0, d1, kk, "p01")
        assert torch.equal(p10.view(kk, d1, d0), w.permute(2, 1, 0).to(torch.bfloat16)), (d0, d1, kk, "p10")


# ------------------------------------------------------------------------------------------------ f4: fused uncertainty maps
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_sample_stats_fused_tail_matches_reference_statistics(golden_dir, dtype):
    """Streaming Welford statistics in the decoder tail (svrs_sample_tail_stats) == the reference's statistics of the
    materialised draws: (a) against the ORACLE's cond_sample on the CPU, (b) against this repo's own sample() stack,
    for several splits of S (partial merges), injected eps."""
    import fixtures as FX
    fx = FX.load(golden_dir, "cond_cr2_p64_b2")
    model, sd = FX.build(fx, device=DEV, dtype=dtype)
    model.eval()
    eng = model._engine()
    r = O.PortableRng(41)
    S = 37
    eu, es = r.randn(1, eng.Wu), r.randn(S, eng.Wz)
    x, y = FX.inputs(fx)
    y1, x1 = y[1:2], x[1:2]
    ref = task_stats(O.cond_sample({k: v.clone() for k, v in sd.items()}, 2, 64, y1, eu, es, training=False).double(), x1.double())
    tol = 2e-5 if dtype == torch.float32 else 2e-2
    with torch.no_grad():
        own = task_stats(model.sample(y1.to(DEV), samples=S, eps_u=eu.to(DEV), eps_s=es.to(DEV)).double(), x1.to(DEV).double())
        for splits in (1, 3, 4, 0):
            st = model.sample_stats(y1.to(DEV), samples=S, target=x1.to(DEV), eps_u=eu.to(DEV), eps_s=es.to(DEV), splits=splits)
            for k in ("mean", "std", "mae", "mse", "mean_bias", "sample0"):
                # the fixture's draws differ by ~6e-5 (untrained prior): below bf16 resolution of the 16-channel operand, so
                # the bf16 std map is compared on an absolute scale
                report(f"sample_stats[{dtype}, splits={splits}] {k} vs oracle", st[k][0], ref[k], tol,
                       atol=5e-5 if (k == "std" and dtype == torch.bfloat16) else 1e-6)
                report(f"sample_stats[{dtype}, splits={splits}] {k} vs own sample() stack", st[k][0], own[k], 1e-4 if dtype == torch.float32 else 2e-2,
                       atol=2e-6)


def test_sample_stats_batched_patches_match_single(golden_dir):
    """B patches in one call (config 5: 16 patches x 32 draws per tile) == the same patches one at a time (eval mode)."""
    import fixtures as FX
    fx = FX.load(golden_dir, "cond_cr2_p64_b2")
    model, _ = FX.build(fx, device=DEV, dtype=torch.bfloat16)
    model.eval()
    eng = model._engine()
    r = O.PortableRng(43)
    B, S = 3, 16
    y = r.rand(B, 4, 32, 32).to(DEV)
    t = r.rand(B, 4, 64, 64).to(DEV)
    eu, es = r.randn(B, eng.Wu).to(DEV), r.randn(B * S, eng.Wz).to(DEV)
    with torch.no_grad():
        allb = model.sample_stats(y, samples=S, target=t, eps_u=eu, eps_s=es)
        for b in range(B):
            one = model.sample_stats(y[b:b + 1], samples=S, target=t[b:b + 1], eps_u=eu[b:b + 1], eps_s=es[b * S:(b + 1) * S])
            for k in allb:
                report(f"batched sample_stats {k} patch {b}", allb[k][b], one[k][0], 1e-5, atol=1e-6)
        # on-device Philox draws: distinct per patch and per draw
        st = model.sample_stats(y, samples=S)
        assert st["std"].shape == (B, 64, 64) and float(st["std"].min()) >= 0 and float(st["std"].mean()) > 0
        assert "mae" not in st


# ------------------------------------------------------------------------------------------------ narrow layers: guard bands
# (compute-sanitizer is closed on the GPU pool: out-of-bounds WRITES are caught with sentinel guard bands around every output,
# partial 16-pixel steps and non-power-of-two maps exercise the tail / division paths of the mma.sync narrow kernels)
@pytest.mark.parametrize("case", [(3, 12, 20, 4, 4, 3), (3, 12, 20, 16, 4, 3), (2, 20, 12, 4, 16, 3), (5, 6, 6, 4, 16, 4), (1, 64, 64, 16, 4, 3),
                                  (2, 10, 6, 4, 4, 4), (7, 4, 4, 16, 4, 4),
                                  # 16 / 64 -> 16 channels: wgrad16 (mma.sync + ldmatrix.trans from staged rows)
                                  (2, 16, 16, 16, 16, 3), (1, 64, 64, 64, 16, 3), (3, 32, 32, 16, 16, 3), (2, 16, 48, 64, 16, 3),
                                  (5, 8, 16, 16, 16, 3)])
def test_narrow_mma_kernels_odd_shapes_and_guard_bands(case):
    N, H, W, Cin, Cout, ks = case
    g = torch.Generator().manual_seed(sum(case) + 5)
    s = 1 if ks == 3 else 2
    x = _rand((N, Cin, H, W), g)
    w = (_rand((Cout, Cin, ks, ks), g) * 0.2).to(torch.bfloat16).float()
    b = torch.randn(Cout, generator=g)
    xr, wr, br = x.double().requires_grad_(True), w.double().requires_grad_(True), b.double().requires_grad_(True)
    yr = F.conv2d(xr, wr, br, stride=s, padding=1)
    gy = _rand(tuple(yr.shape), g)
    yr.backward(gy.double())
    OH, OW = yr.shape[2:]
    xd, wd, bd, gyd = nhwc(x.to(DEV), torch.bfloat16), w.to(DEV), b.to(DEV), nhwc(gy.to(DEV), torch.bfloat16)
    pf, pb = pack(wd, torch.bfloat16)
    y = Guarded((N, OH, OW, Cout), torch.bfloat16)
    dx = Guarded((N, H, W, Cin), torch.bfloat16)
    dw = Guarded((Cout, Cin, ks, ks), torch.float32, fill=0.0)
    db = Guarded((Cout,), torch.float32, fill=0.0)
    lib.conv2d_fprop(xd.data_ptr(), pf.data_ptr(), pb.data_ptr(), bd.data_ptr(), y.t.data_ptr(), BF16, N, H, W, Cin, Cout, ks, 0, st())
    lib.conv2d_dgrad(gyd.data_ptr(), pb.data_ptr(), pf.data_ptr(), dx.t.data_ptr(), BF16, N, H, W, Cin, Cout, ks, st())
    lib.conv2d_wgrad(xd.data_ptr(), gyd.data_ptr(), dw.t.data_ptr(), None, db.t.data_ptr(), BF16, N, H, W, Cin, Cout, ks, 0, st())
    torch.cuda.synchronize()
    report(f"narrow {case} fprop", nchw(y.t), yr, 7e-3)
    report(f"narrow {case} dgrad", nchw(dx.t), xr.grad, 7e-3)
    report(f"narrow {case} wgrad", dw.t, wr.grad, 2e-5)
    report(f"narrow {case} bgrad", db.t, br.grad, 2e-5)
    assert y.intact() and dx.intact() and dw.intact() and db.intact(), "write outside an output buffer"
