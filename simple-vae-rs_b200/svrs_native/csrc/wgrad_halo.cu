// wgrad_halo.cu - halo-reuse variant of the tcgen05 weight-gradient kernel for the 3x3 stride-1 conv form on maps that
// tile into 8 x 16 pixel blocks: Ca % 64 == 0 and Cb % 64 == 0, or Ca == 16 (the 64 -> 16 and 16 -> 16 decoder tails and
// the first conv of the second down_blocks) with Cb == 16 or 64.
//
//   dW_t[a][b] = sum_m G[m][a] * X[m shifted by tap t][b]
//
// wgrad_tc.cu loads one shifted X box per (tap, channel chunk) and pixel step - nine L2 reads of (almost) the same pixels.
// Here a CTA owns ONE chunk of X (b, CB_T = 64 or 16 channels) and ONE tile of G (a, CA_T = 64 or 16 channels); per
// 128-pixel step it loads the X HALO once (18 x 16 pixels x CB_T ch) and the G tile once, and issues for all nine taps
//     D[(taps, b) 128 rows, a CA_T cols] += A^T B      (8 MMAs of K = 16 pixels per accumulator)
// where the A operand is an MN-major descriptor INTO THE HALO: K (pixel) groups of 8 are one halo row apart and the M
// dimension is made of 128 / CB_T channel atoms, LBO bytes apart, each atom one tap:
//   * CB_T = 64 (SWIZZLE_128B): two atoms = a tap pair, LBO = difference of the two taps' halo offsets; five pairs
//     (0,1) (2,3) (4,5) (6,7) (8,-) -> 5 accumulators, 40 MMAs per step.
//   * CB_T = 16 (SWIZZLE_32B, 32-byte rows): eight atoms one pixel apart (LBO = 32 B) starting at dx = -1 of a halo row:
//     atoms 0..2 are the taps (dy, -1) (dy, 0) (dy, +1), atoms 3..7 are ignored by the epilogue; one accumulator per dy ->
//     3 accumulators, 24 MMAs per step.  (Nine taps are never eight equally spaced atoms, so three per MMA is the best a
//     128-row MMA over an X halo gets.)
// Why X and not G carries the halo: shifting G (taps along N, one descriptor per tap) would put 48 columns into an
// MMA only at M = 64 (X has 64 or 16 channels), and M = 64 MMAs cost the same ~58 issue cycles (DESIGN.md §3.1); shifting
// both operands is not a tiling of the image.  Per 128-pixel step, CB_T = 64: 40 x ~58 = 2.3 k cycles of MMA issue against
// ~1.7 k cycles of TMA rows (288 halo + 128 G rows at ~4 cycles each) -> issue-bound; CB_T = 16: 24 x 58 = 1.4 k cycles of
// issue against the same ~1.7 k cycles of rows -> TMA-row-bound.  Measured on B200 at 128 patches and 64 x 64 on 74 CTAs:
// 73 us (64 -> 16) and 50 us (16 -> 16), against 65 and 47 us from these counts (DESIGN.md §3).
// Accumulators (NACC x CA_T TMEM columns) stay resident for the CTA's pixel range.
#include "common.cuh"
#include "taps.cuh"
#include "tc_ptx.cuh"
#include <string.h>
#include <stdlib.h>

namespace svrs {

constexpr int WH_STAGES = 4;
constexpr int WH_MAX_STAGE_BYTES = 18 * 16 * 128 + 128 * 128;   // 64-channel halo (36864) + 64-channel G tile (16384)
constexpr int WH_SMEM_BYTES = WH_STAGES * WH_MAX_STAGE_BYTES + 1024 + 256;
constexpr int WH_THREADS = 192;
constexpr int WH_MAX_ACC = 5;

struct alignas(64) WhParams {
    CUtensorMap x_map;   // (Cb, W, H, N) box (CB_T, 16, 18, 1)
    CUtensorMap g_map;   // (Ca, W, H, N) box (CA_T, 8, 16, 1)
    CUtensorMap dw_map;  // packed mode: fp32 scratch [9*Cb rows][Ca], box (min(32, CA_T) columns, CB_T rows)
    float* dw;
    float* db;                      // != NULL: bias gradient folded in (column sums of G by the idle epilogue warps)
    const __nv_bfloat16* gptr;
    int N, OH, OW, tiles_x, tiles_y;
    int Ca, Cb;
    int a_tiles, b_chunks, ksplit, ksteps_total, packed;
    uint32_t a_rel[WH_MAX_ACC];     // per accumulator: A descriptor low word relative to the halo (start >> 4 | LBO field)
    int tap_of[WH_MAX_ACC * 8];     // [accumulator][atom] -> tap index of the packed / torch gradient, -1 = ignored rows
};

template <int CA_T, int CB_T>
__global__ void __launch_bounds__(WH_THREADS, 1) wgrad3_halo_kernel(const __grid_constant__ WhParams p) {
    constexpr uint32_t XROW = 2u * CB_T, GROW = 2u * CA_T;       // bytes per pixel of the X halo / G tile
    constexpr uint32_t HALO_BYTES = 18u * 16u * XROW;
    constexpr uint32_t G_BYTES = 128u * GROW;
    constexpr uint32_t STAGE_BYTES = HALO_BYTES + G_BYTES;       // 53248 / 40960 / 13312 (multiples of 1024)
    constexpr int NACC = CB_T == 64 ? 5 : 3;
    constexpr int NATOM = 128 / CB_T;                            // channel atoms (taps) per accumulator
    constexpr uint32_t XLT = CB_T == 64 ? 2u : 6u, GLT = CA_T == 64 ? 2u : 6u;   // SWIZZLE_128B / SWIZZLE_32B
    static_assert(STAGE_BYTES % 1024 == 0 && STAGE_BYTES <= WH_MAX_STAGE_BYTES, "stage layout");
    pdl_entry();
    extern __shared__ uint8_t smem_raw[];
    const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
    const uint32_t bar_base = smem_base + WH_STAGES * WH_MAX_STAGE_BYTES;
    auto full_bar = [&](int s) { return bar_base + 8u * s; };
    auto empty_bar = [&](int s) { return bar_base + 8u * (WH_STAGES + s); };
    const uint32_t done_bar = bar_base + 8u * (2 * WH_STAGES);
    const uint32_t tmem_slot = bar_base + 8u * (2 * WH_STAGES + 1);
    uint32_t* tmem_slot_ptr = reinterpret_cast<uint32_t*>(smem_raw + (tmem_slot - smem_u32(smem_raw)));
    const int warp = threadIdx.x / 32, lane = threadIdx.x % 32;

    if (warp == 0 && lane == 0) {
        prefetch_tmap(&p.x_map);
        prefetch_tmap(&p.g_map);
        if (p.packed) prefetch_tmap(&p.dw_map);
        for (int s = 0; s < WH_STAGES; ++s) { mbar_init(full_bar(s), 1); mbar_init(empty_bar(s), 1); }
        mbar_init(done_bar, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 512;" ::"r"(tmem_slot) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot_ptr;
    pdl_wait();     // prologue above overlaps the previous kernel; nothing before this line touches global memory

    int w = blockIdx.x;
    const int bj = w % p.b_chunks; w /= p.b_chunks;     // CB_T-channel chunk of X (b)
    const int at = w % p.a_tiles; w /= p.a_tiles;       // CA_T-channel tile of G (a)
    const int ks = w;
    const int steps_per = (p.ksteps_total + p.ksplit - 1) / p.ksplit;
    const int k_begin = ks * steps_per;
    const int k_end = (k_begin + steps_per) < p.ksteps_total ? (k_begin + steps_per) : p.ksteps_total;
    const int nsteps = k_end > k_begin ? k_end - k_begin : 0;

    if (warp == 0) {
        if (lane == 0) {
            uint32_t stage = 0, phase = 0;
            for (int kstep = k_begin; kstep < k_end; ++kstep) {
                int pt = kstep;
                const int tx = pt % p.tiles_x; pt /= p.tiles_x;
                const int ty = pt % p.tiles_y;
                const int n = pt / p.tiles_y;
                mbar_wait(empty_bar(stage), phase ^ 1u);
                const uint32_t sh = smem_base + stage * STAGE_BYTES;
                mbar_expect_tx(full_bar(stage), STAGE_BYTES);
                tma_load_4d(sh, &p.x_map, full_bar(stage), bj * CB_T, tx * 8 - 1, ty * 16 - 1, n);
                tma_load_4d(sh + HALO_BYTES, &p.g_map, full_bar(stage), at * CA_T, tx * 8, ty * 16, n);
                if (++stage == WH_STAGES) { stage = 0; phase ^= 1u; }
            }
        }
    } else if (warp == 1) {
        if (lane == 0) {
            // D = f32, A = B = bf16, both MN-major, N = CA_T, M = 128
            const uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | (1u << 15) | (1u << 16) | ((uint32_t)(CA_T >> 3) << 17) | ((128u >> 4) << 24);
            const uint32_t a_hi = desc_hi(16u * XROW, XLT), b_hi = desc_hi(8u * GROW, GLT);
            uint32_t a_rel[NACC];
#pragma unroll
            for (int b = 0; b < NACC; ++b) a_rel[b] = p.a_rel[b];
            uint32_t stage = 0, phase = 0;
            for (int kstep = 0; kstep < nsteps; ++kstep) {
                mbar_wait(full_bar(stage), phase);
                tc_fence_after();
                const uint32_t sh = smem_base + stage * STAGE_BYTES;
                const uint32_t a0 = (sh & 0x3FFFF) >> 4;
                const uint32_t b0 = desc_lo(sh + HALO_BYTES, G_BYTES);
#pragma unroll
                for (int k = 0; k < 8; ++k)                        // 16 pixels = 2 halo rows per MMA
#pragma unroll
                    for (int b = 0; b < NACC; ++b)
                        tc_mma_lohi(tmem_base + (uint32_t)(b * CA_T), a0 + a_rel[b] + (2u * XROW) * k, a_hi, b0 + GROW * k, b_hi, idesc,
                                    k ? 1u : (uint32_t)(kstep != 0));
                tc_commit(empty_bar(stage));
                if (kstep == nsteps - 1) tc_commit(done_bar);
                if (++stage == WH_STAGES) { stage = 0; phase ^= 1u; }
            }
        }
    } else if (nsteps > 0) {
        const int q = warp % 4;
        const int m = q * 32 + lane;
        if (p.db) {           // the b-chunk CTAs of a (pixel split, tile of G) share the column sums: chunk bj takes every b_chunks-th step
            __shared__ float csum[128][8];
            constexpr int cg = CA_T / 8, lanes = 128 / cg;
            const int t = threadIdx.x - 64, cq = t % cg, cl = t / cg;
            float acc[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
            const long long sx = p.Ca, sy = (long long)p.OW * p.Ca, sn = (long long)p.OH * p.OW * p.Ca;
            for (int kstep = k_begin + bj; kstep < k_end; kstep += p.b_chunks) {
                int pt = kstep;
                const int tx = pt % p.tiles_x; pt /= p.tiles_x;
                const int ty = pt % p.tiles_y;
                const int n = pt / p.tiles_y;
                colsum_tile8(p.gptr, sn, sy, sx, n, ty * 16, tx * 8, 8, 16, 1, p.N, at * CA_T + cq * 8, cl, lanes, acc);
            }
            colsum_finish(csum, acc, t, cq, cl, cg, lanes, p.db, at * CA_T, p.Ca);
        }
        mbar_wait(done_bar, 0);
        tc_fence_after();
        const int h = m / CB_T, r = m % CB_T;              // h: which atom (tap) of the accumulator, r: channel in the chunk
        if (p.packed) {
            // packed scratch [tap][b][a]: stage each 128 x CA_T accumulator (NATOM taps x CB_T b-rows) in shared memory in the
            // tensor map's swizzled box layout, then ONE thread adds it with TMA tensor reductions (see wgrad_tc.cu)
            constexpr int CWD = CA_T < 32 ? CA_T : 32, NCH = CA_T / CWD;
            constexpr uint32_t ROW_BYTES = 4u * CWD, BOX_BYTES = CB_T * ROW_BYTES, BLK_BYTES = 128u * 4u * CA_T;
            const bool issuer = threadIdx.x == 64;
            for (int b = 0; b < NACC; ++b) {
                const uint32_t buf = smem_base + (uint32_t)(b & 1) * BLK_BYTES;
                if (b >= 2) {
                    if (issuer) bulk_wait_read_1();
                    named_bar_sync(1, 128);
                }
                const uint32_t taddr = tmem_base + (uint32_t)(b * CA_T) + ((uint32_t)(q * 32) << 16);
#pragma unroll
                for (int c0 = 0; c0 < CA_T; c0 += CWD) {
                    uint32_t v[32];
                    const uint32_t box = buf + (uint32_t)(h * NCH + c0 / CWD) * BOX_BYTES;
                    if (CWD == 32) { tmem_ld32(taddr + c0, v); tmem_ld_wait(); stage_row_swizzled<8>(box, r, ROW_BYTES, v); }
                    else { tmem_ld16(taddr + c0, v); tmem_ld_wait(); stage_row_swizzled<4>(box, r, ROW_BYTES, v); }
                }
                fence_proxy_async_smem();
                named_bar_sync(1, 128);
                if (issuer) {
                    for (int hh = 0; hh < NATOM; ++hh) {
                        const int tap = p.tap_of[b * 8 + hh];
                        if (tap < 0) continue;
                        for (int cc = 0; cc < NCH; ++cc)
                            tma_reduce_add_2d(&p.dw_map, buf + (uint32_t)(hh * NCH + cc) * BOX_BYTES, at * CA_T + cc * CWD, tap * p.Cb + bj * CB_T);
                    }
                    bulk_commit();
                }
            }
            if (issuer) bulk_wait_all();
        } else {
            const int cb = bj * CB_T + r;
            for (int b = 0; b < NACC; ++b) {
                const int tap = p.tap_of[b * 8 + h];
                const uint32_t taddr = tmem_base + (uint32_t)(b * CA_T) + ((uint32_t)(q * 32) << 16);
                for (int c0 = 0; c0 < CA_T; c0 += 32) {
                    uint32_t v[32];
                    if (CA_T >= 32) tmem_ld32(taddr + c0, v); else tmem_ld16(taddr + c0, v);
                    tmem_ld_wait();
                    if (tap >= 0) {
#pragma unroll
                        for (int j = 0; j < (CA_T < 32 ? CA_T : 32); ++j) {
                            const int ca = at * CA_T + c0 + j;
                            atomicAdd(p.dw + ((long long)ca * p.Cb + cb) * 9 + tap, __uint_as_float(v[j]));
                        }
                    }
                }
            }
        }
    }

    tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 512;" ::"r"(tmem_base) : "memory");
    }
}

int get_halo_mode();

// Which (Ca, Cb) the halo kernel takes.  Ca = 16 layers on maps that do not tile into 8 x 16 pixels go to wgrad_tc.
static bool wh_channels_ok(int Ca, int Cb) {
    return (Ca % 64 == 0 && Cb % 64 == 0) || (Ca == 16 && (Cb == 16 || Cb == 64));
}

bool wgrad_halo_supported(const TapGeom& g, int KK) {
    return get_halo_mode() != 0 && KK == 9 && g.nprob == 1 && g.prob[0].ntaps == 9 && wh_channels_ok(g.Nc, g.K) &&
           g.OW % 8 == 0 && g.OH % 16 == 0 && g.IH == g.OH && g.IW == g.OW;
}

static void wh_plan(const TapGeom& g, WhParams& p) {
    memset(&p, 0, sizeof(p));
    p.N = g.N; p.OH = g.OH; p.OW = g.OW; p.tiles_x = g.OW / 8; p.tiles_y = g.OH / 16;
    p.Ca = g.Nc; p.Cb = g.K;
    p.a_tiles = p.Ca / (p.Ca % 64 == 0 ? 64 : 16); p.b_chunks = p.Cb / (p.Cb % 64 == 0 ? 64 : 16);
    p.ksteps_total = p.tiles_x * p.tiles_y * g.N;
    int base = p.a_tiles * p.b_chunks;
    static int ctas_target = 0;
    // about half the SMs (measured on the bench step, as for wgrad_tc: weight gradients run next to the dgrad chain)
    if (!ctas_target) { const char* e = getenv("SVRS_WG_CTAS"); ctas_target = e ? atoi(e) : num_sms() / 2; }
    int ksplit = (ctas_target + base - 1) / base;
    // every split pays the first load and the TMA-reduce epilogue again: at least 4 pixel steps per split (as wgrad_tc)
    if (ksplit > p.ksteps_total / 4) ksplit = p.ksteps_total / 4;
    if (ksplit < 1) ksplit = 1;
    const int steps_per = (p.ksteps_total + ksplit - 1) / ksplit;      // exact: every split owns >= 1 k-step (slab mode)
    p.ksplit = (p.ksteps_total + steps_per - 1) / steps_per;
}

int wgrad_halo_splits(const TapGeom& g) {
    WhParams p;
    wh_plan(g, p);
    return p.ksplit;
}

int launch_wgrad3_halo(const TapGeom& g, const void* gmat, const void* x, float* dw, int packed, float* db, cudaStream_t st) {
    static bool attr_set = false;
    if (!attr_set) {
        cudaError_t e = cudaFuncSetAttribute(wgrad3_halo_kernel<64, 64>, cudaFuncAttributeMaxDynamicSharedMemorySize, WH_SMEM_BYTES);
        if (e == cudaSuccess) e = cudaFuncSetAttribute(wgrad3_halo_kernel<16, 64>, cudaFuncAttributeMaxDynamicSharedMemorySize, WH_SMEM_BYTES);
        if (e == cudaSuccess) e = cudaFuncSetAttribute(wgrad3_halo_kernel<16, 16>, cudaFuncAttributeMaxDynamicSharedMemorySize, WH_SMEM_BYTES);
        if (e != cudaSuccess) { set_error("wgrad3_halo: cudaFuncSetAttribute: %s", cudaGetErrorString(e)); return SVRS_E_CUDA; }
        attr_set = true;
    }
    if (!wh_channels_ok(g.Nc, g.K)) { set_error("wgrad3_halo: unsupported channels Ca=%d Cb=%d", g.Nc, g.K); return SVRS_E_UNSUPPORTED; }
    WhParams p;
    wh_plan(g, p);
    p.dw = dw;
    p.packed = packed;
    p.db = db;
    p.gptr = reinterpret_cast<const __nv_bfloat16*>(gmat);
    const int ca_t = p.Ca % 64 == 0 ? 64 : 16, cb_t = p.Cb % 64 == 0 ? 64 : 16;
    const uint32_t xrow = 2u * (uint32_t)cb_t;
    const Prob& pb = g.prob[0];
    for (int i = 0; i < WH_MAX_ACC * 8; ++i) p.tap_of[i] = -1;
    int off[9];                                     // halo pixel offset ((dy+1)*16 + (dx+1)) per tap
    for (int t = 0; t < 9; ++t) off[t] = (pb.taps[t].dy + 1) * 16 + (pb.taps[t].dx + 1);
    if (cb_t == 64) {
        for (int b = 0; b < 5; ++b) {               // tap pairs (0,1) (2,3) (4,5) (6,7) (8,-)
            // tail pair: the second atom is any valid view, its rows are ignored by the epilogue
            const uint32_t o0 = (uint32_t)off[2 * b] * xrow, o1 = 2 * b + 1 < 9 ? (uint32_t)off[2 * b + 1] * xrow : o0 + xrow;
            if (o1 <= o0) { set_error("wgrad3_halo: taps not in ascending halo order"); return SVRS_E_ARG; }   // LBO is unsigned
            p.a_rel[b] = (o0 >> 4) | ((((o1 - o0) >> 4) & 0x3FFF) << 16);
            p.tap_of[b * 8] = 2 * b;
            if (2 * b + 1 < 9) p.tap_of[b * 8 + 1] = 2 * b + 1;
        }
    } else {
        for (int b = 0; b < 3; ++b) p.a_rel[b] = ((b * 16u * xrow) >> 4) | ((xrow >> 4) << 16);   // atoms one pixel apart
        for (int t = 0; t < 9; ++t) p.tap_of[(off[t] / 16) * 8 + off[t] % 16] = t;
    }
    int rc = make_act_map(&p.x_map, x, p.Cb, g.IW, g.IH, g.N, g.i_sx, g.i_sy, g.i_sn, 16, 18, 1, cb_t);
    if (rc) return rc;
    rc = make_act_map(&p.g_map, gmat, p.Ca, g.OW, g.OH, g.N, g.o_sx, g.o_sy, g.o_sn, 8, 16, 1, ca_t);
    if (rc) return rc;
    if (packed) {
        rc = make_f32_2d_map(&p.dw_map, dw, p.Ca, 9ll * p.Cb, ca_t < 32 ? ca_t : 32, cb_t);
        if (rc) return rc;
    }
    const int grid = p.a_tiles * p.b_chunks * p.ksplit;
    if (ca_t == 64) SVRS_LAUNCH((wgrad3_halo_kernel<64, 64>), grid, WH_THREADS, WH_SMEM_BYTES, st, p);
    else if (cb_t == 64) SVRS_LAUNCH((wgrad3_halo_kernel<16, 64>), grid, WH_THREADS, WH_SMEM_BYTES, st, p);
    else SVRS_LAUNCH((wgrad3_halo_kernel<16, 16>), grid, WH_THREADS, WH_SMEM_BYTES, st, p);
    return check_launch("wgrad3_halo_kernel");
}

}  // namespace svrs
