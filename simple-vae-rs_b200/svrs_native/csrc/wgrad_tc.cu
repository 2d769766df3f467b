// wgrad_tc.cu - tcgen05 / TMEM / TMA weight-gradient kernel for sm_100a (bf16 in, fp32 accumulate).
//
//   dW_t[a][b] = sum over output-grid pixels m of  G[m][a] * X_t[m shifted by tap t][b]
//
// GEMM view per CTA:  D[(tap, b) rows, a columns] += Xstack^T * G, reduction (K) over pixels.
//   * M (128 rows of one "M-block") = 128/cwx boxes of X, each cwx channels wide (cwx = 64/32/16) taken at one or
//     more taps; the boxes are the same TMA tiles the forward kernel reads (cwx ch x 128 pixels, 128/64/32-byte
//     swizzle) and are fed to tcgen05.mma as an MN-MAJOR A operand (channels contiguous, pixels = K), boxes one LBO apart.
//   * N = up to 128 channels of G (MN-major B operand, boxes cwg = min(64, Ca) channels wide).
//   * K = 128 pixels per pipeline stage (8 MMAs of K=16); the pixel range is split over CTAs.
//   * every CTA keeps up to 512/N M-blocks of accumulators resident in TMEM for its whole pixel range and
//     finishes with fp32 atomics into the torch-layout gradient dw[(a*Cb + b)*KK + tap].
// TMA zero-fill implements the convolution padding for X and masks out-of-range images for G.  It also pads ragged channel
// counts (Ca or Cb % 8 == 0 but not a multiple of the box width): the last G / X box reads zeros past Ca / Cb, so those
// accumulator columns / rows are zero, and the epilogues clip them (3-D reduce map, masked atomics, masked bias sums).
#include "common.cuh"
#include "taps.cuh"
#include "tc_ptx.cuh"
#include <string.h>
#include <stdlib.h>

namespace svrs {

// Shared memory: a ring of X slots (one M-block each: 128 box-channel rows x 128 pixels) and a ring of G slots (up to 128
// channels x 128 pixels).  The G tile of a pixel step is loaded ONCE and stays resident while all M-blocks of the CTA's
// group consume it (it used to travel with every X block: (group + 1) instead of 2 * group boxes per step - these layers
// are bound by the SM's L2 ingest).
constexpr int WG_XSLOTS = 4;
constexpr int WG_GSLOTS = 2;
constexpr int WG_X_BYTES = 128 * 128 * 2;
constexpr int WG_G_BYTES = 128 * 128 * 2;
constexpr int WG_SMEM_BYTES = WG_XSLOTS * WG_X_BYTES + WG_GSLOTS * WG_G_BYTES + 1024 + 256;
constexpr int WG_THREADS = 192;
constexpr int WG_MAX_GROUP = 16;

struct WgTap { int map, dy, dx, tapid; };
struct alignas(64) WgParams {
    CUtensorMap x_maps[4];    // input views (parity classes)
    CUtensorMap g_map;        // output-grid operand
    CUtensorMap dw_map;       // packed mode: fp32 scratch [KK][Cb][Ca], box (min(32, n_tile) columns, cwx rows, 1 tap)
    float* dw;
    float* db;                         // != NULL: bias gradient (column sums of G) folded in, see colsum_tile8
    const __nv_bfloat16* gptr;         // G base (output view) and its element strides, for the folded column sums
    long long g_sn, g_sy, g_sx;
    int N, OH, OW, BW, BH, BNI;
    int tiles_x, tiles_y, tiles_n;     // pixel tiling of the output grid
    int Ca, Cb, KK;
    int n_tile, n_tiles;               // columns (a) per CTA
    int cwx, cwg;                      // box widths (channels) of the X and G operands
    int cb_chunks;                     // ceil(Cb / cwx)
    int bpb;                           // boxes per M-block = 128 / cwx
    int nboxes, nblocks, group, ngroups;
    int ksplit, ksteps_total;
    int ntaps, packed;
    long long* prof;                   // debug (SVRS_WG_PROF=1): per-CTA clock64 stamps, 8 per CTA
    WgTap taps[16];
};

__global__ void __launch_bounds__(WG_THREADS, 1) wgrad_tc_kernel(const __grid_constant__ WgParams p) {
    pdl_entry();
    extern __shared__ uint8_t smem_raw[];
    const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
    const uint32_t g_base = smem_base + WG_XSLOTS * WG_X_BYTES;
    const uint32_t bar_base = g_base + WG_GSLOTS * WG_G_BYTES;
    auto xfull = [&](int s) { return bar_base + 8u * s; };
    auto xempty = [&](int s) { return bar_base + 8u * (WG_XSLOTS + s); };
    auto gfull = [&](int s) { return bar_base + 8u * (2 * WG_XSLOTS + s); };
    auto gempty = [&](int s) { return bar_base + 8u * (2 * WG_XSLOTS + WG_GSLOTS + s); };
    const uint32_t done_bar = bar_base + 8u * (2 * WG_XSLOTS + 2 * WG_GSLOTS);
    const uint32_t tmem_slot = bar_base + 8u * (2 * WG_XSLOTS + 2 * WG_GSLOTS + 1);
    uint32_t* tmem_slot_ptr = reinterpret_cast<uint32_t*>(smem_raw + (tmem_slot - smem_u32(smem_raw)));
    const int warp = threadIdx.x / 32, lane = threadIdx.x % 32;
    long long* prof = p.prof ? p.prof + 8ll * blockIdx.x : nullptr;
    if (prof && threadIdx.x == 0) prof[0] = clock64();

    if (warp == 0 && lane == 0) {
        for (int i = 0; i < 4; ++i) prefetch_tmap(&p.x_maps[i]);
        prefetch_tmap(&p.g_map);
        if (p.packed) prefetch_tmap(&p.dw_map);
        for (int s = 0; s < WG_XSLOTS; ++s) { mbar_init(xfull(s), 1); mbar_init(xempty(s), 1); }
        for (int s = 0; s < WG_GSLOTS; ++s) { mbar_init(gfull(s), 1); mbar_init(gempty(s), 1); }
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
    if (prof && threadIdx.x == 0) prof[1] = clock64();

    // work item: (pixel split ks, column tile nt, M-block group grp)
    int w = blockIdx.x;
    const int grp = w % p.ngroups; w /= p.ngroups;
    const int nt = w % p.n_tiles; w /= p.n_tiles;
    const int ks = w;
    const int blk0 = grp * p.group;
    const int nblk = (p.nblocks - blk0) < p.group ? (p.nblocks - blk0) : p.group;
    const int steps_per = (p.ksteps_total + p.ksplit - 1) / p.ksplit;
    const int k_begin = ks * steps_per;
    const int k_end = (k_begin + steps_per) < p.ksteps_total ? (k_begin + steps_per) : p.ksteps_total;
    const int nsteps = k_end > k_begin ? k_end - k_begin : 0;
    const int g_boxes = (p.n_tile + p.cwg - 1) / p.cwg;
    const uint32_t x_box = 128u * (uint32_t)p.cwx * 2u;   // bytes of one X box  (128 pixels x cwx ch)
    const uint32_t g_box = 128u * (uint32_t)p.cwg * 2u;

    if (warp == 0) {
        if (lane == 0) {
            uint32_t xs = 0, xph = 0, gs = 0, gph = 0;
            for (int kstep = k_begin; kstep < k_end; ++kstep) {
                int pt = kstep;
                const int tx = pt % p.tiles_x; pt /= p.tiles_x;
                const int ty = pt % p.tiles_y;
                const int tn = pt / p.tiles_y;
                const int x0 = tx * p.BW, y0 = ty * p.BH, n0 = tn * p.BNI;
                mbar_wait(gempty(gs), gph ^ 1u);
                const uint32_t sg = g_base + gs * WG_G_BYTES;
                mbar_expect_tx(gfull(gs), (uint32_t)g_boxes * g_box);
                for (int gbx = 0; gbx < g_boxes; ++gbx)
                    tma_load_4d(sg + gbx * g_box, &p.g_map, gfull(gs), nt * p.n_tile + gbx * p.cwg, x0, y0, n0);
                if (++gs == WG_GSLOTS) { gs = 0; gph ^= 1u; }
                for (int b = 0; b < nblk; ++b) {
                    mbar_wait(xempty(xs), xph ^ 1u);
                    const uint32_t sx = smem_base + xs * WG_X_BYTES;
                    mbar_expect_tx(xfull(xs), (uint32_t)p.bpb * x_box);
                    for (int h = 0; h < p.bpb; ++h) {
                        int box = p.bpb * (blk0 + b) + h;
                        if (box >= p.nboxes) box = p.nboxes - 1;       // tail: duplicate (rows are ignored by the epilogue)
                        const WgTap tp = p.taps[box / p.cb_chunks];
                        const int cj = box % p.cb_chunks;
                        tma_load_4d(sx + h * x_box, &p.x_maps[tp.map], xfull(xs), cj * p.cwx, x0 + tp.dx, y0 + tp.dy, n0);
                    }
                    if (++xs == WG_XSLOTS) { xs = 0; xph ^= 1u; }
                }
            }
        }
    } else if (warp == 1) {
        if (lane == 0) {
            // D = f32, A = B = bf16, both MN-major (bits 15, 16), N = n_tile, M = 128
            const uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | (1u << 15) | (1u << 16) |
                                   ((uint32_t)(p.n_tile >> 3) << 17) | ((128u >> 4) << 24);
            const uint32_t a_hi = desc_hi(16u * (uint32_t)p.cwx, p.cwx == 64 ? 2u : (p.cwx == 32 ? 4u : 6u));   // 8 pixel rows
            const uint32_t b_hi = desc_hi(16u * (uint32_t)p.cwg, p.cwg == 64 ? 2u : (p.cwg == 32 ? 4u : 6u));
            const uint32_t kadv_x16 = 2u * (uint32_t)p.cwx, kadv_g16 = 2u * (uint32_t)p.cwg;                    // 16 pixel rows, >> 4
            uint32_t xs = 0, xph = 0, gs = 0, gph = 0;
            for (int kstep = 0; kstep < nsteps; ++kstep) {
                mbar_wait(gfull(gs), gph);
                const uint32_t b0 = desc_lo(g_base + gs * WG_G_BYTES, g_box);
                for (int b = 0; b < nblk; ++b) {
                    mbar_wait(xfull(xs), xph);
                    tc_fence_after();
                    if (prof && kstep == 0 && b == 0) prof[2] = clock64();
                    const uint32_t a0 = desc_lo(smem_base + xs * WG_X_BYTES, x_box);
                    const uint32_t d_tmem = tmem_base + (uint32_t)(b * p.n_tile);
#pragma unroll
                    for (int k = 0; k < 8; ++k)     // 8 x (K = 16 pixels)
                        tc_mma_lohi(d_tmem, a0 + kadv_x16 * k, a_hi, b0 + kadv_g16 * k, b_hi, idesc, k ? 1u : (uint32_t)(kstep != 0));
                    tc_commit(xempty(xs));
                    if (b == nblk - 1) tc_commit(gempty(gs));      // every M-block of the group has consumed this G tile
                    if (kstep == nsteps - 1 && b == nblk - 1) { tc_commit(done_bar); if (prof) prof[3] = clock64(); }
                    if (++xs == WG_XSLOTS) { xs = 0; xph ^= 1u; }
                }
                if (++gs == WG_GSLOTS) { gs = 0; gph ^= 1u; }
            }
        }
    } else if (nsteps > 0) {
        const int q = warp % 4;
        const int m = q * 32 + lane;
        if (p.db) {          // the CTAs of a (pixel split, column tile) share its G tiles' column sums: group g takes every ngroups-th step
            __shared__ float csum[128][8];
            const int cg = p.n_tile / 8, lanes = 128 / cg;
            const int t = threadIdx.x - 64, cq = t % cg, cl = t / cg;
            float acc[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
            // Ca % 8 == 0: an 8-column group lies wholly inside or wholly past the last G column (ragged last tile)
            const int kfirst = nt * p.n_tile + cq * 8 < p.Ca ? k_begin + grp : k_end;
            for (int kstep = kfirst; kstep < k_end; kstep += p.ngroups) {
                int pt = kstep;
                const int tx = pt % p.tiles_x; pt /= p.tiles_x;
                const int ty = pt % p.tiles_y;
                const int tn = pt / p.tiles_y;
                colsum_tile8(p.gptr, p.g_sn, p.g_sy, p.g_sx, tn * p.BNI, ty * p.BH, tx * p.BW, p.BW, p.BH, p.BNI, p.N,
                             nt * p.n_tile + cq * 8, cl, lanes, acc);
            }
            colsum_finish(csum, acc, t, cq, cl, cg, lanes, p.db, nt * p.n_tile, p.Ca);
        }
        mbar_wait(done_bar, 0);
        tc_fence_after();
        if (prof && threadIdx.x == 64) prof[4] = clock64();
        if (p.packed) {
            // Packed scratch [tap][b][a] (a fastest): stage each 128 x n_tile accumulator block in shared memory (the
            // pipeline stages are idle by now) in the tensor map's swizzled box layout and let ONE thread add it to the
            // scratch with a few TMA tensor reductions - boxes of (32 | 16 columns) x (cwx rows), i.e. one X box each.
            // Two staging buffers: block b+1 is read out of TMEM while the reductions of block b are still in flight.
            const int cwd = p.n_tile < 32 ? p.n_tile : 32;
            const int nch = p.n_tile / cwd;
            const uint32_t row_bytes = 4u * (uint32_t)cwd;
            const uint32_t box_bytes = (uint32_t)p.cwx * row_bytes;
            const uint32_t blk_bytes = 128u * 4u * (uint32_t)p.n_tile;
            const int h = m / p.cwx, r = m % p.cwx;
            const bool issuer = threadIdx.x == 64;
            for (int b = 0; b < nblk; ++b) {
                const uint32_t buf = smem_base + (uint32_t)(b & 1) * blk_bytes;
                if (b >= 2) {
                    if (issuer) bulk_wait_read_1();      // the reductions that last read this buffer are done with it
                    named_bar_sync(1, 128);
                }
                const uint32_t taddr = tmem_base + (uint32_t)(b * p.n_tile) + ((uint32_t)(q * 32) << 16);
                for (int c0 = 0; c0 < p.n_tile; c0 += 32) {
                    uint32_t v[32];
                    const uint32_t box = buf + (uint32_t)(h * nch + c0 / 32) * box_bytes;
                    if (cwd == 32) { tmem_ld32(taddr + c0, v); tmem_ld_wait(); stage_row_swizzled<8>(box, r, row_bytes, v); }
                    else { tmem_ld16(taddr + c0, v); tmem_ld_wait(); stage_row_swizzled<4>(box, r, row_bytes, v); }
                }
                fence_proxy_async_smem();
                named_bar_sync(1, 128);
                if (issuer) {
                    for (int hh = 0; hh < p.bpb; ++hh) {
                        const int box = p.bpb * (blk0 + b) + hh;
                        if (box >= p.nboxes) break;                       // tail rows of the last M-block
                        const int tapid = p.taps[box / p.cb_chunks].tapid, row0 = (box % p.cb_chunks) * p.cwx;
                        for (int cc = 0; cc < nch; ++cc)      // the map clips columns >= Ca and rows >= Cb of a ragged box
                            tma_reduce_add_3d(&p.dw_map, buf + (uint32_t)(hh * nch + cc) * box_bytes, nt * p.n_tile + cc * cwd, row0, tapid);
                    }
                    bulk_commit();
                }
            }
            if (issuer) bulk_wait_all();
        } else {
            for (int b = 0; b < nblk; ++b) {
                const int box = p.bpb * (blk0 + b) + m / p.cwx;
                const int bx = box < p.nboxes ? box : 0;
                const int tapid = p.taps[bx / p.cb_chunks].tapid;
                const int cb = (bx % p.cb_chunks) * p.cwx + (m % p.cwx);
                const bool row_ok = box < p.nboxes && cb < p.Cb;         // rows past Cb: zero fill of a ragged X box
                const uint32_t taddr = tmem_base + (uint32_t)(b * p.n_tile) + ((uint32_t)(q * 32) << 16);
                for (int c0 = 0; c0 < p.n_tile; c0 += 32) {
                    uint32_t v[32];
                    const int cols = (p.n_tile - c0 >= 32) ? 32 : 16;
                    if (cols == 32) tmem_ld32(taddr + c0, v); else tmem_ld16(taddr + c0, v);
                    tmem_ld_wait();
                    if (row_ok) {
#pragma unroll
                        for (int j = 0; j < 32; ++j) {
                            const int ca = nt * p.n_tile + c0 + j;
                            if (j < cols && ca < p.Ca)
                                atomicAdd(p.dw + ((long long)ca * p.Cb + cb) * p.KK + tapid, __uint_as_float(v[j]));
                        }
                    }
                }
            }
        }
    }

    if (prof && threadIdx.x == 64) { prof[5] = clock64(); prof[7] = nsteps; }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 512;" ::"r"(tmem_base) : "memory");
    }
}

// Debug aid: SVRS_WG_PROF=1 makes every launch synchronous and prints the mean / max per-CTA phase times (cycles).
static void wg_prof_report(const WgParams& p, int grid, long long* dprof) {
    cudaDeviceSynchronize();
    long long* h = (long long*)malloc(sizeof(long long) * 8 * grid);
    cudaMemcpy(h, dprof, sizeof(long long) * 8 * grid, cudaMemcpyDeviceToHost);
    double sum[5] = {0, 0, 0, 0, 0}, mx[5] = {0, 0, 0, 0, 0};
    int live = 0;
    double ldsum = 0;
    for (int c = 0; c < grid; ++c) {
        const long long* t = h + 8 * c;
        if (t[7] <= 0) continue;
        ldsum += (double)t[6];
        ++live;
        double d[5] = {(double)(t[1] - t[0]), (double)(t[2] - t[1]), (double)(t[3] - t[2]), (double)(t[4] - t[3]), (double)(t[5] - t[4])};
        for (int i = 0; i < 5; ++i) { sum[i] += d[i]; if (d[i] > mx[i]) mx[i] = d[i]; }
    }
    fprintf(stderr, "[wgrad_tc] grid %d live %d ksplit %d ksteps %d group %d n_tile %d cwx %d cwg %d | cycles mean(max): setup %.0f(%.0f) "
            "first-load %.0f(%.0f) mma-issue %.0f(%.0f) mma-drain %.0f(%.0f) epilogue %.0f(%.0f) of which tmem-ld %.0f\n", grid, live, p.ksplit,
            p.ksteps_total, p.group, p.n_tile, p.cwx, p.cwg, sum[0] / live, mx[0], sum[1] / live, mx[1], sum[2] / live, mx[2],
            sum[3] / live, mx[3], sum[4] / live, mx[4], ldsum / live);
    free(h);
    cudaFree(dprof);
}

bool wgrad_tc_supported(int dtype, int Ca, int Cb, int OW, int OH) {
    int bw, bh, bn;
    // Ca, Cb: multiples of 8 (16-byte rows for the TMA maps), at least 16 (see chunk_width); G / X boxes past Ca / Cb are
    // zero-filled (see wg_plan)
    return dtype == SVRS_BF16 && Ca >= 16 && Ca % 8 == 0 && chunk_width(Cb) != 0 && pick_box(OW, OH, bw, bh, bn);
}

// Tiling / split plan of one launch (everything except the tensor maps).  The pixel split is exact - every split owns at
// least one k-step - because in packed mode each split writes a whole slab that the reduction later reads.
static int wg_plan(const TapGeom& g, int KK, WgParams& p) {
    memset(&p, 0, sizeof(p));
    if (!pick_box(g.OW, g.OH, p.BW, p.BH, p.BNI)) { set_error("wgrad_tc: unsupported spatial dims"); return SVRS_E_UNSUPPORTED; }
    p.N = g.N; p.OH = g.OH; p.OW = g.OW;
    p.tiles_x = g.OW / p.BW; p.tiles_y = g.OH / p.BH; p.tiles_n = (g.N + p.BNI - 1) / p.BNI;
    p.Ca = g.Nc; p.Cb = g.K; p.KK = KK;
    // G boxes: one box of 16 / 32 / 64 columns covering Ca <= 64, otherwise 128-column tiles of two 64-column boxes.  Ca = 16,
    // 32 and multiples of 64 fill their boxes; other multiples of 8 leave zero-filled columns in the last box.
    p.cwg = p.Ca <= 16 ? 16 : (p.Ca <= 32 ? 32 : 64);
    p.n_tile = p.Ca <= 64 ? p.cwg : 128;
    p.n_tiles = (p.Ca + p.n_tile - 1) / p.n_tile;
    p.cwx = chunk_width(p.Cb);
    p.cb_chunks = (p.Cb + p.cwx - 1) / p.cwx;
    p.bpb = 128 / p.cwx;
    const Prob& pb = g.prob[0];
    p.ntaps = pb.ntaps;
    p.nboxes = pb.ntaps * p.cb_chunks;
    p.nblocks = (p.nboxes + p.bpb - 1) / p.bpb;
    // M-blocks per CTA: as many accumulator blocks as TMEM holds (512 / n_tile columns).  MEASURED (SVRS_WG_GROUP A/B,
    // SVRS_WG_PROF): on the 4x4 / 8x8 maps the TMA-reduce epilogue (group x 64 KB per CTA at ~20 B/clk/SM, the chip's
    // fp32 L2-reduction rate) is 2-4x longer than the MMA phase, yet ONE block per CTA (a quarter of the reduction traffic,
    // same operand loads) was 1.5x SLOWER overall (wgrad_tc 1.04 -> 1.53 ms per step): twice the CTAs, each paying the
    // ~2 us first-load latency, and multi-wave grids on the 1024->512 layers.
    static const int group_env = [] { const char* e = getenv("SVRS_WG_GROUP"); return e ? atoi(e) : 0; }();
    p.group = group_env > 0 ? group_env : 512 / p.n_tile;
    if (p.group > 512 / p.n_tile) p.group = 512 / p.n_tile;
    if (p.group > WG_MAX_GROUP) p.group = WG_MAX_GROUP;
    if (p.group > p.nblocks) p.group = p.nblocks;
    p.ngroups = (p.nblocks + p.group - 1) / p.group;
    p.ksteps_total = p.tiles_x * p.tiles_y * p.tiles_n;
    int base = p.ngroups * p.n_tiles;
    // split-K over pixels until about HALF the SMs have a CTA.  MEASURED (SVRS_WG_TARGET_CTAS sweep on the bench step): a
    // target of 148 CTAs costs 3 % of the whole step against 60-74 - every extra split pays another TMA-reduce epilogue
    // (group x 64 KB through the L2 fp32 adder) and the weight gradients run on side streams next to the dgrad chain, so a
    // grid that takes every SM only queues behind (or in front of) the kernel it is supposed to overlap with.
    static const int target = getenv("SVRS_WG_TARGET_CTAS") ? atoi(getenv("SVRS_WG_TARGET_CTAS")) : num_sms() / 2;
    int ksplit = (target + base / 2) / base;
    // every split pays the fixed costs again (first load ~4 k cycles, TMA-reduce epilogue of group x 64 KB ~10 k cycles): a CTA
    // should own at least a few 128-pixel steps of MMA work
    static const int min_ksteps = getenv("SVRS_WG_MIN_KSTEPS") ? atoi(getenv("SVRS_WG_MIN_KSTEPS")) : 4;     // measured on the bench step: 1 -> 4 = -0.9 %, 16 = +4 %
    if (ksplit > p.ksteps_total / min_ksteps) ksplit = p.ksteps_total / min_ksteps;
    if (ksplit > p.ksteps_total) ksplit = p.ksteps_total;
    if (ksplit < 1) ksplit = 1;
    const int steps_per = (p.ksteps_total + ksplit - 1) / ksplit;
    p.ksplit = (p.ksteps_total + steps_per - 1) / steps_per;
    return 0;
}

int wgrad_tc_splits(const TapGeom& g, int KK) {
    WgParams p;
    return wg_plan(g, KK, p) ? 0 : p.ksplit;
}

// g: geometry of the forward-form conv whose output grid carries `gmat` (channels Ca = g.Nc) and whose input view
// carries `x` (channels Cb = g.K);  dw torch layout [(a*Cb + b)*KK + tap]
int launch_wgrad_tc(const TapGeom& g, const void* gmat, const void* x, float* dw, int packed, int KK, float* db, cudaStream_t st) {
    static bool attr_set = false;
    if (!attr_set) {
        cudaError_t e = cudaFuncSetAttribute(wgrad_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, WG_SMEM_BYTES);
        if (e != cudaSuccess) { set_error("wgrad_tc: cudaFuncSetAttribute: %s", cudaGetErrorString(e)); return SVRS_E_CUDA; }
        attr_set = true;
    }
    WgParams p;
    if (int rc = wg_plan(g, KK, p)) return rc;
    p.dw = dw;
    p.packed = packed;
    const Prob& pb = g.prob[0];
    p.db = db;
    p.gptr = reinterpret_cast<const __nv_bfloat16*>(gmat) + pb.out_off;
    p.g_sn = g.o_sn; p.g_sy = g.o_sy; p.g_sx = g.o_sx;
    long long offs[4]; int nmaps = 0;
    for (int t = 0; t < pb.ntaps; ++t) {
        const Tap& tp = pb.taps[t];
        int mi = -1;
        for (int i = 0; i < nmaps; ++i) if (offs[i] == tp.in_off) mi = i;
        if (mi < 0) { if (nmaps == 4) { set_error("wgrad_tc: too many input views"); return SVRS_E_ARG; } offs[nmaps] = tp.in_off; mi = nmaps++; }
        p.taps[t].map = mi; p.taps[t].dy = tp.dy; p.taps[t].dx = tp.dx; p.taps[t].tapid = t;
    }
    const __nv_bfloat16* xb = reinterpret_cast<const __nv_bfloat16*>(x);
    for (int i = 0; i < 4; ++i) {
        long long off = i < nmaps ? offs[i] : offs[0];
        int rc = make_act_map(&p.x_maps[i], xb + off, p.Cb, g.IW, g.IH, g.N, g.i_sx, g.i_sy, g.i_sn, p.BW, p.BH, p.BNI, p.cwx);
        if (rc) return rc;
    }
    const __nv_bfloat16* gb = reinterpret_cast<const __nv_bfloat16*>(gmat) + pb.out_off;
    int rc = make_act_map(&p.g_map, gb, p.Ca, g.OW, g.OH, g.N, g.o_sx, g.o_sy, g.o_sn, p.BW, p.BH, p.BNI, p.cwg);
    if (rc) return rc;

    if (packed) {
        rc = make_f32_3d_map(&p.dw_map, dw, p.Ca, p.Cb, KK, p.n_tile < 32 ? p.n_tile : 32, p.cwx);
        if (rc) return rc;
    }

    int grid = p.ngroups * p.n_tiles * p.ksplit;
    static const bool prof_on = getenv("SVRS_WG_PROF") != nullptr;
    if (prof_on) {
        cudaMalloc(&p.prof, sizeof(long long) * 8 * grid);
        cudaMemset(p.prof, 0, sizeof(long long) * 8 * grid);
    }
    SVRS_LAUNCH((wgrad_tc_kernel), grid, WG_THREADS, WG_SMEM_BYTES, st, p);
    if (prof_on) wg_prof_report(p, grid, p.prof);
    return check_launch("wgrad_tc_kernel");
}

}  // namespace svrs
