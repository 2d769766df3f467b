// conv_tc.cu - tcgen05 / TMEM / TMA implicit-GEMM convolution for sm_100a (bf16 in, fp32 accumulate in TMEM).
//
// One persistent, warp-specialised kernel runs every "multi-tap GEMM" conv form of taps.cuh
// (k3s1 fprop/dgrad, k4s2 fprop/dgrad, transposed k4s2 fprop/dgrad):
//
//   D[128 output pixels, n_tile channels] = sum over taps t, cw-channel chunks c
//        A_t,c [128 pixels shifted by (dy_t, dx_t), cw ch]  x  W_t,c [n_tile, cw ch]^T
//
//   * A tiles are fetched by TMA from the NHWC activation tensor with a 4-D box
//     (cw ch, BW, BH, BN images; BW*BH*BN = 128) whose start coordinate carries the tap shift;
//     out-of-range rows/columns are ZERO-FILLED by the TMA unit, which implements the conv padding.
//     Stride-2 forms read through one of four "parity" tensor maps (element stride 2 in W and H).
//   * the channel chunk cw is 64, 32 or 16 (reduction channels % 64 / 32 / 16 == 0): rows of 128 / 64 / 32 bytes
//     in the matching SWIZZLE_128B / 64B / 32B K-major layout (8-row groups 1024 / 512 / 256 B apart), consumed
//     directly by tcgen05.mma (M=128, N=n_tile, K=16) through shared-memory descriptors.  For cw < 64 a pipeline
//     stage carries 64/cw (tap, chunk) pairs so a stage always moves ~16 KB of activations.
//     Reduction channels that are a multiple of 8 but not of 16 (16-byte rows, e.g. 168 / 424) take ceil(K / cw) chunks
//     of cw = 64 (or the narrowest of 16 / 32 / 64 covering K <= 64): both tensor maps keep the true K as their inner
//     dimension, so the channels past K in the last box arrive as TMA zero fill in A and B and add nothing.
//   * accumulators live in TMEM (2 stages x 256 columns) so the epilogue of tile i overlaps the
//     main loop of tile i+1; the epilogue (4 warps) does tcgen05.ld -> +bias -> activation -> bf16 ->
//     128-bit global stores, one output pixel (row) per thread.  Output channels are padded to a multiple of 16
//     for the MMA (weight rows beyond Nc are TMA zero fill) and masked at the store.
//   * warp roles: warp 0 = TMA producer, warp 1 = TMEM allocator + MMA issuer, warps 2..5 = epilogue.
#include "common.cuh"
#include <stdlib.h>
#include "taps.cuh"
#include <cuda.h>
#include <string.h>
#include "tc_ptx.cuh"

namespace svrs {

constexpr int TC_STAGES = 4;
constexpr int TC_A_BYTES = 128 * 128;        // 128 pixels x 64 bf16 (or 64/cw pairs of 128 x cw)
constexpr int TC_B_BYTES = 256 * 128;        // up to 256 output channels x 64 bf16
constexpr int TC_STAGE_BYTES = TC_A_BYTES + TC_B_BYTES;
constexpr int TC_SMEM_BYTES = TC_STAGES * TC_STAGE_BYTES + 1024 /*align*/ + 256 /*barriers*/;
constexpr int TC_THREADS = 64 + 32 * TC_EPI_WARPS;   // TMA warp + MMA warp + 8 epilogue warps

struct TcTap {
    int map;    // which input tensor map (parity class)
    int dy, dx; // shift of the box start
    int wtap;   // tap index in the packed weights
};
struct TcProb {
    int ntaps;
    int pad_;
    long long out_off;
    TcTap taps[16];
};
struct alignas(64) TcParams {
    CUtensorMap in_maps[4];
    CUtensorMap w_map;
    __nv_bfloat16* out;
    const float* bias;
    long long o_sn, o_sy, o_sx;
    int N, OH, OW;
    int BW, BH, BNI;
    int tiles_x, tiles_y, tiles_n;
    int Nc, n_tile, n_tiles, kchunks;
    int cw, tg;          // channel chunk width (16/32/64), (tap,chunk) pairs per pipeline stage (64/cw)
    int act, nprob;
    float* out2;             // optional fp32 NCHW-flat second output (see EpiRow), per-sample stride out2_ld
    long long out2_ld;
    double* bn_sums;         // optional BatchNorm statistics scratch (SVRS_BN_REPLICAS x double[2*Nc])
    TcProb prob[4];
};

// ------------------------------------------------------------------------------------------ kernel
template <bool EXTRA>
__global__ void __launch_bounds__(TC_THREADS, 1) conv_tc_kernel(const __grid_constant__ TcParams p) {
    pdl_entry();
    extern __shared__ uint8_t smem_raw[];
    const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
    const uint32_t bar_base = smem_base + TC_STAGES * TC_STAGE_BYTES;
    // barriers: full[4] empty[4] tmem_full[2] tmem_empty[2], then the TMEM base address slot
    auto full_bar = [&](int s) { return bar_base + 8u * s; };
    auto empty_bar = [&](int s) { return bar_base + 8u * (TC_STAGES + s); };
    auto tfull_bar = [&](int s) { return bar_base + 8u * (2 * TC_STAGES + s); };
    auto tempty_bar = [&](int s) { return bar_base + 8u * (2 * TC_STAGES + 2 + s); };
    const uint32_t tmem_slot = bar_base + 8u * (2 * TC_STAGES + 4);
    uint32_t* tmem_slot_ptr = reinterpret_cast<uint32_t*>(smem_raw + (tmem_slot - smem_u32(smem_raw)));

    const int warp = threadIdx.x / 32, lane = threadIdx.x % 32;
    __shared__ float s_bn[EXTRA ? 2 * EPI_BN_MAXC : 1];
    if (EXTRA && p.bn_sums) epi_bn_zero(s_bn);

    if (warp == 0 && lane == 0) {
        for (int i = 0; i < 4; ++i) prefetch_tmap(&p.in_maps[i]);
        prefetch_tmap(&p.w_map);
        for (int s = 0; s < TC_STAGES; ++s) { mbar_init(full_bar(s), 1); mbar_init(empty_bar(s), 1); }
        for (int s = 0; s < 2; ++s) { mbar_init(tfull_bar(s), 1); mbar_init(tempty_bar(s), TC_EPI_WARPS); }
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

    const int tiles_pix = p.tiles_x * p.tiles_y * p.tiles_n;
    const int tiles_per_prob = tiles_pix * p.n_tiles;
    const int total_tiles = tiles_per_prob * p.nprob;
    const uint32_t a_box = 128u * (uint32_t)p.cw * 2u;            // bytes of one activation box
    const uint32_t b_box = (uint32_t)p.n_tile * (uint32_t)p.cw * 2u;  // bytes of one weight box

    if (warp == 0) {
        // ================================ TMA producer ================================
        if (lane == 0) {
            uint32_t stage = 0, phase = 0;
            for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
                const int pr = tile / tiles_per_prob;
                int rem = tile % tiles_per_prob;
                const int nt = rem % p.n_tiles;
                int pt = rem / p.n_tiles;
                const int tx = pt % p.tiles_x; pt /= p.tiles_x;
                const int ty = pt % p.tiles_y;
                const int tn = pt / p.tiles_y;
                const int x0 = tx * p.BW, y0 = ty * p.BH, n0 = tn * p.BNI;
                const TcProb& pb = p.prob[pr];
                const int npairs = pb.ntaps * p.kchunks;
                for (int i0 = 0; i0 < npairs; i0 += p.tg) {
                    const int cnt = (npairs - i0) < p.tg ? (npairs - i0) : p.tg;
                    mbar_wait(empty_bar(stage), phase ^ 1u);
                    const uint32_t sa = smem_base + stage * TC_STAGE_BYTES;
                    mbar_expect_tx(full_bar(stage), (uint32_t)cnt * (a_box + b_box));
                    for (int j = 0; j < cnt; ++j) {
                        const int t = (i0 + j) / p.kchunks, kc = (i0 + j) % p.kchunks;
                        const TcTap tp = pb.taps[t];
                        tma_load_4d(sa + j * a_box, &p.in_maps[tp.map], full_bar(stage), kc * p.cw, x0 + tp.dx, y0 + tp.dy, n0);
                        tma_load_3d(sa + TC_A_BYTES + j * b_box, &p.w_map, full_bar(stage), kc * p.cw, nt * p.n_tile, tp.wtap);
                    }
                    if (++stage == TC_STAGES) { stage = 0; phase ^= 1u; }
                }
            }
        }
    } else if (warp == 1) {
        // ================================ MMA issuer (one thread; issue-bound, see tc_ptx.cuh) ================================
        if (lane == 0) {
            // instruction descriptor: D=f32, A=B=bf16, both K-major, N = n_tile, M = 128
            const uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(p.n_tile >> 3) << 17) | ((128u >> 4) << 24);
            const uint32_t ltype = p.cw == 64 ? 2u : (p.cw == 32 ? 4u : 6u);         // SWIZZLE_128B / 64B / 32B
            const uint32_t hi = desc_hi(16u * (uint32_t)p.cw, ltype);                // SBO = 8 rows x (cw * 2 B)
            const uint32_t a_box16 = a_box >> 4, b_box16 = b_box >> 4;
            const int ksub = p.cw / 16;
            uint32_t stage = 0, phase = 0, acc = 0, acc_phase = 0;
            for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
                const int pr = tile / tiles_per_prob;
                const int npairs = p.prob[pr].ntaps * p.kchunks;
                mbar_wait(tempty_bar(acc), acc_phase ^ 1u);
                tc_fence_after();
                const uint32_t d_tmem = tmem_base + acc * 256u;
                for (int i0 = 0; i0 < npairs; i0 += p.tg) {
                    const int cnt = (npairs - i0) < p.tg ? (npairs - i0) : p.tg;
                    mbar_wait(full_bar(stage), phase);
                    tc_fence_after();
                    const uint32_t sa = smem_base + stage * TC_STAGE_BYTES;
                    uint32_t a_lo = desc_lo(sa, 16u), b_lo = desc_lo(sa + TC_A_BYTES, 16u);
                    if (ksub == 4) {                 // cw = 64: one pair per stage, 4 K-steps
#pragma unroll
                        for (int k = 0; k < 4; ++k)
                            tc_mma_lohi(d_tmem, a_lo + 2u * k, hi, b_lo + 2u * k, hi, idesc, k ? 1u : (uint32_t)(i0 != 0));
                    } else {
                        for (int j = 0; j < cnt; ++j) {
                            for (int k = 0; k < ksub; ++k)
                                tc_mma_lohi(d_tmem, a_lo + 2u * k, hi, b_lo + 2u * k, hi, idesc, (uint32_t)((i0 | j | k) != 0));
                            a_lo += a_box16;
                            b_lo += b_box16;
                        }
                    }
                    tc_commit(empty_bar(stage));                          // frees the smem stage when these MMAs retire
                    if (i0 + cnt >= npairs) tc_commit(tfull_bar(acc));    // accumulator complete -> epilogue
                    if (++stage == TC_STAGES) { stage = 0; phase ^= 1u; }
                }
                if (++acc == 2) { acc = 0; acc_phase ^= 1u; }
            }
        }
    } else {
        // ================================ epilogue (8 warps) ================================
        const int q = warp % 4;                         // TMEM lane quarter this warp may access
        const int half = (warp - 2) / 4;                // which half of the tile's column chunks
        const int r = q * 32 + lane;                    // accumulator row == pixel within the tile
        const int ix = r % p.BW, iy = (r / p.BW) % p.BH, in = r / (p.BW * p.BH);
        uint32_t acc = 0, acc_phase = 0;
        for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
            const int pr = tile / tiles_per_prob;
            int rem = tile % tiles_per_prob;
            const int nt = rem % p.n_tiles;
            int pt = rem / p.n_tiles;
            const int tx = pt % p.tiles_x; pt /= p.tiles_x;
            const int ty = pt % p.tiles_y;
            const int tn = pt / p.tiles_y;
            const int n = tn * p.BNI + in;
            const int c_base = nt * p.n_tile;
            __nv_bfloat16* orow = p.out + p.prob[pr].out_off + (long long)n * p.o_sn +
                                  (long long)(ty * p.BH + iy) * p.o_sy + (long long)(tx * p.BW + ix) * p.o_sx + c_base;
            mbar_wait(tfull_bar(acc), acc_phase);
            tc_fence_after();
            const uint32_t taddr = tmem_base + acc * 256u + ((uint32_t)(q * 32) << 16);
            EpiRow er;
            er.o2 = nullptr; er.hw = 0; er.sbn = nullptr;
            if (EXTRA) {
                er.o2 = p.out2 ? p.out2 + (long long)n * p.out2_ld + (long long)(ty * p.BH + iy) * p.OW + (tx * p.BW + ix) : nullptr;
                er.hw = p.OH * p.OW;
                er.sbn = p.bn_sums ? s_bn : nullptr;
            }
            epi_dispatch<EXTRA>(p.act, taddr, p.n_tile, half, (!EXTRA || p.out) ? orow : nullptr, p.bias, c_base, p.Nc, n < p.N, er);
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(tempty_bar(acc));
            if (++acc == 2) { acc = 0; acc_phase ^= 1u; }
        }
        if (EXTRA && p.bn_sums) epi_bn_flush(s_bn, p.bn_sums, p.Nc, threadIdx.x - 64, 32 * TC_EPI_WARPS);
    }

    tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 512;" ::"r"(tmem_base) : "memory");
    }
}

// ------------------------------------------------------------------------------------------ host side
typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                    const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                    CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static PFN_encodeTiled get_encode() {
    static PFN_encodeTiled fn = nullptr;
    if (!fn) {
        void* ptr = nullptr;
        cudaDriverEntryPointQueryResult qres;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &qres) == cudaSuccess && qres == cudaDriverEntryPointSuccess)
            fn = (PFN_encodeTiled)ptr;
    }
    return fn;
}

static CUtensorMapSwizzle swizzle_for(int cw) {
    return cw == 64 ? CU_TENSOR_MAP_SWIZZLE_128B : (cw == 32 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_32B);
}

// Channel chunk of a tcgen05 operand with C channels: the widest of 64 / 32 / 16 dividing C; for C % 16 != 0 with 16-byte
// rows (C % 8 == 0) the last chunk is ragged: 64 when C > 64, otherwise the narrowest width covering C.  0 = unsupported:
// rows that are not 16-byte multiples (no TMA map describes them), and C = 8, which would fill half of every MMA with zero
// fill - 8-channel operands stay on the CUDA-core kernels, no measurement shows the tensor cores winning there.
int chunk_width(int C) {
    if (C % 16 == 0) return C % 64 == 0 ? 64 : (C % 32 == 0 ? 32 : 16);
    if (C % 8 != 0 || C < 24) return 0;
    return C > 32 ? 64 : (C > 16 ? 32 : 16);
}

// 4-D activation view map: dims (C, W, H, N) with arbitrary element strides for W/H/N; box (cw, BW, BH, BNI)
int make_act_map(CUtensorMap* m, const void* base, int C, int W, int H, int N, long long sx, long long sy, long long sn,
                 int BW, int BH, int BNI, int cw) {
    PFN_encodeTiled enc = get_encode();
    if (!enc) { set_error("cuTensorMapEncodeTiled unavailable"); return SVRS_E_CUDA; }
    cuuint64_t dims[4] = {(cuuint64_t)C, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)N};
    cuuint64_t strides[3] = {(cuuint64_t)sx * 2, (cuuint64_t)sy * 2, (cuuint64_t)sn * 2};
    cuuint32_t box[4] = {(cuuint32_t)cw, (cuuint32_t)BW, (cuuint32_t)BH, (cuuint32_t)BNI};
    cuuint32_t es[4] = {1, 1, 1, 1};
    CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, const_cast<void*>(base), dims, strides, box, es,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, swizzle_for(cw), CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) { set_error("cuTensorMapEncodeTiled(activation) failed: %d (C=%d W=%d H=%d N=%d cw=%d)", (int)r, C, W, H, N, cw); return SVRS_E_CUDA; }
    return 0;
}

int make_f32_2d_map(CUtensorMap* m, const void* base, long long inner, long long rows, int box_inner, int box_rows) {
    PFN_encodeTiled enc = get_encode();
    if (!enc) { set_error("cuTensorMapEncodeTiled unavailable"); return SVRS_E_CUDA; }
    cuuint64_t dims[2] = {(cuuint64_t)inner, (cuuint64_t)rows};
    cuuint64_t strides[1] = {(cuuint64_t)inner * 4};
    cuuint32_t box[2] = {(cuuint32_t)box_inner, (cuuint32_t)box_rows};
    cuuint32_t es[2] = {1, 1};
    CUtensorMapSwizzle sw = box_inner * 4 == 128 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B;
    CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<void*>(base), dims, strides, box, es,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, sw, CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) { set_error("cuTensorMapEncodeTiled(f32 2d) failed: %d (inner=%lld rows=%lld box %dx%d)", (int)r, inner, rows, box_inner, box_rows); return SVRS_E_CUDA; }
    return 0;
}

// fp32 [d2][d1][d0] (d0 contiguous), box (box0 = 32 or 16 columns, box1 rows, 1): the per-tap packed gradient seen with its
// true extents, so a box that reaches past d0 or d1 is clipped by TMA instead of spilling into the next tap
int make_f32_3d_map(CUtensorMap* m, const void* base, long long d0, long long d1, long long d2, int box0, int box1) {
    PFN_encodeTiled enc = get_encode();
    if (!enc) { set_error("cuTensorMapEncodeTiled unavailable"); return SVRS_E_CUDA; }
    cuuint64_t dims[3] = {(cuuint64_t)d0, (cuuint64_t)d1, (cuuint64_t)d2};
    cuuint64_t strides[2] = {(cuuint64_t)d0 * 4, (cuuint64_t)(d0 * d1) * 4};
    cuuint32_t box[3] = {(cuuint32_t)box0, (cuuint32_t)box1, 1};
    cuuint32_t es[3] = {1, 1, 1};
    CUtensorMapSwizzle sw = box0 * 4 == 128 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B;
    CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, const_cast<void*>(base), dims, strides, box, es,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, sw, CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) { set_error("cuTensorMapEncodeTiled(f32 3d) failed: %d (%lld x %lld x %lld box %dx%d)", (int)r, d0, d1, d2, box0, box1); return SVRS_E_CUDA; }
    return 0;
}

// weights in NK pack [tap][Nc][K] (K contiguous): dims (K, Nc, taps), box (cw, n_tile, 1)
static int make_w_map(CUtensorMap* m, const void* base, int K, int Nc, int taps, int n_tile, int cw) {
    PFN_encodeTiled enc = get_encode();
    if (!enc) { set_error("cuTensorMapEncodeTiled unavailable"); return SVRS_E_CUDA; }
    cuuint64_t dims[3] = {(cuuint64_t)K, (cuuint64_t)Nc, (cuuint64_t)taps};
    cuuint64_t strides[2] = {(cuuint64_t)K * 2, (cuuint64_t)K * Nc * 2};
    cuuint32_t box[3] = {(cuuint32_t)cw, (cuuint32_t)n_tile, 1};
    cuuint32_t es[3] = {1, 1, 1};
    CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, const_cast<void*>(base), dims, strides, box, es,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, swizzle_for(cw), CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) { set_error("cuTensorMapEncodeTiled(weights) failed: %d (K=%d Nc=%d taps=%d)", (int)r, K, Nc, taps); return SVRS_E_CUDA; }
    return 0;
}

// image planes [planes][S][S] of 2- or 4-byte elements (no swizzle): dims (S, S, planes), box (box_w, box_h, box_c)
int make_plane_map_3d(CUtensorMap* m, const void* base, int elem_bytes, int S, long long planes, int box_w, int box_h, int box_c) {
    PFN_encodeTiled enc = get_encode();
    if (!enc) { set_error("cuTensorMapEncodeTiled unavailable"); return SVRS_E_CUDA; }
    cuuint64_t dims[3] = {(cuuint64_t)S, (cuuint64_t)S, (cuuint64_t)planes};
    cuuint64_t strides[2] = {(cuuint64_t)S * elem_bytes, (cuuint64_t)S * S * elem_bytes};
    cuuint32_t box[3] = {(cuuint32_t)box_w, (cuuint32_t)box_h, (cuuint32_t)box_c};
    cuuint32_t es[3] = {1, 1, 1};
    CUresult r = enc(m, elem_bytes == 4 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32 : CU_TENSOR_MAP_DATA_TYPE_UINT16, 3, const_cast<void*>(base),
                     dims, strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE,
                     CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) { set_error("cuTensorMapEncodeTiled(planes) failed: %d (S=%d planes=%lld box %dx%dx%d)", (int)r, S, planes, box_w, box_h, box_c); return SVRS_E_CUDA; }
    return 0;
}

int make_w_map_pub(CUtensorMap* m, const void* base, int K, int Nc, int taps, int n_tile, int cw) {
    return make_w_map(m, base, K, Nc, taps, n_tile, cw);
}
bool halo_supported(int form, int Cr, int Cw, int OW, int OH);
bool convT_halo_supported(int Cr, int Cw, int W, int H);
int launch_convT_halo(const void* in, const void* w_nk, const float* bias, void* out, int N, int H, int W, int Cr, int Cw, int act,
                      const ConvExtra& ex, cudaStream_t st);
int launch_conv3_halo(int form, const void* in, const void* w_nk, const float* bias, void* out, int N, int H, int W, int Cr, int Cw,
                      int act, const ConvExtra& ex, cudaStream_t st);

bool pick_box(int OW, int OH, int& BW, int& BH, int& BNI) {
    BW = OW < 128 ? OW : 128;
    if (128 % BW || OW % BW) return false;
    BH = 128 / BW;
    if (BH > OH) BH = OH;
    if (OH % BH) return false;
    BNI = 128 / (BW * BH);
    return BW * BH * BNI == 128 && BW <= 256 && BH <= 256 && BNI <= 256;
}

bool tc_supported(int dtype, int K, int Nc, int OW, int OH) {
    int bw, bh, bn;
    // K % 8: 16-byte rows for the TMA maps (a ragged last chunk is zero-filled up to the UMMA K of 16, see chunk_width);
    // Nc % 4: 8-byte aligned output rows (N is padded to 16 for the MMA)
    return dtype == SVRS_BF16 && chunk_width(K) != 0 && Nc % 4 == 0 && Nc >= 4 && pick_box(OW, OH, bw, bh, bn);
}

// form: 0 conv3 fprop, 1 conv3 dgrad, 2 conv4s2 (strided read), 3 convT4s2 (strided write).
// in: tensor being read [N, H, W, Cr] ; out: tensor written ; w_nk: NK pack [tap][Cw][Cr]
int launch_conv_tc(int form, const void* in, const void* w_nk, const float* bias, void* out, int N, int H, int W, int Cr, int Cw,
                   int act, const ConvExtra& ex, cudaStream_t st) {
    if (ex.bn_sums && Cw > EPI_BN_MAXC) { set_error("conv_tc: fused BatchNorm statistics need Cout <= %d", EPI_BN_MAXC); return SVRS_E_UNSUPPORTED; }
    if (ex.out2 && form == 3) { set_error("conv_tc: NCHW second output is not available for the transposed form"); return SVRS_E_UNSUPPORTED; }
    if ((ex.out2 || ex.bn_sums) && (act == SVRS_ACT_SIGMOID || (act == SVRS_ACT_HARDTANH7 && !bias))) {
        set_error("conv_tc: epilogue extras support no activation or bias + Hardtanh only");
        return SVRS_E_UNSUPPORTED;
    }
    if (halo_supported(form, Cr, Cw, W, H)) return launch_conv3_halo(form, in, w_nk, bias, out, N, H, W, Cr, Cw, act, ex, st);
    if (form == 3 && convT_halo_supported(Cr, Cw, W, H)) return launch_convT_halo(in, w_nk, bias, out, N, H, W, Cr, Cw, act, ex, st);
    static bool attr_set = false;
    if (!attr_set) {
        cudaError_t e = cudaFuncSetAttribute(conv_tc_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, TC_SMEM_BYTES);
        if (e == cudaSuccess) e = cudaFuncSetAttribute(conv_tc_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, TC_SMEM_BYTES);
        if (e != cudaSuccess) { set_error("conv_tc: cudaFuncSetAttribute: %s", cudaGetErrorString(e)); return SVRS_E_CUDA; }
        attr_set = true;
    }
    TapGeom g;
    int ntaps_total;
    if (form == 0) { geom_conv3(g, N, H, W, Cr, Cw, false); ntaps_total = 9; }
    else if (form == 1) { geom_conv3(g, N, H, W, Cr, Cw, true); ntaps_total = 9; }
    else if (form == 2) { geom_conv4s2(g, N, H, W, Cr, Cw); ntaps_total = 16; }
    else { geom_convT4s2(g, N, H, W, Cr, Cw); ntaps_total = 16; }

    TcParams p;
    memset(&p, 0, sizeof(p));
    if (!pick_box(g.OW, g.OH, p.BW, p.BH, p.BNI)) { set_error("conv_tc: unsupported spatial dims %dx%d", g.OW, g.OH); return SVRS_E_UNSUPPORTED; }
    p.out = reinterpret_cast<__nv_bfloat16*>(out);
    p.bias = bias;
    p.out2 = ex.out2; p.out2_ld = ex.out2_ld; p.bn_sums = ex.bn_sums;
    p.o_sn = g.o_sn; p.o_sy = g.o_sy; p.o_sx = g.o_sx;
    p.N = N; p.OH = g.OH; p.OW = g.OW;
    p.tiles_x = g.OW / p.BW; p.tiles_y = g.OH / p.BH; p.tiles_n = (N + p.BNI - 1) / p.BNI;
    p.Nc = Cw;
    int npad = (Cw + 15) / 16 * 16;
    p.n_tile = npad <= 256 ? npad : 256;
    // few pixel tiles (4x4 / 8x8 maps): trade MMA width for CTAs only while fewer than `want` CTAs would have work.
    {
        long long pix_tiles = (long long)p.tiles_x * p.tiles_y * p.tiles_n * g.nprob;
        // Measured (bench step, 128 patches): shrinking N for >= 96 CTAs cost 6.6 % of the whole step against >= 32 - on the
        // 4x4 / 8x8 maps a CTA's time is dominated by the weight stream and the ~58-cycle MMA issue floor, so 64 CTAs issuing
        // N = 128 / 256 MMAs beat 128 CTAs issuing N = 64 MMAs, and leave SMs to the kernels of the parallel streams.
        static const int want = getenv("SVRS_TC_WANT_CTAS") ? atoi(getenv("SVRS_TC_WANT_CTAS")) : 32;
        while (p.n_tile > 64 && p.n_tile % 32 == 0 && pix_tiles * ((Cw + p.n_tile - 1) / p.n_tile) < want) p.n_tile /= 2;
    }
    p.n_tiles = (Cw + p.n_tile - 1) / p.n_tile;
    p.cw = chunk_width(Cr);
    p.tg = 64 / p.cw;
    p.kchunks = (Cr + p.cw - 1) / p.cw;      // the last chunk may be ragged: TMA zero-fills its channels past Cr
    p.act = act; p.nprob = g.nprob;

    // input maps: distinct in_off values become distinct tensor maps (parity classes of a stride-2 read)
    long long offs[4]; int nmaps = 0;
    for (int pr = 0; pr < g.nprob; ++pr) {
        p.prob[pr].ntaps = g.prob[pr].ntaps;
        p.prob[pr].out_off = g.prob[pr].out_off;
        for (int t = 0; t < g.prob[pr].ntaps; ++t) {
            const Tap& tp = g.prob[pr].taps[t];
            int mi = -1;
            for (int i = 0; i < nmaps; ++i) if (offs[i] == tp.in_off) mi = i;
            if (mi < 0) { if (nmaps == 4) { set_error("conv_tc: too many input views"); return SVRS_E_ARG; } offs[nmaps] = tp.in_off; mi = nmaps++; }
            TcTap& o = p.prob[pr].taps[t];
            o.map = mi; o.dy = tp.dy; o.dx = tp.dx;
            o.wtap = (int)(tp.w_off / ((long long)Cr * Cw));
        }
    }
    const __nv_bfloat16* inb = reinterpret_cast<const __nv_bfloat16*>(in);
    for (int i = 0; i < 4; ++i) {
        long long off = i < nmaps ? offs[i] : offs[0];
        int rc = make_act_map(&p.in_maps[i], inb + off, Cr, g.IW, g.IH, N, g.i_sx, g.i_sy, g.i_sn, p.BW, p.BH, p.BNI, p.cw);
        if (rc) return rc;
    }
    int rc = make_w_map(&p.w_map, w_nk, Cr, Cw, ntaps_total, p.n_tile, p.cw);
    if (rc) return rc;

    long long total = (long long)p.tiles_x * p.tiles_y * p.tiles_n * p.n_tiles * p.nprob;
    int grid = (int)(total < num_sms() ? total : num_sms());
    if (grid < 1) return 0;
    if (ex.out2 || ex.bn_sums) SVRS_LAUNCH((conv_tc_kernel<true>), grid, TC_THREADS, TC_SMEM_BYTES, st, p);
    else SVRS_LAUNCH((conv_tc_kernel<false>), grid, TC_THREADS, TC_SMEM_BYTES, st, p);
    return check_launch("conv_tc_kernel");
}

}  // namespace svrs
