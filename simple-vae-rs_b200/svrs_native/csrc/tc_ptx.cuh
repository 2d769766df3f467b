// tc_ptx.cuh - inline-PTX wrappers shared by the tcgen05 kernels (conv_tc.cu, wgrad_tc.cu): mbarrier, TMA bulk tensor
// loads, tcgen05.mma / commit / ld / fences, and shared-memory matrix descriptors.
#pragma once
#include <cuda.h>
#include <stdint.h>

namespace svrs {

// ------------------------------------------------------------------------------------------ PTX wrappers
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    asm volatile(
        "{\n\t"
        ".reg .pred P1;\n\t"
        "WAIT_LOOP:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n\t"
        "@P1 bra DONE;\n\t"
        "bra WAIT_LOOP;\n\t"
        "DONE:\n\t"
        "}" ::"r"(bar), "r"(parity)
        : "memory");
}
__device__ __forceinline__ void tma_load_4d(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1, int c2, int c3) {
    asm volatile(
        "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
        ::"r"(dst), "l"(map), "r"(bar), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
        : "memory");
}
__device__ __forceinline__ void tma_load_3d(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1, int c2) {
    asm volatile(
        "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
        ::"r"(dst), "l"(map), "r"(bar), "r"(c0), "r"(c1), "r"(c2)
        : "memory");
}
// ---- TMA tensor reduction (shared -> global, element-wise add done by L2) and bulk-group bookkeeping --------------
__device__ __forceinline__ void tma_reduce_add_2d(const CUtensorMap* map, uint32_t src, int c0, int c1) {
    asm volatile("cp.reduce.async.bulk.tensor.2d.global.shared::cta.add.tile.bulk_group [%0, {%2, %3}], [%1];"
                 ::"l"(map), "r"(src), "r"(c0), "r"(c1)
                 : "memory");
}
__device__ __forceinline__ void tma_reduce_add_3d(const CUtensorMap* map, uint32_t src, int c0, int c1, int c2) {
    asm volatile("cp.reduce.async.bulk.tensor.3d.global.shared::cta.add.tile.bulk_group [%0, {%2, %3, %4}], [%1];"
                 ::"l"(map), "r"(src), "r"(c0), "r"(c1), "r"(c2)
                 : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_read_1() { asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void named_bar_sync(int id, int nthreads) {
    asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}
__device__ __forceinline__ void st_shared_v4(uint32_t addr, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
    asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}
// ---- bias gradient folded into the wgrad kernels ---------------------------------------------------------------------
// The four epilogue warps are idle while the MMA warp runs the pixel loop; they use that time to sum the CTA's G (= dy)
// tiles over pixels straight from global memory (the same lines TMA is pulling through L2): thread = (8-channel group q,
// pixel lane), 16-byte loads.  `acc` holds the thread's 8 partial channel sums.
__device__ __forceinline__ void colsum_tile8(const __nv_bfloat16* __restrict__ g, long long sn, long long sy, long long sx,
                                             int n0, int y0, int x0, int BW, int BH, int BNI, int N, int c0,
                                             int lane, int lanes, float* acc) {
    const int npix = BW * BH * BNI;
    // four independent 16-byte loads in flight per thread (the loop used to issue one at a time: on the weight-heavy 4x4
    // layers the few CTAs that fold the bias gradient then finished 30 us after everyone else - SVRS_WG_PROF "drain" max)
    for (int i0 = lane; i0 < npix; i0 += 4 * lanes) {
        uint4 r[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int i = i0 + u * lanes;
            const int bx = i % BW, by = (i / BW) % BH, n = n0 + i / (BW * BH);
            r[u] = make_uint4(0u, 0u, 0u, 0u);
            if (i < npix && n < N)
                r[u] = __ldg(reinterpret_cast<const uint4*>(g + (long long)n * sn + (long long)(y0 + by) * sy + (long long)(x0 + bx) * sx + c0));
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const uint32_t w[4] = {r[u].x, r[u].y, r[u].z, r[u].w};
#pragma unroll
            for (int j = 0; j < 4; ++j) { acc[2 * j] += __uint_as_float(w[j] << 16); acc[2 * j + 1] += __uint_as_float(w[j] & 0xffff0000u); }
        }
    }
}
// fold the pixel lanes through shared memory (csum: 128 x 8 floats) and add the CTA's sums to db; t = thread 0..127
__device__ __forceinline__ void colsum_finish(float (*csum)[8], const float* acc, int t, int q, int lane, int cg, int lanes,
                                              float* db, int c_base, int C) {
#pragma unroll
    for (int j = 0; j < 8; ++j) csum[t][j] = acc[j];
    named_bar_sync(2, 128);
    if (lane == 0) {
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            float v = 0.f;
            for (int l = 0; l < lanes; ++l) v += csum[l * cg + q][j];
            const int c = c_base + q * 8 + j;
            if (c < C) atomicAdd(db + c, v);
        }
    }
}

// Stage one accumulator row for a TMA tensor store/reduce: `row_bytes` (128 or 64) of fp32 per row, rows packed, the
// tensor map's SWIZZLE_128B / SWIZZLE_64B pattern applied (16-byte chunk index ^= row bits; `box` is 1024-byte aligned).
template <int NV4>
__device__ __forceinline__ void stage_row_swizzled(uint32_t box, int r, uint32_t row_bytes, const uint32_t* v) {
    const uint32_t mask = row_bytes == 128u ? 7u : 3u;
#pragma unroll
    for (int j = 0; j < NV4; ++j) {
        uint32_t off = (uint32_t)r * row_bytes + 16u * j;
        off ^= ((off >> 7) & mask) << 4;
        st_shared_v4(box + off, v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
    }
}

__device__ __forceinline__ void prefetch_tmap(const CUtensorMap* map) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(map) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_commit(uint32_t bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void tc_mma_bf16(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t"
        "}" ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
        : "memory");
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&r)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
          "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
          "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
          "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&r)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
          "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// Shared-memory matrix descriptors (tcgen05 "SmemDescriptor"): start address bits [0,14) (>>4), leading byte offset
// bits [16,30) (>>4), stride byte offset bits [32,46) (>>4), version = 1 at bit 46, layout type bits [61,64):
// 2 = SWIZZLE_128B, 4 = SWIZZLE_64B, 6 = SWIZZLE_32B.
//
// K-major operand: rows of cw*2 bytes (cw = 64/32/16 bf16 -> 128/64/32-byte swizzle), 8-row groups `sbo` bytes apart.
__device__ __forceinline__ uint64_t make_kmajor_desc(uint32_t saddr, uint32_t sbo, uint32_t ltype) {
    uint64_t d = 0;
    d |= (uint64_t)((saddr & 0x3FFFF) >> 4);
    d |= (uint64_t)1 << 16;                          // LBO unused for swizzled K-major layouts
    d |= (uint64_t)((sbo >> 4) & 0x3FFF) << 32;
    d |= (uint64_t)1 << 46;
    d |= (uint64_t)ltype << 61;
    return d;
}
// MN-major operand: the MN dimension is contiguous inside a row (cw elements), K runs across rows; 8-row (K) groups
// are `sbo` bytes apart and consecutive cw-element MN spans `lbo` bytes apart.
__device__ __forceinline__ uint64_t make_mn_desc(uint32_t saddr, uint32_t lbo, uint32_t sbo, uint32_t ltype) {
    uint64_t d = 0;
    d |= (uint64_t)((saddr & 0x3FFFF) >> 4);
    d |= (uint64_t)((lbo >> 4) & 0x3FFF) << 16;
    d |= (uint64_t)((sbo >> 4) & 0x3FFF) << 32;
    d |= (uint64_t)1 << 46;
    d |= (uint64_t)ltype << 61;
    return d;
}

// Split-word descriptor helpers for the MMA issue loops.  MEASURED on B200 (tools/mma_rate.cu): one thread can issue a
// tcgen05.mma every ~58 cycles at best, independent of N and of accumulator dependencies, so a 128x64x16 MMA (32 cycles of
// tensor work) is ISSUE-bound; every extra ALU instruction in the issue loop costs throughput.  The loops therefore keep the
// descriptor's high word constant and bump only the low word (start address >> 4) with 32-bit adds.
__device__ __forceinline__ uint32_t desc_lo(uint32_t saddr, uint32_t lbo) { return ((saddr & 0x3FFFF) >> 4) | (((lbo >> 4) & 0x3FFF) << 16); }
__device__ __forceinline__ uint32_t desc_hi(uint32_t sbo, uint32_t ltype) { return ((sbo >> 4) & 0x3FFF) | (1u << 14) | (ltype << 29); }
__device__ __forceinline__ void tc_mma_lohi(uint32_t d_tmem, uint32_t a_lo, uint32_t a_hi, uint32_t b_lo, uint32_t b_hi,
                                            uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        ".reg .b64 da, db;\n\t"
        "setp.ne.b32 p, %6, 0;\n\t"
        "mov.b64 da, {%1, %2};\n\t"
        "mov.b64 db, {%3, %4};\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %5, p;\n\t"
        "}" ::"r"(d_tmem), "r"(a_lo), "r"(a_hi), "r"(b_lo), "r"(b_hi), "r"(idesc), "r"(accumulate)
        : "memory");
}

// ------------------------------------------------------------------------------------------ shared conv epilogue
// 8 epilogue warps: warp e = (lane quarter q = e % 4, column half = e / 4).  Each thread owns ONE accumulator row (pixel)
// and walks its half of the tile's 32-column chunks: tcgen05.ld -> (+bias) -> (activation) -> bf16 -> 16-byte stores.
// Specialised at compile time on (activation, bias) so the inner loop carries no per-element branches.
constexpr int TC_EPI_WARPS = 8;

// Optional extras of the shared epilogue (svrs_conv2d_fprop_ex):
//   o2   - this thread's pixel in a second, fp32 output kept in the reference's NCHW-flat order (channel c at o2[c * hw]);
//          the posterior / prior heads are written there straight from the fp32 accumulators (no bf16 rounding, no
//          separate layout kernel).
//   sbn  - CTA-shared float[2][EPI_BN_MAXC]: per-channel sum and sum of squares of the conv output (BatchNorm batch
//          statistics taken from the fp32 accumulators instead of a separate read of the stored tensor).
constexpr int EPI_BN_MAXC = 256;
struct EpiRow {
    float* o2;
    int hw;
    float* sbn;
};

// column sums over the 32 lanes of a warp (transpose-reduce butterfly, 31 shuffles): on return lane l holds
// sum over lanes of v[l]
__device__ __forceinline__ float warp_colsum32(float (&v)[32], int lane) {
#pragma unroll
    for (int s = 16; s >= 1; s >>= 1) {
        const bool up = (lane & s) != 0;
#pragma unroll
        for (int j = 0; j < s; ++j) {
            const float send = up ? v[j] : v[j + s];
            const float keep = up ? v[j + s] : v[j];
            v[j] = keep + __shfl_xor_sync(0xffffffffu, send, s);
        }
    }
    return v[0];
}

// EXTRA = false is the plain epilogue (bf16 NHWC stores only); the extras live in a separate instantiation so that the
// common path carries none of their code (measured: folding them into one body cost every launch 1.5-3 us).
template <int ACT, bool BIAS, bool EXTRA>
__device__ __forceinline__ void epi_chunk8(const uint32_t* v, __nv_bfloat16* dst, const float* bias, int c, int Nc, bool vec_ok,
                                           float* o2, int hw) {
    float f[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) {
        float x = __uint_as_float(v[e]);
        if (BIAS) x += (c + e < Nc) ? __ldg(bias + c + e) : 0.f;
        if (ACT == SVRS_ACT_SIGMOID) x = 1.0f / (1.0f + __expf(-x));
        else if (ACT == SVRS_ACT_HARDTANH7) x = fminf(fmaxf(x, -7.0f), 7.0f);
        f[e] = x;
    }
    if (EXTRA) {
        if (o2) {
#pragma unroll
            for (int e = 0; e < 8; ++e)
                if (c + e < Nc) o2[(long long)(c + e) * hw] = f[e];
        }
        if (dst == nullptr) return;
    }
    if (vec_ok) {
        __nv_bfloat162 h0 = __floats2bfloat162_rn(f[0], f[1]), h1 = __floats2bfloat162_rn(f[2], f[3]);
        __nv_bfloat162 h2 = __floats2bfloat162_rn(f[4], f[5]), h3 = __floats2bfloat162_rn(f[6], f[7]);
        uint4 o;
        o.x = *reinterpret_cast<uint32_t*>(&h0); o.y = *reinterpret_cast<uint32_t*>(&h1);
        o.z = *reinterpret_cast<uint32_t*>(&h2); o.w = *reinterpret_cast<uint32_t*>(&h3);
        *reinterpret_cast<uint4*>(dst) = o;
    } else {
#pragma unroll
        for (int e = 0; e < 8; ++e)
            if (c + e < Nc) dst[e] = __float2bfloat16_rn(f[e]);
    }
}

// taddr: TMEM address of (this warp's lane quarter, accumulator column 0); orow: output row pointer at channel c_base
// (nullptr, EXTRA only: no NHWC output); er: optional extras (second output / BatchNorm statistics), see EpiRow
template <int ACT, bool BIAS, bool EXTRA>
__device__ __forceinline__ void epi_rows(uint32_t taddr, int n_tile, int half, __nv_bfloat16* orow, const float* bias,
                                         int c_base, int Nc, bool row_ok, const EpiRow& er) {
    const bool vec_ok = (Nc % 8 == 0);
    const int chunks = (n_tile + 31) / 32;
    const int cbeg = half == 0 ? 0 : (chunks + 1) / 2, cend = half == 0 ? (chunks + 1) / 2 : chunks;
    for (int ch = cbeg; ch < cend; ++ch) {
        const int c0 = ch * 32;
        uint32_t v[32];
        const int cols = (n_tile - c0 >= 32) ? 32 : 16;
        if (cols == 32) tmem_ld32(taddr + c0, v); else tmem_ld16(taddr + c0, v);
        tmem_ld_wait();
        if (row_ok) {
#pragma unroll
            for (int j = 0; j < 32; j += 8) {
                const int c = c_base + c0 + j;
                if (j < cols && c < Nc) {
                    if (EXTRA) epi_chunk8<ACT, BIAS, true>(v + j, orow ? orow + c0 + j : nullptr, bias, c, Nc, vec_ok, er.o2, er.hw);
                    else epi_chunk8<ACT, BIAS, false>(v + j, orow + c0 + j, bias, c, Nc, vec_ok, nullptr, 0);
                }
            }
        }
        if (EXTRA && er.sbn) {          // warp-uniform
            const int lane = threadIdx.x & 31;
            float a[32];
            // two passes over the chunk (sum, then sum of squares) so only v[] and one work array are live at a time
#pragma unroll
            for (int j = 0; j < 32; ++j) {
                const int c = c_base + c0 + j;
                float x = 0.f;
                if (row_ok && j < cols && c < Nc) {
                    x = __uint_as_float(v[j]);
                    if (BIAS) x += __ldg(bias + c);
                }
                a[j] = x;
            }
            const float s1 = warp_colsum32(a, lane);
#pragma unroll
            for (int j = 0; j < 32; ++j) {
                const int c = c_base + c0 + j;
                float x = 0.f;
                if (row_ok && j < cols && c < Nc) {
                    x = __uint_as_float(v[j]);
                    if (BIAS) x += __ldg(bias + c);
                }
                a[j] = x * x;
            }
            const float s2 = warp_colsum32(a, lane);
            const int c = c_base + c0 + lane;
            if (lane < cols && c < Nc) {
                atomicAdd(er.sbn + c, s1);
                atomicAdd(er.sbn + EPI_BN_MAXC + c, s2);
            }
        }
    }
}

// EXTRA kernels (heads with an fp32 NCHW-flat second output, BatchNorm producers) are separate instantiations of the conv
// kernels; the plain kernels carry none of that code, shared memory or register pressure.
template <bool EXTRA>
__device__ __forceinline__ void epi_dispatch(int act, uint32_t taddr, int n_tile, int half, __nv_bfloat16* orow, const float* bias,
                                             int c_base, int Nc, bool row_ok, const EpiRow& er) {
    if (EXTRA) {        // heads (o2: no activation or bias + Hardtanh) and BatchNorm producers (no activation)
        if (act == SVRS_ACT_HARDTANH7) epi_rows<SVRS_ACT_HARDTANH7, true, true>(taddr, n_tile, half, orow, bias, c_base, Nc, row_ok, er);
        else if (bias) epi_rows<SVRS_ACT_NONE, true, true>(taddr, n_tile, half, orow, bias, c_base, Nc, row_ok, er);
        else epi_rows<SVRS_ACT_NONE, false, true>(taddr, n_tile, half, orow, bias, c_base, Nc, row_ok, er);
        return;
    }
    if (bias) {
        if (act == SVRS_ACT_SIGMOID) epi_rows<SVRS_ACT_SIGMOID, true, false>(taddr, n_tile, half, orow, bias, c_base, Nc, row_ok, er);
        else if (act == SVRS_ACT_HARDTANH7) epi_rows<SVRS_ACT_HARDTANH7, true, false>(taddr, n_tile, half, orow, bias, c_base, Nc, row_ok, er);
        else epi_rows<SVRS_ACT_NONE, true, false>(taddr, n_tile, half, orow, bias, c_base, Nc, row_ok, er);
    } else {
        epi_rows<SVRS_ACT_NONE, false, false>(taddr, n_tile, half, orow, bias, c_base, Nc, row_ok, er);
    }
}

// BatchNorm statistics: zero the CTA's shared partial sums (all threads, before the first __syncthreads of the kernel) and
// flush them (epilogue threads, after their tile loop) to one of the SVRS_BN_REPLICAS copies of the double[2C] scratch.
__device__ __forceinline__ void epi_bn_zero(float* sbn) {
    for (int i = threadIdx.x; i < 2 * EPI_BN_MAXC; i += blockDim.x) sbn[i] = 0.f;
}
__device__ __forceinline__ void epi_bn_flush(const float* sbn, double* sums, int C, int epi_tid, int epi_threads) {
    named_bar_sync(3, epi_threads);
    double* dst = sums + (size_t)(blockIdx.x % SVRS_BN_REPLICAS) * 2 * C;
    for (int c = epi_tid; c < C; c += epi_threads) {
        const float s1 = sbn[c], s2 = sbn[EPI_BN_MAXC + c];
        if (s1 != 0.f || s2 != 0.f) { atomicAdd(dst + c, (double)s1); atomicAdd(dst + C + c, (double)s2); }
    }
}

// extras of svrs_conv2d_fprop_ex / svrs_convT2d_fprop_ex (host side)
struct ConvExtra {
    float* out2 = nullptr;        // fp32 NCHW-flat second output
    long long out2_ld = 0;
    double* bn_sums = nullptr;    // BatchNorm statistics scratch
};

// host helpers (conv_tc.cu)
int make_act_map(CUtensorMap* m, const void* base, int C, int W, int H, int N, long long sx, long long sy, long long sn,
                 int BW, int BH, int BNI, int cw);
bool pick_box(int OW, int OH, int& BW, int& BH, int& BNI);
// fp32 matrix [rows][inner] (inner contiguous), box (box_inner = 32 or 16 columns, box_rows), swizzle matching the box width
int make_f32_2d_map(CUtensorMap* m, const void* base, long long inner, long long rows, int box_inner, int box_rows);
// fp32 [d2][d1][d0] (d0 contiguous), box (box0 = 32 or 16 columns, box1 rows, 1), OOB parts of a box are clipped
int make_f32_3d_map(CUtensorMap* m, const void* base, long long d0, long long d1, long long d2, int box0, int box1);
int chunk_width(int C);   // 64 / 32 / 16 (last chunk ragged when C % 16 != 0) / 0 (C % 8 != 0 or C == 8: unsupported)

}  // namespace svrs
