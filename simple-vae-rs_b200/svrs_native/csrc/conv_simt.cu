// conv_simt.cu - CUDA-core (fp32 FMA) multi-tap GEMM convolution: fprop/dgrad for every conv form,
// and the matching wgrad.  This is the exact-fp32 path (parity mode, 1e-5) and the path for layers
// whose channel counts are too small / odd for the tcgen05 kernel (Cin or Cout in {4, 16}, cr != 2).
// Accumulation is always fp32; T is the storage type of activations and packed weights.
#include "common.cuh"
#include <stdlib.h>
#include "taps.cuh"
#include "tc_ptx.cuh"

namespace svrs {

struct ConvArgs {
    const void* in;
    void* out;
    const void* w;      // KN pack [tap][K][Nc]
    const float* bias;  // [Nc] or null
    int act;
    double* bn_sums;    // optional: SVRS_BN_REPLICAS x double[2*Nc] BatchNorm statistics of the output (conv_pixel only)
    TapGeom g;
};

constexpr int BK = 16;

}  // namespace svrs
#include "conv_narrow.cuh"   // bf16 narrow layers on mma.sync (needs ConvArgs)
namespace svrs {
extern int g_tc_enabled_narrow;   // follows svrs_set_tc_enabled: 0 keeps the narrow layers on the CUDA-core kernel (A/B tests)

template <typename T, int BM, int BN>
__global__ void __launch_bounds__(256) conv_taps_kernel(const __grid_constant__ ConvArgs a) {
    pdl_entry();
    constexpr int TM = 4, TN = 4;
    constexpr int TX = BN / TN;            // threads along channels
    static_assert((BM / TM) * TX == 256, "256 threads");
    constexpr int A_VECS = BM * BK / 4 / 256;  // float4 loads of A per thread
    constexpr int B_VECS_TOTAL = BK * BN / 4;
    constexpr int PADM = 4;

    __shared__ float As[BK][BM + PADM];
    __shared__ float Bs[BK][BN];

    const TapGeom& g = a.g;
    const Prob& pb = g.prob[blockIdx.z];
    const T* __restrict__ in = reinterpret_cast<const T*>(a.in);
    const T* __restrict__ w = reinterpret_cast<const T*>(a.w);
    T* __restrict__ out = reinterpret_cast<T*>(a.out) + pb.out_off;

    const int tid = threadIdx.x;
    const int tx = tid % TX, ty = tid / TX;
    const long long M = (long long)g.N * g.OH * g.OW;
    const long long m0 = (long long)blockIdx.x * BM;
    const int n0 = blockIdx.y * BN;
    const int K = g.K, Nc = g.Nc;
    const bool vecA = (K % 4 == 0);
    const bool vecB = (Nc % 4 == 0);

    // per-thread A-load coordinates
    int a_pix[A_VECS], a_kq[A_VECS], a_oy[A_VECS], a_ox[A_VECS];
    long long a_nbase[A_VECS];
    bool a_ok[A_VECS];
#pragma unroll
    for (int i = 0; i < A_VECS; ++i) {
        int v = tid + i * 256;
        a_pix[i] = v / (BK / 4);
        a_kq[i] = v % (BK / 4);
        long long m = m0 + a_pix[i];
        a_ok[i] = m < M;
        long long mm = a_ok[i] ? m : 0;
        int n = (int)(mm / ((long long)g.OH * g.OW));
        int r = (int)(mm % ((long long)g.OH * g.OW));
        a_oy[i] = r / g.OW;
        a_ox[i] = r % g.OW;
        a_nbase[i] = (long long)n * g.i_sn;
    }

    float acc[TM][TN];
#pragma unroll
    for (int i = 0; i < TM; ++i)
#pragma unroll
        for (int j = 0; j < TN; ++j) acc[i][j] = 0.f;

    const int kchunks = (K + BK - 1) / BK;
    for (int t = 0; t < pb.ntaps; ++t) {
        const Tap tp = pb.taps[t];
        const T* __restrict__ wt = w + tp.w_off;
        for (int kc = 0; kc < kchunks; ++kc) {
            const int k0 = kc * BK;
            // ---- A tile: [BM pixels][BK channels], shifted by the tap, zero outside the view
#pragma unroll
            for (int i = 0; i < A_VECS; ++i) {
                float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
                int iy = a_oy[i] + tp.dy, ix = a_ox[i] + tp.dx;
                int kk = k0 + a_kq[i] * 4;
                if (a_ok[i] && iy >= 0 && iy < g.IH && ix >= 0 && ix < g.IW && kk < K) {
                    const T* p = in + tp.in_off + a_nbase[i] + (long long)iy * g.i_sy + (long long)ix * g.i_sx + kk;
                    if (vecA) {
                        v = ld4(p);
                    } else {
                        v.x = Cvt<T>::to_f(p[0]);
                        if (kk + 1 < K) v.y = Cvt<T>::to_f(p[1]);
                        if (kk + 2 < K) v.z = Cvt<T>::to_f(p[2]);
                        if (kk + 3 < K) v.w = Cvt<T>::to_f(p[3]);
                    }
                }
                int kb = a_kq[i] * 4;
                As[kb + 0][a_pix[i]] = v.x;
                As[kb + 1][a_pix[i]] = v.y;
                As[kb + 2][a_pix[i]] = v.z;
                As[kb + 3][a_pix[i]] = v.w;
            }
            // ---- B tile: [BK][BN] of W_t (row k, contiguous along output channels)
            for (int v = tid; v < B_VECS_TOTAL; v += 256) {
                int kr = v / (BN / 4), nq = v % (BN / 4);
                int kk = k0 + kr, nn = n0 + nq * 4;
                float4 b = make_float4(0.f, 0.f, 0.f, 0.f);
                if (kk < K && nn < Nc) {
                    const T* p = wt + (long long)kk * Nc + nn;
                    if (vecB) {
                        b = ld4(p);
                    } else {
                        b.x = Cvt<T>::to_f(p[0]);
                        if (nn + 1 < Nc) b.y = Cvt<T>::to_f(p[1]);
                        if (nn + 2 < Nc) b.z = Cvt<T>::to_f(p[2]);
                        if (nn + 3 < Nc) b.w = Cvt<T>::to_f(p[3]);
                    }
                }
                *reinterpret_cast<float4*>(&Bs[kr][nq * 4]) = b;
            }
            __syncthreads();
#pragma unroll
            for (int k = 0; k < BK; ++k) {
                float4 av = *reinterpret_cast<const float4*>(&As[k][ty * TM]);
                float4 bv = *reinterpret_cast<const float4*>(&Bs[k][tx * TN]);
                float ar[4] = {av.x, av.y, av.z, av.w};
                float br[4] = {bv.x, bv.y, bv.z, bv.w};
#pragma unroll
                for (int i = 0; i < TM; ++i)
#pragma unroll
                    for (int j = 0; j < TN; ++j) acc[i][j] = fmaf(ar[i], br[j], acc[i][j]);
            }
            __syncthreads();
        }
    }

    // ---- epilogue: bias, activation, store (4 consecutive channels per row)
    const int nn = n0 + tx * TN;
    if (nn >= Nc) return;
    float bz[4] = {0.f, 0.f, 0.f, 0.f};
    if (a.bias) {
#pragma unroll
        for (int j = 0; j < 4; ++j)
            if (nn + j < Nc) bz[j] = a.bias[nn + j];
    }
#pragma unroll
    for (int i = 0; i < TM; ++i) {
        long long m = m0 + ty * TM + i;
        if (m >= M) continue;
        int n = (int)(m / ((long long)g.OH * g.OW));
        int r = (int)(m % ((long long)g.OH * g.OW));
        int oy = r / g.OW, ox = r % g.OW;
        T* p = out + (long long)n * g.o_sn + (long long)oy * g.o_sy + (long long)ox * g.o_sx + nn;
        float4 v;
        v.x = apply_act(acc[i][0] + bz[0], a.act);
        v.y = apply_act(acc[i][1] + bz[1], a.act);
        v.z = apply_act(acc[i][2] + bz[2], a.act);
        v.w = apply_act(acc[i][3] + bz[3], a.act);
        if (vecB) {
            st4(p, v);
        } else {
            p[0] = Cvt<T>::from_f(v.x);
            if (nn + 1 < Nc) p[1] = Cvt<T>::from_f(v.y);
            if (nn + 2 < Nc) p[2] = Cvt<T>::from_f(v.z);
            if (nn + 3 < Nc) p[3] = Cvt<T>::from_f(v.w);
        }
    }
}

// ------------------------------------------------------------------------------------------------
// Narrow layers (reduction and output channels both in {4, 16}: the first and last convs of every sub-network at full
// resolution).  They are HBM-bound streaming ops (a few hundred FLOP per pixel), so the GEMM tiling above only adds
// barriers: here one thread owns one output pixel, the per-tap weights sit in shared memory (broadcast float4 reads) and
// the taps are a register loop.  No barriers after the weight stage-in.
// ------------------------------------------------------------------------------------------------
// TO = storage type of the OUTPUT (fp32 output from bf16 operands: the sigmoid tail that feeds the NLL, so x_hat is
// never rounded to bf16).  a.bn_sums != NULL: per-channel sum / sum of squares of the fp32 results (BatchNorm batch
// statistics fused into the producer; warp shuffle -> shared -> one double atomic per channel and block).
template <typename T, int CR, int CW, typename TO>
__global__ void __launch_bounds__(256) conv_pixel_kernel(const __grid_constant__ ConvArgs a) {
    pdl_entry();
    __shared__ __align__(16) float ws[16 * CR * CW];
    __shared__ float s_bn[2 * CW];
    const TapGeom& g = a.g;
    const Prob& pb = g.prob[blockIdx.z];
    const T* __restrict__ in = reinterpret_cast<const T*>(a.in);
    const T* __restrict__ w = reinterpret_cast<const T*>(a.w);
    TO* __restrict__ out = reinterpret_cast<TO*>(a.out) + pb.out_off;
    for (int i = threadIdx.x; i < pb.ntaps * CR * CW; i += 256)
        ws[i] = Cvt<T>::to_f(w[pb.taps[i / (CR * CW)].w_off + i % (CR * CW)]);
    if (threadIdx.x < 2 * CW) s_bn[threadIdx.x] = 0.f;
    __syncthreads();
    const long long M = (long long)g.N * g.OH * g.OW;
    const long long m = (long long)blockIdx.x * 256 + threadIdx.x;
    const bool live = m < M;
    if (!live && !a.bn_sums) return;
    float acc[CW];
#pragma unroll
    for (int c = 0; c < CW; ++c) acc[c] = 0.f;
    if (live) {
        const int n = (int)(m / ((long long)g.OH * g.OW));
        const int r = (int)(m % ((long long)g.OH * g.OW));
        const int oy = r / g.OW, ox = r % g.OW;
#pragma unroll
        for (int c = 0; c < CW; ++c) acc[c] = a.bias ? a.bias[c] : 0.f;
        const T* base = in + (long long)n * g.i_sn;
        for (int t = 0; t < pb.ntaps; ++t) {
            const Tap tp = pb.taps[t];
            const int iy = oy + tp.dy, ix = ox + tp.dx;
            if (iy < 0 || iy >= g.IH || ix < 0 || ix >= g.IW) continue;
            const T* px = base + tp.in_off + (long long)iy * g.i_sy + (long long)ix * g.i_sx;
            float xv[CR];
#pragma unroll
            for (int k = 0; k < CR; k += 4) {
                float4 v = ld4(px + k);
                xv[k] = v.x; xv[k + 1] = v.y; xv[k + 2] = v.z; xv[k + 3] = v.w;
            }
            const float* wt = ws + t * CR * CW;
#pragma unroll
            for (int k = 0; k < CR; ++k)
#pragma unroll
                for (int c = 0; c < CW; c += 4) {
                    float4 wv = *reinterpret_cast<const float4*>(wt + k * CW + c);
                    acc[c] = fmaf(xv[k], wv.x, acc[c]); acc[c + 1] = fmaf(xv[k], wv.y, acc[c + 1]);
                    acc[c + 2] = fmaf(xv[k], wv.z, acc[c + 2]); acc[c + 3] = fmaf(xv[k], wv.w, acc[c + 3]);
                }
        }
        TO* po = out + (long long)n * g.o_sn + (long long)oy * g.o_sy + (long long)ox * g.o_sx;
#pragma unroll
        for (int c = 0; c < CW; c += 4)
            st4(po + c, make_float4(apply_act(acc[c], a.act), apply_act(acc[c + 1], a.act), apply_act(acc[c + 2], a.act),
                                    apply_act(acc[c + 3], a.act)));
    }
    if (a.bn_sums) {                     // block-uniform; dead threads of the last block contribute zeros
#pragma unroll
        for (int c = 0; c < CW; ++c) {
            const float s1 = warp_sum(acc[c]), s2 = warp_sum(acc[c] * acc[c]);
            if (threadIdx.x % 32 == 0) { atomicAdd(&s_bn[c], s1); atomicAdd(&s_bn[CW + c], s2); }
        }
        __syncthreads();
        if (threadIdx.x < 2 * CW && s_bn[threadIdx.x] != 0.f)
            atomicAdd(a.bn_sums + (size_t)((blockIdx.x + blockIdx.z) % SVRS_BN_REPLICAS) * 2 * CW + threadIdx.x, (double)s_bn[threadIdx.x]);
    }
}

template <typename T, typename TO>
static void launch_pixel(const ConvArgs& a, dim3 grid, cudaStream_t st) {
    const int K = a.g.K, Nc = a.g.Nc;
    if (K == 4 && Nc == 4) SVRS_LAUNCH((conv_pixel_kernel<T, 4, 4, TO>), grid, 256, 0, st, a);
    else if (K == 4 && Nc == 16) SVRS_LAUNCH((conv_pixel_kernel<T, 4, 16, TO>), grid, 256, 0, st, a);
    else if (K == 16 && Nc == 4) SVRS_LAUNCH((conv_pixel_kernel<T, 16, 4, TO>), grid, 256, 0, st, a);
    else SVRS_LAUNCH((conv_pixel_kernel<T, 16, 16, TO>), grid, 256, 0, st, a);
}

static bool pixel_kernel_takes(const TapGeom& g, int dtype) {
    return (g.K == 4 || g.K == 16) && (g.Nc == 4 || g.Nc == 16) && (g.K == 4 || g.Nc == 4 || dtype == SVRS_F32);
}

// out_dtype: storage type of the output (== dtype except for the bf16 -> fp32 tail, conv_pixel only)
static int launch_conv(const ConvArgs& a, int dtype, cudaStream_t st, int out_dtype = -1) {
    const TapGeom& g = a.g;
    long long M = (long long)g.N * g.OH * g.OW;
    if (M == 0) return 0;
    if (out_dtype < 0) out_dtype = dtype;
    if (g_tc_enabled_narrow && narrow_mma_takes(g, dtype) && (out_dtype == SVRS_BF16 || out_dtype == SVRS_F32)) {
        launch_narrow(a, out_dtype, st);
        return check_launch("conv_narrow_mma_kernel");
    }
    if (pixel_kernel_takes(g, dtype)) {
        dim3 grid((unsigned)((M + 255) / 256), 1, g.nprob);
        if (dtype == SVRS_F32 && out_dtype == SVRS_F32) launch_pixel<float, float>(a, grid, st);
        else if (dtype == SVRS_BF16 && out_dtype == SVRS_BF16) launch_pixel<__nv_bfloat16, __nv_bfloat16>(a, grid, st);
        else if (dtype == SVRS_BF16 && out_dtype == SVRS_F32) launch_pixel<__nv_bfloat16, float>(a, grid, st);
        else { set_error("conv: unsupported (dtype, out_dtype) = (%d, %d)", dtype, out_dtype); return SVRS_E_UNSUPPORTED; }
        return check_launch("conv_pixel_kernel");
    }
    if (out_dtype != dtype || a.bn_sums) {
        set_error("conv: fp32 output / fused BatchNorm statistics are not available on the generic SIMT kernel (K=%d Nc=%d)", g.K, g.Nc);
        return SVRS_E_UNSUPPORTED;
    }
    if (g.Nc <= 16) {
        dim3 grid((unsigned)((M + 255) / 256), (g.Nc + 15) / 16, g.nprob);
        if (dtype == SVRS_F32) SVRS_LAUNCH((conv_taps_kernel<float, 256, 16>), grid, 256, 0, st, a);
        else SVRS_LAUNCH((conv_taps_kernel<__nv_bfloat16, 256, 16>), grid, 256, 0, st, a);
    } else {
        dim3 grid((unsigned)((M + 63) / 64), (g.Nc + 63) / 64, g.nprob);
        if (dtype == SVRS_F32) SVRS_LAUNCH((conv_taps_kernel<float, 64, 64>), grid, 256, 0, st, a);
        else SVRS_LAUNCH((conv_taps_kernel<__nv_bfloat16, 64, 64>), grid, 256, 0, st, a);
    }
    return check_launch("conv_taps_kernel");
}

// ------------------------------------------------------------------------------------------------
// wgrad:  dW_t[a][b] += sum_m G[m][a] * X_t[m (+shift)][b]      (m over the output grid of `g`)
// G lives on the output grid (channels Ca = g.Nc), X on the input view (channels Cb = g.K).
// Destination is the torch layout dw[(a*Cb + b)*KK + tap], fp32 atomics; K (pixels) is split over grid.z.
// ------------------------------------------------------------------------------------------------
struct WgradArgs {
    const void* gmat;  // operand on the output grid
    const void* x;     // operand on the input view
    float* dw;
    int KK;
    int ksplit;
    TapGeom g;         // prob[0].taps[t].w_off unused; tap id = t
};

}  // namespace svrs
#include "wgrad_narrow.cuh"   // bf16 narrow weight gradients on mma.sync + movmatrix (needs WgradArgs)
namespace svrs {

template <typename T>
__global__ void __launch_bounds__(256) wgrad_taps_kernel(const __grid_constant__ WgradArgs a) {
    pdl_entry();
    constexpr int BA = 64, BB = 64, BP = 16;
    __shared__ float Gs[BP][BA];
    __shared__ float Xs[BP][BB];
    const TapGeom& g = a.g;
    const Prob& pb = g.prob[0];
    const T* __restrict__ G = reinterpret_cast<const T*>(a.gmat) + pb.out_off;
    const T* __restrict__ X = reinterpret_cast<const T*>(a.x);
    const int Ca = g.Nc, Cb = g.K;
    const int b_tiles = (Cb + BB - 1) / BB;
    const int a0 = (blockIdx.x / b_tiles) * BA;
    const int b0 = (blockIdx.x % b_tiles) * BB;
    const int t = blockIdx.y;
    const Tap tp = pb.taps[t];
    const long long M = (long long)g.N * g.OH * g.OW;
    long long chunk = (M + a.ksplit - 1) / a.ksplit;
    chunk = (chunk + BP - 1) / BP * BP;
    const long long mbeg = (long long)blockIdx.z * chunk;
    const long long mend = mbeg + chunk < M ? mbeg + chunk : M;
    const int tid = threadIdx.x;
    const int tx = tid % 16, ty = tid / 16;
    const bool vecG = (Ca % 4 == 0), vecX = (Cb % 4 == 0);
    const int lp = tid / 16;       // pixel within the BP chunk
    const int lq = (tid % 16) * 4; // channel quad

    float acc[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;

    for (long long mb = mbeg; mb < mend; mb += BP) {
        long long m = mb + lp;
        float4 gv = make_float4(0.f, 0.f, 0.f, 0.f), xv = gv;
        if (m < mend) {
            int n = (int)(m / ((long long)g.OH * g.OW));
            int r = (int)(m % ((long long)g.OH * g.OW));
            int oy = r / g.OW, ox = r % g.OW;
            int ca = a0 + lq;
            if (ca < Ca) {
                const T* p = G + (long long)n * g.o_sn + (long long)oy * g.o_sy + (long long)ox * g.o_sx + ca;
                if (vecG) gv = ld4(p);
                else {
                    gv.x = Cvt<T>::to_f(p[0]);
                    if (ca + 1 < Ca) gv.y = Cvt<T>::to_f(p[1]);
                    if (ca + 2 < Ca) gv.z = Cvt<T>::to_f(p[2]);
                    if (ca + 3 < Ca) gv.w = Cvt<T>::to_f(p[3]);
                }
            }
            int iy = oy + tp.dy, ix = ox + tp.dx;
            int cb = b0 + lq;
            if (iy >= 0 && iy < g.IH && ix >= 0 && ix < g.IW && cb < Cb) {
                const T* p = X + tp.in_off + (long long)n * g.i_sn + (long long)iy * g.i_sy + (long long)ix * g.i_sx + cb;
                if (vecX) xv = ld4(p);
                else {
                    xv.x = Cvt<T>::to_f(p[0]);
                    if (cb + 1 < Cb) xv.y = Cvt<T>::to_f(p[1]);
                    if (cb + 2 < Cb) xv.z = Cvt<T>::to_f(p[2]);
                    if (cb + 3 < Cb) xv.w = Cvt<T>::to_f(p[3]);
                }
            }
        }
        *reinterpret_cast<float4*>(&Gs[lp][lq]) = gv;
        *reinterpret_cast<float4*>(&Xs[lp][lq]) = xv;
        __syncthreads();
#pragma unroll
        for (int k = 0; k < BP; ++k) {
            float4 av = *reinterpret_cast<const float4*>(&Gs[k][ty * 4]);
            float4 bv = *reinterpret_cast<const float4*>(&Xs[k][tx * 4]);
            float ar[4] = {av.x, av.y, av.z, av.w};
            float br[4] = {bv.x, bv.y, bv.z, bv.w};
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(ar[i], br[j], acc[i][j]);
        }
        __syncthreads();
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        int ca = a0 + ty * 4 + i;
        if (ca >= Ca) continue;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            int cb = b0 + tx * 4 + j;
            if (cb >= Cb) continue;
            atomicAdd(&a.dw[((long long)ca * Cb + cb) * a.KK + t], acc[i][j]);
        }
    }
}

// column sums of a contiguous [M][C] matrix, atomically added to out[C] (bias gradients)
template <typename T>
__global__ void __launch_bounds__(256) colsum_kernel(const T* __restrict__ x, long long M, int C,
                                                      float* __restrict__ out, long long rows_per_block) {
    pdl_entry();
    __shared__ float red[8][33];
    const int lx = threadIdx.x % 32, ly = threadIdx.x / 32;
    const long long r0 = (long long)blockIdx.x * rows_per_block;
    long long r1 = r0 + rows_per_block;
    if (r1 > M) r1 = M;
    for (int c0 = 0; c0 < C; c0 += 32) {
        int c = c0 + lx;
        float s = 0.f;
        if (c < C)
            for (long long r = r0 + ly; r < r1; r += 8) s += Cvt<T>::to_f(x[r * C + c]);
        red[ly][lx] = s;
        __syncthreads();
        if (ly == 0 && c < C) {
            float tot = 0.f;
#pragma unroll
            for (int k = 0; k < 8; ++k) tot += red[k][lx];
            atomicAdd(&out[c], tot);
        }
        __syncthreads();
    }
}

// ------------------------------------------------------------------------------------------------
// wgrad for narrow layers (min(Ca, Cb) <= 16: the 4- and 16-channel layers at full resolution).  These are
// pure streaming reductions (a few hundred outputs, half a million pixels): every thread owns one 4x4 (a, b)
// register tile of one tap and walks its own strided pixel subset straight from global memory (the 4-channel
// vectors of neighbouring taps hit L1), so the loop has no shared memory and no barriers; the per-thread tiles
// are combined by warp shuffles + one shared-memory pass and a single atomic per output per CTA.
// grid = (taps, pixel splits, sub-tile groups); block = SUB sub-tiles x (256 / SUB) pixel lanes.
// ------------------------------------------------------------------------------------------------
template <typename T, int SUB>
__global__ void __launch_bounds__(256) wgrad_direct_kernel(const __grid_constant__ WgradArgs a) {
    pdl_entry();
    constexpr int L = 256 / SUB;   // pixel lanes per sub-tile
    __shared__ float red[(L > 32 ? L / 32 : 1)][SUB][16];
    const TapGeom& g = a.g;
    const Prob& pb = g.prob[0];
    const T* __restrict__ G = reinterpret_cast<const T*>(a.gmat) + pb.out_off;
    const T* __restrict__ X = reinterpret_cast<const T*>(a.x);
    const int Ca = g.Nc, Cb = g.K;
    const int qa = (Ca + 3) / 4, qb = (Cb + 3) / 4;
    const int t = blockIdx.x;
    const Tap tp = pb.taps[t];
    const int lane = threadIdx.x % L;
    const int sub = threadIdx.x / L + blockIdx.z * SUB;
    const bool sub_ok = sub < qa * qb;
    const int a0 = (sub_ok ? sub / qb : 0) * 4, b0 = (sub_ok ? sub % qb : 0) * 4;
    const long long M = (long long)g.N * g.OH * g.OW;
    long long chunk = (M + gridDim.y - 1) / gridDim.y;
    const long long mbeg = (long long)blockIdx.y * chunk;
    const long long mend = mbeg + chunk < M ? mbeg + chunk : M;
    const bool vecG = (Ca % 4 == 0), vecX = (Cb % 4 == 0);
    float acc[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
    if (sub_ok) {
        const int ohw = g.OH * g.OW;
        constexpr int U = 4;      // pixels in flight per thread: issue all loads of a group before the FMAs (ILP)
        for (long long m0 = mbeg + lane; m0 < mend; m0 += (long long)L * U) {
            float4 gv[U], xv[U];
#pragma unroll
            for (int u = 0; u < U; ++u) {
                gv[u] = make_float4(0.f, 0.f, 0.f, 0.f);
                xv[u] = gv[u];
                const long long m = m0 + (long long)u * L;
                if (m >= mend) continue;
                const int n = (int)(m / ohw);
                const int r = (int)(m - (long long)n * ohw);
                const int oy = r / g.OW, ox = r - oy * g.OW;
                const int iy = oy + tp.dy, ix = ox + tp.dx;
                if (iy < 0 || iy >= g.IH || ix < 0 || ix >= g.IW) continue;
                const T* pg = G + (long long)n * g.o_sn + (long long)oy * g.o_sy + (long long)ox * g.o_sx + a0;
                const T* px = X + tp.in_off + (long long)n * g.i_sn + (long long)iy * g.i_sy + (long long)ix * g.i_sx + b0;
                if (vecG) gv[u] = ld4(pg);
                else {
                    gv[u].x = Cvt<T>::to_f(pg[0]);
                    gv[u].y = a0 + 1 < Ca ? Cvt<T>::to_f(pg[1]) : 0.f;
                    gv[u].z = a0 + 2 < Ca ? Cvt<T>::to_f(pg[2]) : 0.f;
                    gv[u].w = a0 + 3 < Ca ? Cvt<T>::to_f(pg[3]) : 0.f;
                }
                if (vecX) xv[u] = ld4(px);
                else {
                    xv[u].x = Cvt<T>::to_f(px[0]);
                    xv[u].y = b0 + 1 < Cb ? Cvt<T>::to_f(px[1]) : 0.f;
                    xv[u].z = b0 + 2 < Cb ? Cvt<T>::to_f(px[2]) : 0.f;
                    xv[u].w = b0 + 3 < Cb ? Cvt<T>::to_f(px[3]) : 0.f;
                }
            }
#pragma unroll
            for (int u = 0; u < U; ++u) {
                const float ga[4] = {gv[u].x, gv[u].y, gv[u].z, gv[u].w}, xb[4] = {xv[u].x, xv[u].y, xv[u].z, xv[u].w};
#pragma unroll
                for (int i = 0; i < 4; ++i)
#pragma unroll
                    for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(ga[i], xb[j], acc[i][j]);
            }
        }
    }
    // reduce over the pixel lanes of each sub-tile
    constexpr int WL = L < 32 ? L : 32;
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            float v = acc[i][j];
#pragma unroll
            for (int o = WL / 2; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
            acc[i][j] = v;
        }
    if (L > 32) {
        const int wsub = lane / 32;   // warp index within the sub-tile
        if (lane % 32 == 0) {
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) red[wsub][threadIdx.x / L][i * 4 + j] = acc[i][j];
        }
        __syncthreads();
        if (lane == 0) {
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    float v = 0.f;
                    for (int w2 = 0; w2 < L / 32; ++w2) v += red[w2][threadIdx.x / L][i * 4 + j];
                    acc[i][j] = v;
                }
        }
    }
    if (lane == 0 && sub_ok) {
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            if (a0 + i >= Ca) continue;
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                if (b0 + j >= Cb) continue;
                atomicAdd(&a.dw[((long long)(a0 + i) * Cb + b0 + j) * a.KK + t], acc[i][j]);
            }
        }
    }
}

// ------------------------------------------------------------------------------------------------
// wgrad for the 4 <-> 16 and 4 <-> 4 channel layers (the image-side ends of every sub-network at full resolution).
// One WARP per tap (TPW taps per warp for the 4x4 case), lanes = 32 consecutive output pixels, so a warp reads its G and
// X vectors fully coalesced and a thread keeps the whole CA x CB outer-product tile of its tap(s) in registers: per
// pixel it issues 1-2 vector loads per operand and CA*CB FMAs - no shared memory, no per-pixel 64-bit index math (the
// image index is uniform per 32-pixel group).  The nine / sixteen warps of a CTA walk the same pixels, so all but the
// first tap's loads hit L1.  Lanes are folded with shuffles at the end; one atomic per output per CTA.
// ------------------------------------------------------------------------------------------------
// raw (unconverted) channel vectors: NW 32-bit words, loaded with the widest access that fits
template <int NW> __device__ __forceinline__ void load_raw(const void* p, uint32_t* w) {
    if (NW == 2) { uint2 r = __ldg(reinterpret_cast<const uint2*>(p)); w[0] = r.x; w[1] = r.y; }
    else {
#pragma unroll
        for (int i = 0; i < NW / 4; ++i) {
            uint4 r = __ldg(reinterpret_cast<const uint4*>(p) + i);
            w[4 * i] = r.x; w[4 * i + 1] = r.y; w[4 * i + 2] = r.z; w[4 * i + 3] = r.w;
        }
    }
}
template <typename T, int C> __device__ __forceinline__ void raw_to_float(const uint32_t* w, float* o);
template <int C> __device__ __forceinline__ void raw_to_float_f32(const uint32_t* w, float* o) {
#pragma unroll
    for (int i = 0; i < C; ++i) o[i] = __uint_as_float(w[i]);
}
template <> __device__ __forceinline__ void raw_to_float<float, 4>(const uint32_t* w, float* o) { raw_to_float_f32<4>(w, o); }
template <> __device__ __forceinline__ void raw_to_float<float, 16>(const uint32_t* w, float* o) { raw_to_float_f32<16>(w, o); }
template <int C> __device__ __forceinline__ void raw_to_float_bf16(const uint32_t* w, float* o) {
#pragma unroll
    for (int i = 0; i < C / 2; ++i) { o[2 * i] = __uint_as_float(w[i] << 16); o[2 * i + 1] = __uint_as_float(w[i] & 0xffff0000u); }
}
template <> __device__ __forceinline__ void raw_to_float<__nv_bfloat16, 4>(const uint32_t* w, float* o) { raw_to_float_bf16<4>(w, o); }
template <> __device__ __forceinline__ void raw_to_float<__nv_bfloat16, 16>(const uint32_t* w, float* o) { raw_to_float_bf16<16>(w, o); }

template <typename T, int CA, int CB, int TPW>
__global__ void __launch_bounds__(512, 1) wgrad_narrow_kernel(const __grid_constant__ WgradArgs a) {
    pdl_entry();
    __shared__ float red[16][TPW * CA * CB];
    const TapGeom& g = a.g;
    const Prob& pb = g.prob[0];
    const T* __restrict__ G = reinterpret_cast<const T*>(a.gmat) + pb.out_off;
    const T* __restrict__ X = reinterpret_cast<const T*>(a.x);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    // blockIdx.z selects a GROUP of taps: the taps of a layer are spread over several small CTAs (3-4 warps) instead of
    // one 9..16-warp CTA per SM, so that 4-5 CTAs with DIFFERENT pixel ranges are resident per SM - the kernel was bound by
    // the number of distinct loads in flight (one pixel stream per SM: 0.3 TB/s), not by FMA issue
    const int t0 = (blockIdx.z * (blockDim.x >> 5) + warp) * TPW;
    Tap tp[TPW];
    bool tap_ok[TPW];
#pragma unroll
    for (int j = 0; j < TPW; ++j) { tap_ok[j] = t0 + j < pb.ntaps; tp[j] = pb.taps[tap_ok[j] ? t0 + j : 0]; }
    float acc[TPW][CA][CB];
#pragma unroll
    for (int j = 0; j < TPW; ++j)
#pragma unroll
        for (int ia = 0; ia < CA; ++ia)
#pragma unroll
            for (int ib = 0; ib < CB; ++ib) acc[j][ia][ib] = 0.f;
    const int ohw = g.OH * g.OW;
    const int groups = g.N * (ohw / 32);          // 32-pixel groups; ohw % 32 == 0 (checked by the launcher)
    // Three pixel groups in flight per thread (raw, unconverted vectors: 10 registers per group for 4 x 16 bf16): with
    // one 9..16-warp CTA per SM the loop would otherwise be exposed to the full L2 latency once per group.
    constexpr int GW = CA * (int)sizeof(T) / 4, XW = CB * (int)sizeof(T) / 4;
    struct Slot { uint32_t g[GW]; uint32_t x[TPW][XW]; };
    auto issue = [&](int gi, Slot& sl) {
#pragma unroll
        for (int i = 0; i < GW; ++i) sl.g[i] = 0u;
#pragma unroll
        for (int j = 0; j < TPW; ++j)
#pragma unroll
            for (int i = 0; i < XW; ++i) sl.x[j][i] = 0u;
        if (gi >= groups) return;
        const int m0 = gi * 32;
        const int n = m0 / ohw;
        const int r = m0 - n * ohw + lane;
        const int oy = r / g.OW, ox = r - oy * g.OW;
        load_raw<GW>(G + (long long)n * g.o_sn + (long long)oy * g.o_sy + (long long)ox * g.o_sx, sl.g);
#pragma unroll
        for (int j = 0; j < TPW; ++j) {
            const int iy = oy + tp[j].dy, ix = ox + tp[j].dx;
            if (tap_ok[j] && iy >= 0 && iy < g.IH && ix >= 0 && ix < g.IW)
                load_raw<XW>(X + tp[j].in_off + (long long)n * g.i_sn + (long long)iy * g.i_sy + (long long)ix * g.i_sx, sl.x[j]);
        }
    };
    auto compute = [&](const Slot& sl) {
        float gv[CA];
        raw_to_float<T, CA>(sl.g, gv);
#pragma unroll
        for (int j = 0; j < TPW; ++j) {
            float xv[CB];
            raw_to_float<T, CB>(sl.x[j], xv);
#pragma unroll
            for (int ia = 0; ia < CA; ++ia)
#pragma unroll
                for (int ib = 0; ib < CB; ++ib) acc[j][ia][ib] = fmaf(gv[ia], xv[ib], acc[j][ia][ib]);
        }
    };
    const int st = gridDim.x;
    Slot s0, s1, s2;
    issue(blockIdx.x, s0);
    issue(blockIdx.x + st, s1);
    for (int gi = blockIdx.x; gi < groups; gi += 3 * st) {
        issue(gi + 2 * st, s2); compute(s0);
        issue(gi + 3 * st, s0); compute(s1);
        issue(gi + 4 * st, s1); compute(s2);
    }
    // fold the 32 lanes; lane 0 parks the warp's tile in shared memory, then the warp issues its atomics in parallel
#pragma unroll
    for (int j = 0; j < TPW; ++j)
#pragma unroll
        for (int ia = 0; ia < CA; ++ia)
#pragma unroll
            for (int ib = 0; ib < CB; ++ib) {
                float v = acc[j][ia][ib];
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
                if (lane == 0) red[warp][(j * CA + ia) * CB + ib] = v;
            }
    __syncwarp();
    for (int e = lane; e < TPW * CA * CB; e += 32) {
        const int ib = e % CB, ia = (e / CB) % CA, j = e / (CA * CB);
        if (t0 + j < pb.ntaps) atomicAdd(&a.dw[((long long)ia * CB + ib) * a.KK + t0 + j], red[warp][e]);
    }
}

// true (and launched) when the shape is one of the narrow forms
template <typename T>
static bool try_launch_wgrad_narrow(const WgradArgs& a, cudaStream_t st, int& rc) {
    const TapGeom& g = a.g;
    const int Ca = g.Nc, Cb = g.K, ntaps = g.prob[0].ntaps;
    const long long ohw = (long long)g.OH * g.OW;
    static const bool disabled = getenv("SVRS_NO_NARROW") != nullptr;
    if (disabled) return false;
    if (g.nprob != 1 || ohw % 32 != 0 || (long long)g.N * ohw >= (1ll << 31) || ntaps > 16) return false;
    const int groups = (int)((long long)g.N * ohw / 32);
    const int warps = (Ca == 4 && Cb == 4) ? (ntaps + 3) / 4 : ntaps;       // warps needed for all taps
    // warps per CTA: 3 (nine taps) or 4 (sixteen taps / the 4x4 form); tap groups in grid.z
    const int wpc = warps % 3 == 0 ? 3 : (warps >= 4 ? 4 : warps);
    const int zg = (warps + wpc - 1) / wpc;
    int per_sm = 65536 / (128 * 32 * wpc);                                  // CTAs per SM at 128 registers per thread
    if (per_sm > 5) per_sm = 5;
    int gx = (num_sms() * per_sm + zg - 1) / zg;
    if (gx > groups) gx = groups;
    dim3 grid(gx, 1, zg);
    if (Ca == 4 && Cb == 16) SVRS_LAUNCH((wgrad_narrow_kernel<T, 4, 16, 1>), grid, 32 * wpc, 0, st, a);
    else if (Ca == 16 && Cb == 4) SVRS_LAUNCH((wgrad_narrow_kernel<T, 16, 4, 1>), grid, 32 * wpc, 0, st, a);
    else if (Ca == 4 && Cb == 4) SVRS_LAUNCH((wgrad_narrow_kernel<T, 4, 4, 4>), grid, 32 * wpc, 0, st, a);
    else return false;
    rc = check_launch("wgrad_narrow_kernel");
    return true;
}

template <typename T>
static int launch_wgrad_direct(const WgradArgs& a, cudaStream_t st) {
    const TapGeom& g = a.g;
    const long long M = (long long)g.N * g.OH * g.OW;
    const int subs = ((g.Nc + 3) / 4) * ((g.K + 3) / 4);
    const int ntaps = g.prob[0].ntaps;
    int SUB = subs <= 1 ? 1 : subs <= 4 ? 4 : subs <= 16 ? 16 : 64;
    int groups = (subs + SUB - 1) / SUB;
    const int L = 256 / SUB;
    long long want = 8LL * num_sms();
    long long split = (want + (long long)ntaps * groups - 1) / ((long long)ntaps * groups);
    long long maxsplit = (M + 8LL * L - 1) / (8LL * L);      // >= 8 pixels per thread
    if (split > maxsplit) split = maxsplit;
    if (split < 1) split = 1;
    if (split > 65535) split = 65535;
    dim3 grid(ntaps, (unsigned)split, groups);
    if (SUB == 1) SVRS_LAUNCH((wgrad_direct_kernel<T, 1>), grid, 256, 0, st, a);
    else if (SUB == 4) SVRS_LAUNCH((wgrad_direct_kernel<T, 4>), grid, 256, 0, st, a);
    else if (SUB == 16) SVRS_LAUNCH((wgrad_direct_kernel<T, 16>), grid, 256, 0, st, a);
    else SVRS_LAUNCH((wgrad_direct_kernel<T, 64>), grid, 256, 0, st, a);
    return check_launch("wgrad_direct_kernel");
}

static int launch_wgrad(WgradArgs& a, int dtype, int ksplit, cudaStream_t st) {
    const TapGeom& g = a.g;
    long long M = (long long)g.N * g.OH * g.OW;
    if (M == 0) return 0;
    if ((g.Nc <= 16 || g.K <= 16) && ksplit <= 0) {
        a.ksplit = 1;
        int rc = 0;
        if (dtype == SVRS_F32 ? try_launch_wgrad_narrow<float>(a, st, rc) : try_launch_wgrad_narrow<__nv_bfloat16>(a, st, rc)) return rc;
        return dtype == SVRS_F32 ? launch_wgrad_direct<float>(a, st) : launch_wgrad_direct<__nv_bfloat16>(a, st);
    }
    int tiles = ((g.Nc + 63) / 64) * ((g.K + 63) / 64);
    int ntaps = g.prob[0].ntaps;
    if (ksplit <= 0) {
        long long want = 4LL * num_sms();
        long long base = (long long)tiles * ntaps;
        ksplit = (int)((want + base - 1) / base);
        long long maxsplit = (M + 255) / 256;  // at least 256 pixels per CTA
        if (ksplit > maxsplit) ksplit = (int)maxsplit;
        if (ksplit < 1) ksplit = 1;
    }
    a.ksplit = ksplit;
    dim3 grid(tiles, ntaps, ksplit);
    if (dtype == SVRS_F32) SVRS_LAUNCH((wgrad_taps_kernel<float>), grid, 256, 0, st, a);
    else SVRS_LAUNCH((wgrad_taps_kernel<__nv_bfloat16>), grid, 256, 0, st, a);
    return check_launch("wgrad_taps_kernel");
}

// vectorised variant: thread t owns channel quad (t % cg) and row lane (t / cg), cg = C/4 divides 256
template <typename T>
__global__ void __launch_bounds__(256) colsum_vec_kernel(const T* __restrict__ x, long long M, int C,
                                                          float* __restrict__ out, long long rows_per_block) {
    pdl_entry();
    __shared__ float red[256][4];
    const int cg = C / 4;
    const int q = threadIdx.x % cg, lane = threadIdx.x / cg, lanes = 256 / cg;
    const long long r0 = (long long)blockIdx.x * rows_per_block;
    long long r1 = r0 + rows_per_block;
    if (r1 > M) r1 = M;
    float4 s = make_float4(0.f, 0.f, 0.f, 0.f);
    for (long long r = r0 + lane; r < r1; r += lanes) {
        float4 v = ld4(x + r * C + q * 4);
        s.x += v.x; s.y += v.y; s.z += v.z; s.w += v.w;
    }
    red[threadIdx.x][0] = s.x; red[threadIdx.x][1] = s.y; red[threadIdx.x][2] = s.z; red[threadIdx.x][3] = s.w;
    __syncthreads();
    if (lane == 0) {
        for (int l = 1; l < lanes; ++l) {
            s.x += red[l * cg + q][0]; s.y += red[l * cg + q][1]; s.z += red[l * cg + q][2]; s.w += red[l * cg + q][3];
        }
        atomicAdd(&out[q * 4 + 0], s.x); atomicAdd(&out[q * 4 + 1], s.y);
        atomicAdd(&out[q * 4 + 2], s.z); atomicAdd(&out[q * 4 + 3], s.w);
    }
}

static int launch_colsum(const void* x, int dtype, long long M, int C, float* out, cudaStream_t st) {
    if (M == 0 || C == 0) return 0;
    if (C % 4 == 0 && C / 4 <= 256 && 256 % (C / 4) == 0) {
        int lanes = 256 / (C / 4);
        long long blocks = (M + (long long)lanes * 16 - 1) / ((long long)lanes * 16);
        long long cap = 4LL * num_sms();
        if (blocks > cap) blocks = cap;
        if (blocks < 1) blocks = 1;
        long long rpb = (M + blocks - 1) / blocks;
        blocks = (M + rpb - 1) / rpb;
        if (dtype == SVRS_F32) SVRS_LAUNCH((colsum_vec_kernel<float>), (unsigned)blocks, 256, 0, st, (const float*)x, M, C, out, rpb);
        else SVRS_LAUNCH((colsum_vec_kernel<__nv_bfloat16>), (unsigned)blocks, 256, 0, st, (const __nv_bfloat16*)x, M, C, out, rpb);
        return check_launch("colsum_vec_kernel");
    }
    long long blocks = (M + 511) / 512;
    long long cap = 8LL * num_sms();
    if (blocks > cap) blocks = cap;
    long long rpb = (M + blocks - 1) / blocks;
    blocks = (M + rpb - 1) / rpb;
    if (dtype == SVRS_F32) SVRS_LAUNCH((colsum_kernel<float>), (unsigned)blocks, 256, 0, st, (const float*)x, M, C, out, rpb);
    else SVRS_LAUNCH((colsum_kernel<__nv_bfloat16>), (unsigned)blocks, 256, 0, st, (const __nv_bfloat16*)x, M, C, out, rpb);
    return check_launch("colsum_kernel");
}

}  // namespace svrs

namespace svrs {
bool tc_supported(int dtype, int K, int Nc, int OW, int OH);
int launch_conv_tc(int form, const void* in, const void* w_nk, const float* bias, void* out, int N, int H, int W, int Cr, int Cw,
                   int act, const ConvExtra& ex, cudaStream_t st);
bool wgrad_tc_supported(int dtype, int Ca, int Cb, int OW, int OH);
int launch_wgrad_tc(const TapGeom& g, const void* gmat, const void* x, float* dw, int packed, int KK, float* db, cudaStream_t st);
bool wgrad_halo_supported(const TapGeom& g, int KK);
int launch_wgrad3_halo(const TapGeom& g, const void* gmat, const void* x, float* dw, int packed, float* db, cudaStream_t st);
static int g_tc_enabled = 1;
int g_tc_enabled_narrow = 1;
static inline bool use_tc(const void* w_nk, int dtype, int K, int Nc, int OW, int OH) {
    // layers with both channel counts <= 16 are HBM-bound streaming ops: the per-pixel SIMT kernel beats a padded MMA
    return g_tc_enabled && w_nk != nullptr && !((K == 4 || Nc == 4) && K <= 16 && Nc <= 16) && tc_supported(dtype, K, Nc, OW, OH);
}
}  // namespace svrs

using namespace svrs;

static bool dtype_ok(int d) { return d == SVRS_F32 || d == SVRS_BF16; }

namespace svrs { void set_halo_mode(int m); }
extern "C" void svrs_set_tc_enabled(int enabled) { svrs::g_tc_enabled = enabled; svrs::g_tc_enabled_narrow = enabled; }
extern "C" void svrs_set_halo_mode(int mode) { svrs::set_halo_mode(mode); }
extern "C" int svrs_tc_would_run(int dtype, int K, int Nc, int OH, int OW) {
    return svrs::g_tc_enabled && svrs::tc_supported(dtype, K, Nc, OW, OH) ? 1 : 0;
}

extern "C" int svrs_conv2d_fprop_ex(const void* x, const void* w_kn, const void* w_nk, const float* bias, void* y, int dtype,
                                    int out_dtype, float* y_nchw, int64_t y_nchw_ld, double* bn_sums,
                                    int N, int H, int W, int Cin, int Cout, int ksize, int act, void* stream) {
    SVRS_CHECK_ARG(x && w_kn && (y || y_nchw) && dtype_ok(dtype) && dtype_ok(out_dtype), "conv2d_fprop: null pointer or bad dtype");
    SVRS_CHECK_ARG(ksize == 3 || (ksize == 4 && H % 2 == 0 && W % 2 == 0), "conv2d_fprop: ksize must be 3, or 4 with even H,W");
    SVRS_CHECK_ARG(N >= 0 && H > 0 && W > 0 && Cin > 0 && Cout > 0, "conv2d_fprop: bad dims");
    if (N > 0 && use_tc(w_nk, dtype, Cin, Cout, ksize == 3 ? W : W / 2, ksize == 3 ? H : H / 2)) {
        if (out_dtype != dtype) { set_error("conv2d_fprop_ex: the tensor-core kernels store bf16 (use y_nchw for an fp32 copy)"); return SVRS_E_UNSUPPORTED; }
        ConvExtra ex;
        ex.out2 = y_nchw; ex.out2_ld = y_nchw_ld; ex.bn_sums = bn_sums;
        return launch_conv_tc(ksize == 3 ? 0 : 2, x, w_nk, bias, y, N, H, W, Cin, Cout, act, ex, (cudaStream_t)stream);
    }
    if (y_nchw || !y) { set_error("conv2d_fprop_ex: the NCHW second output needs the tensor-core kernel (Cin=%d Cout=%d)", Cin, Cout); return SVRS_E_UNSUPPORTED; }
    ConvArgs a;
    a.in = x; a.out = y; a.w = w_kn; a.bias = bias; a.act = act; a.bn_sums = bn_sums;
    if (ksize == 3) geom_conv3(a.g, N, H, W, Cin, Cout, false);
    else geom_conv4s2(a.g, N, H, W, Cin, Cout);
    return launch_conv(a, dtype, (cudaStream_t)stream, out_dtype);
}

extern "C" int svrs_conv2d_fprop(const void* x, const void* w_kn, const void* w_nk, const float* bias, void* y, int dtype,
                                 int N, int H, int W, int Cin, int Cout, int ksize, int act, void* stream) {
    return svrs_conv2d_fprop_ex(x, w_kn, w_nk, bias, y, dtype, dtype, nullptr, 0, nullptr, N, H, W, Cin, Cout, ksize, act, stream);
}

extern "C" int svrs_conv2d_dgrad(const void* dy, const void* w_kn, const void* w_nk, void* dx, int dtype,
                                 int N, int H, int W, int Cin, int Cout, int ksize, void* stream) {
    SVRS_CHECK_ARG(dy && w_kn && dx && dtype_ok(dtype), "conv2d_dgrad: null pointer or bad dtype");
    SVRS_CHECK_ARG(ksize == 3 || (ksize == 4 && H % 2 == 0 && W % 2 == 0), "conv2d_dgrad: ksize must be 3, or 4 with even H,W");
    if (N > 0 && ksize == 3 && use_tc(w_nk, dtype, Cout, Cin, W, H))
        return launch_conv_tc(1, dy, w_nk, nullptr, dx, N, H, W, Cout, Cin, SVRS_ACT_NONE, ConvExtra(), (cudaStream_t)stream);
    if (N > 0 && ksize == 4 && use_tc(w_nk, dtype, Cout, Cin, W / 2, H / 2))     // per-parity output grid == coarse grid
        return launch_conv_tc(3, dy, w_nk, nullptr, dx, N, H / 2, W / 2, Cout, Cin, SVRS_ACT_NONE, ConvExtra(), (cudaStream_t)stream);
    ConvArgs a;
    a.in = dy; a.out = dx; a.w = w_kn; a.bias = nullptr; a.act = SVRS_ACT_NONE; a.bn_sums = nullptr;
    if (ksize == 3) geom_conv3(a.g, N, H, W, Cout, Cin, true);
    else geom_convT4s2(a.g, N, H / 2, W / 2, Cout, Cin);
    return launch_conv(a, dtype, (cudaStream_t)stream);
}

extern "C" int svrs_convT2d_fprop_ex(const void* x, const void* w_kn, const void* w_nk, const float* bias, void* y, int dtype,
                                     double* bn_sums, int N, int H, int W, int Cin, int Cout, int act, void* stream) {
    SVRS_CHECK_ARG(x && w_kn && y && dtype_ok(dtype), "convT2d_fprop: null pointer or bad dtype");
    if (N > 0 && use_tc(w_nk, dtype, Cin, Cout, W, H)) {
        ConvExtra ex;
        ex.bn_sums = bn_sums;
        return launch_conv_tc(3, x, w_nk, bias, y, N, H, W, Cin, Cout, act, ex, (cudaStream_t)stream);
    }
    ConvArgs a;
    a.in = x; a.out = y; a.w = w_kn; a.bias = bias; a.act = act; a.bn_sums = bn_sums;
    geom_convT4s2(a.g, N, H, W, Cin, Cout);
    return launch_conv(a, dtype, (cudaStream_t)stream);
}

extern "C" int svrs_convT2d_fprop(const void* x, const void* w_kn, const void* w_nk, const float* bias, void* y, int dtype,
                                  int N, int H, int W, int Cin, int Cout, int act, void* stream) {
    return svrs_convT2d_fprop_ex(x, w_kn, w_nk, bias, y, dtype, nullptr, N, H, W, Cin, Cout, act, stream);
}

extern "C" int svrs_convT2d_dgrad(const void* dy, const void* w_kn, const void* w_nk, void* dx, int dtype,
                                  int N, int H, int W, int Cin, int Cout, void* stream) {
    SVRS_CHECK_ARG(dy && w_kn && dx && dtype_ok(dtype), "convT2d_dgrad: null pointer or bad dtype");
    if (N > 0 && use_tc(w_nk, dtype, Cout, Cin, W, H))
        return launch_conv_tc(2, dy, w_nk, nullptr, dx, N, 2 * H, 2 * W, Cout, Cin, SVRS_ACT_NONE, ConvExtra(), (cudaStream_t)stream);
    ConvArgs a;
    a.in = dy; a.out = dx; a.w = w_kn; a.bias = nullptr; a.act = SVRS_ACT_NONE; a.bn_sums = nullptr;
    geom_conv4s2(a.g, N, 2 * H, 2 * W, Cout, Cin);
    return launch_conv(a, dtype, (cudaStream_t)stream);
}

extern "C" int svrs_conv2d_wgrad(const void* x, const void* dy, float* dw, float* dw_packed, float* db, int dtype,
                                 int N, int H, int W, int Cin, int Cout, int ksize, int ksplit, void* stream) {
    SVRS_CHECK_ARG(x && dy && dtype_ok(dtype), "conv2d_wgrad: null pointer or bad dtype");
    SVRS_CHECK_ARG(ksize == 3 || (ksize == 4 && H % 2 == 0 && W % 2 == 0), "conv2d_wgrad: bad ksize");
    int rc = 0;
    if (dw) {
        WgradArgs a;
        a.gmat = dy; a.x = x; a.dw = dw; a.KK = ksize * ksize;
        if (ksize == 3) geom_conv3(a.g, N, H, W, Cin, Cout, false);
        else geom_conv4s2(a.g, N, H, W, Cin, Cout);
        // the tensor-core kernels fold the bias gradient (column sums of dy) into their idle epilogue warps
        const bool fold_db = db != nullptr && Cout % 8 == 0;
        if (g_tc_enabled && N > 0 && dtype == SVRS_BF16 && wgrad_halo_supported(a.g, a.KK)) {
            rc = launch_wgrad3_halo(a.g, dy, x, dw_packed ? dw_packed : dw, dw_packed != nullptr, fold_db ? db : nullptr, (cudaStream_t)stream);
            if (fold_db) db = nullptr;
        } else if (g_tc_enabled && N > 0 && wgrad_tc_supported(dtype, Cout, Cin, a.g.OW, a.g.OH)) {
            rc = launch_wgrad_tc(a.g, dy, x, dw_packed ? dw_packed : dw, dw_packed != nullptr, a.KK, fold_db ? db : nullptr, (cudaStream_t)stream);
            if (fold_db) db = nullptr;
        } else if (g_tc_enabled_narrow && N > 0 && ksplit <= 0 && wgrad_narrow_mma_takes(a.g, dtype)) {
            rc = launch_wgrad_narrow_mma(a, db, (cudaStream_t)stream);      // bias gradient folded in (one more MMA)
            db = nullptr;
        } else
            rc = launch_wgrad(a, dtype, ksplit, (cudaStream_t)stream);
        if (rc) return rc;
    }
    if (db) {
        int s = ksize == 3 ? 1 : 2;
        rc = launch_colsum(dy, dtype, (long long)N * (H / s) * (W / s), Cout, db, (cudaStream_t)stream);
    }
    return rc;
}

extern "C" int svrs_convT2d_wgrad(const void* x, const void* dy, float* dw, float* dw_packed, float* db, int dtype,
                                  int N, int H, int W, int Cin, int Cout, int ksplit, void* stream) {
    SVRS_CHECK_ARG(x && dy && dtype_ok(dtype), "convT2d_wgrad: null pointer or bad dtype");
    int rc = 0;
    if (dw) {
        // adjoint view: the coarse input x sits on the output grid of a k4s2 conv that reads the fine dy.
        WgradArgs a;
        a.gmat = x; a.x = dy; a.dw = dw; a.KK = 16;
        geom_conv4s2(a.g, N, 2 * H, 2 * W, Cout, Cin);
        if (g_tc_enabled && N > 0 && wgrad_tc_supported(dtype, Cin, Cout, a.g.OW, a.g.OH))
            rc = launch_wgrad_tc(a.g, x, dy, dw_packed ? dw_packed : dw, dw_packed != nullptr, 16, nullptr, (cudaStream_t)stream);
        else
            rc = launch_wgrad(a, dtype, ksplit, (cudaStream_t)stream);
        if (rc) return rc;
    }
    if (db) rc = launch_colsum(dy, dtype, (long long)N * 4 * H * W, Cout, db, (cudaStream_t)stream);
    return rc;
}

// Which layout the weight-gradient kernels leave in `dw_packed` for this problem: 1 = the tcgen05 kernels take it and
// accumulate the per-tap packed scratch [tap][d1][d0]; 0 = a SIMT kernel takes it and accumulates torch layout into `dw`.
// (Same decision tree as svrs_conv2d_wgrad / svrs_convT2d_wgrad; the fused optimiser reads the gradient accordingly.)
extern "C" int svrs_conv2d_wgrad_layout(int dtype, int N, int H, int W, int Cin, int Cout, int ksize) {
    if (!(ksize == 3 || (ksize == 4 && H % 2 == 0 && W % 2 == 0)) || N <= 0) return 0;
    TapGeom g;
    if (ksize == 3) geom_conv3(g, N, H, W, Cin, Cout, false);
    else geom_conv4s2(g, N, H, W, Cin, Cout);
    if (g_tc_enabled && dtype == SVRS_BF16 && wgrad_halo_supported(g, ksize * ksize)) return 1;
    if (g_tc_enabled && wgrad_tc_supported(dtype, Cout, Cin, g.OW, g.OH)) return 1;
    return 0;
}
extern "C" int svrs_convT2d_wgrad_layout(int dtype, int N, int H, int W, int Cin, int Cout) {
    if (N <= 0) return 0;
    TapGeom g;
    geom_conv4s2(g, N, 2 * H, 2 * W, Cout, Cin);
    return (g_tc_enabled && wgrad_tc_supported(dtype, Cin, Cout, g.OW, g.OH)) ? 1 : 0;
}

// Host-only: dump the tap geometry of a conv form so the host logic can be verified without a GPU.
// form: 0 conv3 fprop, 1 conv3 dgrad, 2 conv4s2 (fprop / convT dgrad), 3 convT4s2 (fprop / conv4s2 dgrad).
// H, W are the dims of the tensor being READ.  Layout of `out` (int64):
//   [0..10] = N, OH, OW, IH, IW, K, Nc, nprob, o_sn, o_sy, o_sx ; [11..13] = i_sn, i_sy, i_sx ;
//   then per problem: out_off, ntaps, then per tap: in_off, w_off, dy, dx.   Returns #int64 written, <0 on error.
extern "C" int svrs_debug_tap_geometry(int form, int N, int H, int W, int Cr, int Cw, int64_t* out, int cap) {
    SVRS_CHECK_ARG(out && form >= 0 && form <= 3, "debug_tap_geometry: bad args");
    TapGeom g;
    if (form == 0) geom_conv3(g, N, H, W, Cr, Cw, false);
    else if (form == 1) geom_conv3(g, N, H, W, Cr, Cw, true);
    else if (form == 2) geom_conv4s2(g, N, H, W, Cr, Cw);
    else geom_convT4s2(g, N, H, W, Cr, Cw);
    int n = 0;
    auto put = [&](long long v) { if (n < cap) out[n] = v; ++n; };
    put(g.N); put(g.OH); put(g.OW); put(g.IH); put(g.IW); put(g.K); put(g.Nc); put(g.nprob);
    put(g.o_sn); put(g.o_sy); put(g.o_sx); put(g.i_sn); put(g.i_sy); put(g.i_sx);
    for (int p = 0; p < g.nprob; ++p) {
        put(g.prob[p].out_off); put(g.prob[p].ntaps);
        for (int t = 0; t < g.prob[p].ntaps; ++t) {
            put(g.prob[p].taps[t].in_off); put(g.prob[p].taps[t].w_off); put(g.prob[p].taps[t].dy); put(g.prob[p].taps[t].dx);
        }
    }
    SVRS_CHECK_ARG(n <= cap, "debug_tap_geometry: buffer too small (%d needed)", n);
    return n;
}
