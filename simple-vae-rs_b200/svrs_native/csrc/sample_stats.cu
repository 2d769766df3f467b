// sample_stats.cu - inference side of the path (BASELINE config 5; SURVEY 8.4 rows a14 / f4):
//   * sample_latents_kernel : the S posterior draws z_s = mu3 + eps_s * exp(0.5 * lv3) of every patch (Philox on device)
//                             written straight into the decoder_x input rows [y_enc(b) | z(b, s)]  (cond_vae.py:305-318)
//   * sample_tail_kernel    : the LAST decoder_x layer (nn.Conv2d(16, 4, 3, padding=1) + Sigmoid, cond_vae.py:79-80) over the
//                             S draws of a patch with the per-pixel statistics of BaseVAE.task (models/base.py:305-313, 341)
//                             accumulated WHILE the draws are produced: streaming Welford mean / M2 per channel plus the
//                             |d| and d^2 sums against the target.  The [S, 4, P, P] sample stack never reaches HBM.
// Both are streaming kernels (HBM / FP32-issue bound); nothing here is GEMM-shaped enough for the tensor pipe (16 -> 4 ch).
#include "common.cuh"

namespace svrs {

// Philox4x32-10 + Box-Muller, same generator and counter layout as elbo.cu (counter = (idx4 lo, idx4 hi, stream, step))
__device__ __forceinline__ uint4 ss_philox(uint4 c, uint2 k) {
    const uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u, W0 = 0x9E3779B9u, W1 = 0xBB67AE85u;
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        uint32_t hi0 = __umulhi(M0, c.x), lo0 = M0 * c.x;
        uint32_t hi1 = __umulhi(M1, c.z), lo1 = M1 * c.z;
        c = make_uint4(hi1 ^ c.y ^ k.x, lo1, hi0 ^ c.w ^ k.y, lo0);
        k.x += W0;
        k.y += W1;
    }
    return c;
}
__device__ __forceinline__ float4 ss_normal4(uint64_t seed, uint32_t stream_id, uint64_t idx4, uint32_t step) {
    uint4 r = ss_philox(make_uint4((uint32_t)idx4, (uint32_t)(idx4 >> 32), stream_id, step),
                        make_uint2((uint32_t)seed, (uint32_t)(seed >> 32)));
    const float two_m32 = 2.3283064365386963e-10f;
    float u1a = fminf(((float)r.x + 1.0f) * two_m32, 1.0f), u2a = (float)r.y * two_m32;
    float u1b = fminf(((float)r.z + 1.0f) * two_m32, 1.0f), u2b = (float)r.w * two_m32;
    float ra = sqrtf(-2.0f * logf(u1a)), rb = sqrtf(-2.0f * logf(u1b));
    float sa, ca, sb, cb;
    sincospif(2.0f * u2a, &sa, &ca);
    sincospif(2.0f * u2b, &sb, &cb);
    return make_float4(ra * ca, ra * sa, rb * cb, rb * sb);
}

// stack[(b*S + s)][0:Wz] = yflat[b][:],  stack[(b*S + s)][Wz:2Wz] = mu3[b] + eps(b*S + s) * exp(0.5 * lv3[b])
__global__ void __launch_bounds__(256) sample_latents_kernel(const float* __restrict__ mu3, const float* __restrict__ lv3, long long ld3,
                                                              const float* __restrict__ yflat, long long ldy,
                                                              const float* __restrict__ eps, float* __restrict__ stack,
                                                              int B, int S, int Wz, uint64_t seed, uint32_t sid, uint64_t sample_offset,
                                                              const long long* __restrict__ step_ptr) {
    pdl_entry();
    const int wq = Wz / 4;
    const long long nvec = (long long)B * S * wq;
    const uint32_t step = step_ptr ? (uint32_t)(*step_ptr) : 0u;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < nvec; i += (long long)gridDim.x * blockDim.x) {
        const long long row = i / wq;
        const int j = (int)(i % wq) * 4;
        const int b = (int)(row / S);
        const float4 mu = *reinterpret_cast<const float4*>(mu3 + (long long)b * ld3 + j);
        const float4 lv = *reinterpret_cast<const float4*>(lv3 + (long long)b * ld3 + j);
        float4 e;
        if (eps) e = *reinterpret_cast<const float4*>(eps + row * Wz + j);
        else e = ss_normal4(seed, sid, ((sample_offset + (uint64_t)row) * (uint64_t)Wz + j) >> 2, step);
        float4 z;
        z.x = fmaf(e.x, expf(0.5f * lv.x), mu.x);
        z.y = fmaf(e.y, expf(0.5f * lv.y), mu.y);
        z.z = fmaf(e.z, expf(0.5f * lv.z), mu.z);
        z.w = fmaf(e.w, expf(0.5f * lv.w), mu.w);
        float* dst = stack + row * 2 * Wz;
        *reinterpret_cast<float4*>(dst + Wz + j) = z;
        *reinterpret_cast<float4*>(dst + j) = *reinterpret_cast<const float4*>(yflat + (long long)b * ldy + j);
    }
}

// ---------------------------------------------------------------------------------------------- tail + statistics
constexpr int TS_CIN = 16, TS_COUT = 4, TS_NPART = 10;   // partial record per pixel: mean[4], M2[4], sum|d|, sum d^2

struct TailArgs {
    const void* x;        // [B*S][H][W][16]
    const void* w;        // KN pack [9][16][4]
    const float* bias;    // [4] or null
    const float* target;  // NHWC fp32 [B][H][W][4] or null
    float* part;          // [B][splits][TS_NPART][H*W]
    float* sample0;       // NCHW fp32 [B][4][H][W] or null: the first draw of every patch
    int B, S, H, W, splits;
};

template <typename T> __device__ __forceinline__ void load16(const T* p, float (&v)[16]);
template <> __device__ __forceinline__ void load16<float>(const float* p, float (&v)[16]) {
#pragma unroll
    for (int k = 0; k < 16; k += 4) {
        float4 a = *reinterpret_cast<const float4*>(p + k);
        v[k] = a.x; v[k + 1] = a.y; v[k + 2] = a.z; v[k + 3] = a.w;
    }
}
template <> __device__ __forceinline__ void load16<__nv_bfloat16>(const __nv_bfloat16* p, float (&v)[16]) {
#pragma unroll
    for (int k = 0; k < 16; k += 8) {
        uint4 r = *reinterpret_cast<const uint4*>(p + k);
        const uint32_t u[4] = {r.x, r.y, r.z, r.w};
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            v[k + 2 * q] = __uint_as_float(u[q] << 16);
            v[k + 2 * q + 1] = __uint_as_float(u[q] & 0xffff0000u);
        }
    }
}

template <typename T>
__global__ void __launch_bounds__(128) sample_tail_kernel(const __grid_constant__ TailArgs a) {
    pdl_entry();
    __shared__ __align__(16) float ws[9 * TS_CIN * TS_COUT];
    for (int i = threadIdx.x; i < 9 * TS_CIN * TS_COUT; i += 128) ws[i] = Cvt<T>::to_f(reinterpret_cast<const T*>(a.w)[i]);
    __syncthreads();
    const int HW = a.H * a.W;
    const int pix = blockIdx.x * 128 + threadIdx.x;
    if (pix >= HW) return;
    const int b = blockIdx.y, sp = blockIdx.z;
    const int oy = pix / a.W, ox = pix % a.W;
    const int s0 = (int)((long long)a.S * sp / a.splits), s1 = (int)((long long)a.S * (sp + 1) / a.splits);
    float bz[TS_COUT], tg[TS_COUT] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
    for (int c = 0; c < TS_COUT; ++c) bz[c] = a.bias ? a.bias[c] : 0.f;
    if (a.target) {
        const float4 t = *reinterpret_cast<const float4*>(a.target + ((long long)b * HW + pix) * 4);
        tg[0] = t.x; tg[1] = t.y; tg[2] = t.z; tg[3] = t.w;
    }
    // which of the nine taps fall inside the map (zero padding) - the same for every draw
    int toff[9];
    bool tok[9];
#pragma unroll
    for (int t = 0; t < 9; ++t) {
        const int iy = oy + t / 3 - 1, ix = ox + t % 3 - 1;
        tok[t] = iy >= 0 && iy < a.H && ix >= 0 && ix < a.W;
        toff[t] = (iy * a.W + ix) * TS_CIN;
    }
    float mean[TS_COUT] = {0.f, 0.f, 0.f, 0.f}, m2[TS_COUT] = {0.f, 0.f, 0.f, 0.f};
    float sabs = 0.f, ssq = 0.f;
    const T* xb = reinterpret_cast<const T*>(a.x) + ((long long)b * a.S + s0) * HW * TS_CIN;
    for (int s = s0; s < s1; ++s, xb += (long long)HW * TS_CIN) {
        float acc[TS_COUT];
#pragma unroll
        for (int c = 0; c < TS_COUT; ++c) acc[c] = bz[c];
#pragma unroll
        for (int t = 0; t < 9; ++t) {
            if (!tok[t]) continue;
            float xv[16];
            load16<T>(xb + toff[t], xv);
            const float* wt = ws + t * TS_CIN * TS_COUT;
#pragma unroll
            for (int k = 0; k < TS_CIN; ++k) {
                const float4 wv = *reinterpret_cast<const float4*>(wt + k * TS_COUT);
                acc[0] = fmaf(xv[k], wv.x, acc[0]); acc[1] = fmaf(xv[k], wv.y, acc[1]);
                acc[2] = fmaf(xv[k], wv.z, acc[2]); acc[3] = fmaf(xv[k], wv.w, acc[3]);
            }
        }
        const float inv_n = 1.0f / (float)(s - s0 + 1);
#pragma unroll
        for (int c = 0; c < TS_COUT; ++c) {
            const float v = 1.0f / (1.0f + expf(-acc[c]));          // Sigmoid (cond_vae.py:80)
            acc[c] = v;
            const float dl = v - mean[c];
            mean[c] += dl * inv_n;
            m2[c] = fmaf(dl, v - mean[c], m2[c]);
            const float d = v - tg[c];
            sabs += fabsf(d);
            ssq = fmaf(d, d, ssq);
        }
        if (a.sample0 && s == 0) {
#pragma unroll
            for (int c = 0; c < TS_COUT; ++c) a.sample0[((long long)b * TS_COUT + c) * HW + pix] = acc[c];
        }
    }
    float* pp = a.part + ((long long)(b * a.splits + sp) * TS_NPART) * HW + pix;
#pragma unroll
    for (int c = 0; c < TS_COUT; ++c) { pp[(long long)c * HW] = mean[c]; pp[(long long)(4 + c) * HW] = m2[c]; }
    pp[8LL * HW] = sabs;
    pp[9LL * HW] = ssq;
}

struct TailOut {
    const float* part;
    const float* target;
    float *mean, *std_map, *mae, *mse, *bias_map;
    int B, S, HW, splits;
};

// merge the per-split Welford partials (Chan et al.) and emit the maps of BaseVAE.task (models/base.py:305-313, 341)
__global__ void __launch_bounds__(256) sample_tail_finalize_kernel(const __grid_constant__ TailOut a) {
    pdl_entry();
    const int pix = blockIdx.x * 256 + threadIdx.x;
    if (pix >= a.HW) return;
    const int b = blockIdx.y;
    float mean[4] = {0.f, 0.f, 0.f, 0.f}, m2[4] = {0.f, 0.f, 0.f, 0.f}, sabs = 0.f, ssq = 0.f;
    float na = 0.f;
    for (int sp = 0; sp < a.splits; ++sp) {
        const int s0 = (int)((long long)a.S * sp / a.splits), s1 = (int)((long long)a.S * (sp + 1) / a.splits);
        const float nb = (float)(s1 - s0);
        if (nb == 0.f) continue;
        const float* pp = a.part + ((long long)(b * a.splits + sp) * TS_NPART) * a.HW + pix;
        const float n = na + nb;
#pragma unroll
        for (int c = 0; c < 4; ++c) {
            const float mb = pp[(long long)c * a.HW], qb = pp[(long long)(4 + c) * a.HW];
            const float dl = mb - mean[c];
            mean[c] += dl * (nb / n);
            m2[c] += qb + dl * dl * (na * nb / n);
        }
        sabs += pp[8LL * a.HW];
        ssq += pp[9LL * a.HW];
        na = n;
    }
    const long long o = (long long)b * a.HW + pix;
    float sd = 0.f, bias = 0.f;
    float tg[4] = {0.f, 0.f, 0.f, 0.f};
    if (a.target) {
        const float4 t = *reinterpret_cast<const float4*>(a.target + o * 4);
        tg[0] = t.x; tg[1] = t.y; tg[2] = t.z; tg[3] = t.w;
    }
#pragma unroll
    for (int c = 0; c < 4; ++c) {
        if (a.mean) a.mean[((long long)b * 4 + c) * a.HW + pix] = mean[c];
        sd += sqrtf(m2[c] / (na - 1.0f));            // torch.std: unbiased (S = 1 -> nan, like the reference)
        bias += tg[c] - mean[c];
    }
    if (a.std_map) a.std_map[o] = 0.25f * sd;
    if (a.target) {
        if (a.mae) a.mae[o] = sabs / (4.0f * na);
        if (a.mse) a.mse[o] = ssq / (4.0f * na);
        if (a.bias_map) a.bias_map[o] = 0.25f * bias;
    }
}

}  // namespace svrs

using namespace svrs;

extern "C" int svrs_sample_latents(const float* mu3, const float* lv3, int64_t ld3, const float* yflat, int64_t ldy,
                                   const float* eps, float* stack, int B, int S, int Wz, uint64_t seed, int stream_id,
                                   uint64_t sample_offset, const int64_t* step_ptr, void* stream) {
    SVRS_CHECK_ARG(mu3 && lv3 && yflat && stack, "sample_latents: null pointer");
    SVRS_CHECK_ARG(B > 0 && S > 0 && Wz > 0 && Wz % 4 == 0 && ld3 % 4 == 0 && ldy % 4 == 0, "sample_latents: B, S > 0 and Wz, ld3, ldy multiples of 4 required");
    SVRS_CHECK_ARG(ld3 >= Wz && ldy >= Wz, "sample_latents: row strides ld3 (%lld) and ldy (%lld) must be >= Wz (%d)", (long long)ld3, (long long)ldy, Wz);
    SVRS_CHECK_ARG(al16(mu3) && al16(lv3) && al16(yflat) && al16(eps) && al16(stack), "sample_latents: pointers must be 16B aligned");
    const long long nvec = (long long)B * S * (Wz / 4);
    const int blocks = (int)((nvec + 255) / 256 < (long long)num_sms() * 8 ? (nvec + 255) / 256 : (long long)num_sms() * 8);
    SVRS_LAUNCH(sample_latents_kernel, blocks, 256, 0, (cudaStream_t)stream, mu3, lv3, (long long)ld3, yflat, (long long)ldy, eps, stack,
                B, S, Wz, seed, (uint32_t)stream_id, sample_offset, reinterpret_cast<const long long*>(step_ptr));
    return check_launch("sample_latents_kernel");
}

// default split of the S draws of a pixel over CTAs: enough CTAs for two waves (pixels/128 x B x splits >= 2 x SMs) with at
// least 8 draws per split
extern "C" int svrs_sample_tail_splits(int B, int S, int H, int W) {
    const long long base = (long long)((H * W + 127) / 128) * (B < 1 ? 1 : B);
    int splits = (int)((2LL * num_sms() + base - 1) / base);
    if (splits > S / 8) splits = S / 8;
    return splits < 1 ? 1 : splits;
}

extern "C" int64_t svrs_sample_tail_scratch_floats(int B, int H, int W, int splits) {
    return (int64_t)B * (splits < 1 ? 1 : splits) * TS_NPART * H * W;
}

extern "C" int svrs_sample_tail_stats(const void* x, int dtype, const void* w_kn, const float* bias, const float* target_nhwc,
                                      int B, int S, int H, int W, int Cin, int Cout, int splits, float* scratch,
                                      float* mean_nchw, float* std_map, float* mae_map, float* mse_map, float* bias_map,
                                      float* sample0_nchw, void* stream) {
    SVRS_CHECK_ARG(x && w_kn && scratch, "sample_tail_stats: null pointer");
    SVRS_CHECK_ARG(dtype == SVRS_F32 || dtype == SVRS_BF16, "sample_tail_stats: bad dtype %d", dtype);
    SVRS_CHECK_ARG(al16(x) && al16(target_nhwc), "sample_tail_stats: x and target_nhwc must be 16B aligned");
    SVRS_CHECK_ARG(B > 0 && S > 0 && H > 0 && W > 0, "sample_tail_stats: B, S, H, W must be positive");
    if (Cin != TS_CIN || Cout != TS_COUT) {
        set_error("sample_tail_stats: the fused tail is the 16 -> 4 conv of decoder_x (cond_vae.py:79); got %d -> %d", Cin, Cout);
        return SVRS_E_UNSUPPORTED;
    }
    SVRS_CHECK_ARG(splits >= 1 && splits <= S, "sample_tail_stats: splits (%d) must be in [1, S = %d]", splits, S);
    TailArgs a;
    a.x = x; a.w = w_kn; a.bias = bias; a.target = target_nhwc; a.part = scratch; a.sample0 = sample0_nchw;
    a.B = B; a.S = S; a.H = H; a.W = W; a.splits = splits;
    dim3 grid((H * W + 127) / 128, B, splits);
    if (dtype == SVRS_F32) SVRS_LAUNCH(sample_tail_kernel<float>, grid, 128, 0, (cudaStream_t)stream, a);
    else SVRS_LAUNCH(sample_tail_kernel<__nv_bfloat16>, grid, 128, 0, (cudaStream_t)stream, a);
    int rc = check_launch("sample_tail_kernel");
    if (rc) return rc;
    TailOut o;
    o.part = scratch; o.target = target_nhwc; o.mean = mean_nchw; o.std_map = std_map; o.mae = mae_map; o.mse = mse_map;
    o.bias_map = bias_map; o.B = B; o.S = S; o.HW = H * W; o.splits = splits;
    SVRS_LAUNCH(sample_tail_finalize_kernel, dim3((H * W + 255) / 256, B), 256, 0, (cudaStream_t)stream, o);
    return check_launch("sample_tail_finalize_kernel");
}
