// elbo.cu - reparameterisation (Philox4x32-10 on device) and the fused Gaussian ELBO reductions.
// These kernels are HBM-bound: every operand is read exactly once with 128-bit accesses, partial sums
// go warp-shuffle -> shared -> one double atomic per block per term.
#include "common.cuh"

namespace svrs {

// ---------------------------------------------------------------- Philox4x32-10 + Box-Muller
__device__ __forceinline__ uint4 philox4x32_10(uint4 c, uint2 k) {
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

// 4 normals for elements [4*idx4, 4*idx4+3] of (row-major) stream `stream_id`.
__device__ __forceinline__ float4 philox_normal4(uint64_t seed, uint32_t stream_id, uint64_t idx4, uint32_t step) {
    uint4 r = philox4x32_10(make_uint4((uint32_t)idx4, (uint32_t)(idx4 >> 32), stream_id, step),
                            make_uint2((uint32_t)seed, (uint32_t)(seed >> 32)));
    const float two_m32 = 2.3283064365386963e-10f;
    float u1a = ((float)r.x + 1.0f) * two_m32;  // (0,1]
    float u2a = (float)r.y * two_m32;
    float u1b = ((float)r.z + 1.0f) * two_m32;
    float u2b = (float)r.w * two_m32;
    u1a = fminf(u1a, 1.0f); u1b = fminf(u1b, 1.0f);
    float ra = sqrtf(-2.0f * logf(u1a)), rb = sqrtf(-2.0f * logf(u1b));
    float sa, ca, sb, cb;
    sincospif(2.0f * u2a, &sa, &ca);
    sincospif(2.0f * u2b, &sb, &cb);
    return make_float4(ra * ca, ra * sa, rb * cb, rb * sb);
}

// eps for element (global row gb, column j..j+3): flat index = gb*Wd + j (Wd % 4 == 0)
__device__ __forceinline__ float4 eps4(const float* eps, long long local_off, uint64_t seed, uint32_t sid,
                                       uint64_t gflat, uint32_t step) {
    if (eps) return *reinterpret_cast<const float4*>(eps + local_off);
    return philox_normal4(seed, sid, gflat >> 2, step);
}

__global__ void __launch_bounds__(256) reparam_fwd_kernel(const float* __restrict__ enc, const float* __restrict__ eps,
                                                           float* __restrict__ z, long long z_ld, float* __restrict__ eps_out, int B, int Wd,
                                                           uint64_t seed, uint32_t sid, uint64_t sample_offset,
                                                           const long long* __restrict__ step_ptr) {
    pdl_entry();
    const long long nvec = (long long)B * Wd / 4;
    const int wq = Wd / 4;
    const uint32_t step = step_ptr ? (uint32_t)(*step_ptr) : 0u;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < nvec; i += (long long)gridDim.x * blockDim.x) {
        int b = (int)(i / wq), j = (int)(i % wq) * 4;
        float4 mu = *reinterpret_cast<const float4*>(enc + (long long)b * 2 * Wd + j);
        float4 lv = *reinterpret_cast<const float4*>(enc + (long long)b * 2 * Wd + Wd + j);
        float4 e = eps4(eps, (long long)b * Wd + j, seed, sid, (sample_offset + b) * (uint64_t)Wd + j, step);
        float4 o;
        o.x = fmaf(e.x, expf(0.5f * lv.x), mu.x);
        o.y = fmaf(e.y, expf(0.5f * lv.y), mu.y);
        o.z = fmaf(e.z, expf(0.5f * lv.z), mu.z);
        o.w = fmaf(e.w, expf(0.5f * lv.w), mu.w);
        *reinterpret_cast<float4*>(z + (long long)b * z_ld + j) = o;
        if (eps_out) *reinterpret_cast<float4*>(eps_out + (long long)b * Wd + j) = e;
    }
}

__global__ void __launch_bounds__(256) reparam_bwd_kernel(const float* __restrict__ enc, const float* __restrict__ eps,
                                                           const float* __restrict__ dz, long long dz_ld, float* __restrict__ denc, int B, int Wd,
                                                           uint64_t seed, uint32_t sid, uint64_t sample_offset,
                                                           const long long* __restrict__ step_ptr) {
    pdl_entry();
    const long long nvec = (long long)B * Wd / 4;
    const int wq = Wd / 4;
    const uint32_t step = step_ptr ? (uint32_t)(*step_ptr) : 0u;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < nvec; i += (long long)gridDim.x * blockDim.x) {
        int b = (int)(i / wq), j = (int)(i % wq) * 4;
        float4 lv = *reinterpret_cast<const float4*>(enc + (long long)b * 2 * Wd + Wd + j);
        float4 e = eps4(eps, (long long)b * Wd + j, seed, sid, (sample_offset + b) * (uint64_t)Wd + j, step);
        float4 g = *reinterpret_cast<const float4*>(dz + (long long)b * dz_ld + j);
        float4* pm = reinterpret_cast<float4*>(denc + (long long)b * 2 * Wd + j);
        float4* pl = reinterpret_cast<float4*>(denc + (long long)b * 2 * Wd + Wd + j);
        float4 m = *pm, l = *pl;
        m.x += g.x; m.y += g.y; m.z += g.z; m.w += g.w;
        l.x += g.x * e.x * 0.5f * expf(0.5f * lv.x);
        l.y += g.y * e.y * 0.5f * expf(0.5f * lv.y);
        l.z += g.z * e.z * 0.5f * expf(0.5f * lv.z);
        l.w += g.w * e.w * 0.5f * expf(0.5f * lv.w);
        *pm = m;
        *pl = l;
    }
}

__global__ void philox_normal_kernel(float* __restrict__ out, int B, int Wd, uint64_t seed, uint32_t sid, uint64_t sample_offset,
                                     const long long* __restrict__ step_ptr) {
    pdl_entry();
    const long long nvec = (long long)B * Wd / 4;
    const uint32_t step = step_ptr ? (uint32_t)(*step_ptr) : 0u;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < nvec; i += (long long)gridDim.x * blockDim.x) {
        uint64_t gflat = sample_offset * (uint64_t)Wd + (uint64_t)i * 4;
        *reinterpret_cast<float4*>(out + i * 4) = philox_normal4(seed, sid, gflat >> 2, step);
    }
}

// ---------------------------------------------------------------- ELBO forward reductions
// dtype-generic vector access (the branch is uniform; these kernels are HBM-bound)
__device__ __forceinline__ float4 ld4_dt(const void* p, int dt, long long i4) {
    return dt == SVRS_F32 ? ld4(reinterpret_cast<const float*>(p) + i4 * 4) : ld4(reinterpret_cast<const __nv_bfloat16*>(p) + i4 * 4);
}
__device__ __forceinline__ float ld1_dt(const void* p, int dt, long long i) {
    return dt == SVRS_F32 ? reinterpret_cast<const float*>(p)[i] : __bfloat162float(reinterpret_cast<const __nv_bfloat16*>(p)[i]);
}
__device__ __forceinline__ void st4_dt(void* p, int dt, long long i4, float4 v) {
    if (dt == SVRS_F32) st4(reinterpret_cast<float*>(p) + i4 * 4, v); else st4(reinterpret_cast<__nv_bfloat16*>(p) + i4 * 4, v);
}
__device__ __forceinline__ void st1_dt(void* p, int dt, long long i, float v) {
    if (dt == SVRS_F32) reinterpret_cast<float*>(p)[i] = v; else reinterpret_cast<__nv_bfloat16*>(p)[i] = __float2bfloat16_rn(v);
}

// recon (dtype dtr) and target (dtype dtt) share a layout; each is read once
__device__ __forceinline__ float ssq_segment(const void* __restrict__ r, int dtr, const void* __restrict__ t, int dtt, long long n,
                                             long long gtid, long long gsize) {
    float s = 0.f;
    long long nvec = n / 4;
    for (long long i = gtid; i < nvec; i += gsize) {
        float4 a = ld4_dt(r, dtr, i), b = ld4_dt(t, dtt, i);
        float d0 = a.x - b.x, d1 = a.y - b.y, d2 = a.z - b.z, d3 = a.w - b.w;
        s += d0 * d0 + d1 * d1 + d2 * d2 + d3 * d3;
    }
    for (long long i = nvec * 4 + gtid; i < n; i += gsize) {
        float d = ld1_dt(r, dtr, i) - ld1_dt(t, dtt, i);
        s += d * d;
    }
    return s;
}

struct ElboArgs {
    const void *rx, *x, *ry, *y;
    int dtx, dty;      // dtype of recon_x / recon_y
    int dttx, dtty;    // dtype of the targets x / y
    long long nx, ny;
    const float *mu1, *lv1, *mu2, *lv2, *mu3, *lv3;
    long long ld1, ld2, ld3;
    int W1, W2, B;
};

__global__ void __launch_bounds__(256) elbo_fwd_kernel(const __grid_constant__ ElboArgs a, double* __restrict__ acc) {
    pdl_entry();
    const long long gtid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long gsize = (long long)gridDim.x * blockDim.x;
    float s[4] = {0.f, 0.f, 0.f, 0.f};
    if (a.nx > 0) {
        s[0] = ssq_segment(a.rx, a.dtx, a.x, a.dttx, a.nx, gtid, gsize);
    }
    if (a.ny > 0) {
        s[1] = ssq_segment(a.ry, a.dty, a.y, a.dtty, a.ny, gtid, gsize);
    }
    if (a.mu1) {
        const int wq = a.W1 / 4;
        const long long nvec = (long long)a.B * wq;
        for (long long i = gtid; i < nvec; i += gsize) {
            long long o = (i / wq) * a.ld1 + (i % wq) * 4;
            float4 m = *reinterpret_cast<const float4*>(a.mu1 + o), l = *reinterpret_cast<const float4*>(a.lv1 + o);
            s[2] += (m.x * m.x + expf(l.x) - 1.f - l.x) + (m.y * m.y + expf(l.y) - 1.f - l.y) +
                    (m.z * m.z + expf(l.z) - 1.f - l.z) + (m.w * m.w + expf(l.w) - 1.f - l.w);
        }
    }
    if (a.mu2) {
        const int wq = a.W2 / 4;
        const long long nvec = (long long)a.B * wq;
        for (long long i = gtid; i < nvec; i += gsize) {
            long long r = i / wq, c = (i % wq) * 4;
            float4 m2 = *reinterpret_cast<const float4*>(a.mu2 + r * a.ld2 + c);
            float4 l2 = *reinterpret_cast<const float4*>(a.lv2 + r * a.ld2 + c);
            float4 m3 = *reinterpret_cast<const float4*>(a.mu3 + r * a.ld3 + c);
            float4 l3 = *reinterpret_cast<const float4*>(a.lv3 + r * a.ld3 + c);
            float q2[4] = {l2.x, l2.y, l2.z, l2.w}, q3[4] = {l3.x, l3.y, l3.z, l3.w};
            float p2[4] = {m2.x, m2.y, m2.z, m2.w}, p3[4] = {m3.x, m3.y, m3.z, m3.w};
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                float d = p2[j] - p3[j];
                s[3] += (q3[j] - q2[j] - 1.f) + expf(q2[j] - q3[j]) + d * d * expf(-q3[j]);
            }
        }
    }
    __shared__ double red[8][4];
    const int lane = threadIdx.x % 32, wid = threadIdx.x / 32;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        double v = warp_sum((double)s[k]);
        if (lane == 0) red[wid][k] = v;
    }
    __syncthreads();
    if (threadIdx.x < 4) {
        double v = 0;
#pragma unroll
        for (int w = 0; w < 8; ++w) v += red[w][threadIdx.x];
        if (v != 0.0) atomicAdd(&acc[threadIdx.x], v);
    }
}

__global__ void elbo_finalize_kernel(const double* __restrict__ acc, long long nx, long long ny, int B,
                                     const float* __restrict__ gammas, float* __restrict__ out) {
    pdl_entry();
    if (threadIdx.x != 0 || blockIdx.x != 0) return;
    float gx = gammas[0], gy = gammas[1];
    // loss/cond_vae_loss.py:43-49: n * (mean((r-x)^2) / (2 g^2) + log g)
    out[0] = nx > 0 ? (float)nx * ((float)(acc[0] / (double)nx) / (2.f * gx * gx) + logf(gx)) : 0.f;
    out[1] = 0.5f * (float)(acc[2] / (double)B);
    out[2] = ny > 0 ? (float)ny * ((float)(acc[1] / (double)ny) / (2.f * gy * gy) + logf(gy)) : 0.f;
    out[3] = 0.5f * (float)(acc[3] / (double)B);
    out[4] = ((out[0] + out[1]) + out[2]) + out[3];   // loss = mse_x + kld_u + mse_y + kld_z (cond_vae.py:346)
}

// ---------------------------------------------------------------- ELBO backward
struct ElboBwdArgs {
    ElboArgs f;
    void *drx, *dry;
    int dtdx, dtdy;    // dtype of d_recon_x / d_recon_y
    int act;           // SVRS_ACT_SIGMOID: recon = sigmoid(pre) and d_recon_* receives the gradient wrt `pre`
    float *dmu1, *dlv1, *dmu2, *dlv2, *dmu3, *dlv3;
    long long dld1, dld2, dld3;
    const double* acc;
    const float* gammas;
    const float* gout;
    float* dgammas;
};

__device__ __forceinline__ float nll_d(float r, float t, float coef, int act) {
    float g = (r - t) * coef;
    if (act == SVRS_ACT_SIGMOID) g = g * r * (1.f - r);      // chain through the decoder's final nn.Sigmoid (cond_vae.py:80,143)
    return g;
}
__device__ __forceinline__ void nll_bwd_segment(const void* __restrict__ r, int dtr, const void* __restrict__ t, int dtt,
                                                void* __restrict__ dr, int dtd, long long n, float coef, int act,
                                                long long gtid, long long gsize) {
    long long nvec = n / 4;
    for (long long i = gtid; i < nvec; i += gsize) {
        float4 a = ld4_dt(r, dtr, i), b = ld4_dt(t, dtt, i);
        st4_dt(dr, dtd, i, make_float4(nll_d(a.x, b.x, coef, act), nll_d(a.y, b.y, coef, act), nll_d(a.z, b.z, coef, act), nll_d(a.w, b.w, coef, act)));
    }
    for (long long i = nvec * 4 + gtid; i < n; i += gsize)
        st1_dt(dr, dtd, i, nll_d(ld1_dt(r, dtr, i), ld1_dt(t, dtt, i), coef, act));
}

__global__ void __launch_bounds__(256) elbo_bwd_kernel(const __grid_constant__ ElboBwdArgs a) {
    pdl_entry();
    const ElboArgs& f = a.f;
    const long long gtid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long gsize = (long long)gridDim.x * blockDim.x;
    const float gx = a.gammas[0], gy = a.gammas[1];
    const float g_msex = a.gout[0], g_klu = a.gout[1], g_msey = a.gout[2], g_klz = a.gout[3];
    if (gtid == 0 && a.dgammas) {
        // d/dg [ ssq/(2 g^2) + n log g ] = -ssq/g^3 + n/g
        a.dgammas[0] = f.nx > 0 ? g_msex * ((float)(-a.acc[0]) / (gx * gx * gx) + (float)f.nx / gx) : 0.f;
        a.dgammas[1] = f.ny > 0 ? g_msey * ((float)(-a.acc[1]) / (gy * gy * gy) + (float)f.ny / gy) : 0.f;
    }
    if (f.nx > 0 && a.drx) {
        float c = g_msex / (gx * gx);
        nll_bwd_segment(f.rx, f.dtx, f.x, f.dttx, a.drx, a.dtdx, f.nx, c, a.act, gtid, gsize);
    }
    if (f.ny > 0 && a.dry) {
        float c = g_msey / (gy * gy);
        nll_bwd_segment(f.ry, f.dty, f.y, f.dtty, a.dry, a.dtdy, f.ny, c, a.act, gtid, gsize);
    }
    const float invB = 1.0f / (float)f.B;
    if (f.mu1 && (a.dmu1 || a.dlv1)) {
        const int wq = f.W1 / 4;
        const long long nvec = (long long)f.B * wq;
        const float k = g_klu * invB;
        for (long long i = gtid; i < nvec; i += gsize) {
            long long r = i / wq, c = (i % wq) * 4;
            if (a.dmu1) {
                float4 m = *reinterpret_cast<const float4*>(f.mu1 + r * f.ld1 + c);
                *reinterpret_cast<float4*>(a.dmu1 + r * a.dld1 + c) = make_float4(k * m.x, k * m.y, k * m.z, k * m.w);
            }
            if (a.dlv1) {
                float4 l = *reinterpret_cast<const float4*>(f.lv1 + r * f.ld1 + c);
                *reinterpret_cast<float4*>(a.dlv1 + r * a.dld1 + c) =
                    make_float4(k * 0.5f * (expf(l.x) - 1.f), k * 0.5f * (expf(l.y) - 1.f), k * 0.5f * (expf(l.z) - 1.f), k * 0.5f * (expf(l.w) - 1.f));
            }
        }
    }
    if (f.mu2) {
        const int wq = f.W2 / 4;
        const long long nvec = (long long)f.B * wq;
        const float k = g_klz * invB;
        for (long long i = gtid; i < nvec; i += gsize) {
            long long r = i / wq, c = (i % wq) * 4;
            float4 m2 = *reinterpret_cast<const float4*>(f.mu2 + r * f.ld2 + c);
            float4 l2 = *reinterpret_cast<const float4*>(f.lv2 + r * f.ld2 + c);
            float4 m3 = *reinterpret_cast<const float4*>(f.mu3 + r * f.ld3 + c);
            float4 l3 = *reinterpret_cast<const float4*>(f.lv3 + r * f.ld3 + c);
            float q2[4] = {l2.x, l2.y, l2.z, l2.w}, q3[4] = {l3.x, l3.y, l3.z, l3.w};
            float p2[4] = {m2.x, m2.y, m2.z, m2.w}, p3[4] = {m3.x, m3.y, m3.z, m3.w};
            float o_m2[4], o_l2[4], o_l3[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                float d = p2[j] - p3[j];
                float e23 = expf(q2[j] - q3[j]);
                float em3 = expf(-q3[j]);
                o_m2[j] = k * d * em3;
                o_l2[j] = k * 0.5f * (e23 - 1.f);
                o_l3[j] = k * 0.5f * (1.f - e23 - d * d * em3);
            }
            if (a.dmu2) *reinterpret_cast<float4*>(a.dmu2 + r * a.dld2 + c) = make_float4(o_m2[0], o_m2[1], o_m2[2], o_m2[3]);
            if (a.dlv2) *reinterpret_cast<float4*>(a.dlv2 + r * a.dld2 + c) = make_float4(o_l2[0], o_l2[1], o_l2[2], o_l2[3]);
            if (a.dmu3) *reinterpret_cast<float4*>(a.dmu3 + r * a.dld3 + c) = make_float4(-o_m2[0], -o_m2[1], -o_m2[2], -o_m2[3]);
            if (a.dlv3) *reinterpret_cast<float4*>(a.dlv3 + r * a.dld3 + c) = make_float4(o_l3[0], o_l3[1], o_l3[2], o_l3[3]);
        }
    }
}

static unsigned ew_grid2(long long nvec) {
    long long b = (nvec + 255) / 256, cap = 8LL * num_sms();
    if (b > cap) b = cap;
    if (b < 1) b = 1;
    return (unsigned)b;
}

}  // namespace svrs

using namespace svrs;

extern "C" int svrs_reparam_fwd(const float* enc, const float* eps, float* z, int64_t z_ld, float* eps_out, int B, int Wd,
                                uint64_t seed, uint32_t stream_id, uint64_t sample_offset, const int64_t* step_ptr, void* stream) {
    SVRS_CHECK_ARG(enc && z && B >= 0 && Wd > 0 && Wd % 4 == 0 && z_ld % 4 == 0 && z_ld >= Wd, "reparam_fwd: bad args (Wd, z_ld %% 4 != 0?)");
    SVRS_CHECK_ARG(al16(enc) && al16(eps) && al16(z) && al16(eps_out), "reparam_fwd: pointers must be 16B aligned");
    if (B == 0) return 0;
    SVRS_LAUNCH((reparam_fwd_kernel), ew_grid2((long long)B * Wd / 4), 256, 0, (cudaStream_t)stream, enc, eps, z, z_ld, eps_out, B, Wd, seed, stream_id, sample_offset, (const long long*)step_ptr);
    return check_launch("reparam_fwd");
}

extern "C" int svrs_reparam_bwd(const float* enc, const float* eps, const float* dz, int64_t dz_ld, float* denc, int B, int Wd,
                                uint64_t seed, uint32_t stream_id, uint64_t sample_offset, const int64_t* step_ptr, void* stream) {
    SVRS_CHECK_ARG(enc && dz && denc && B >= 0 && Wd > 0 && Wd % 4 == 0 && dz_ld % 4 == 0 && dz_ld >= Wd, "reparam_bwd: bad args");
    SVRS_CHECK_ARG(al16(enc) && al16(eps) && al16(dz) && al16(denc), "reparam_bwd: pointers must be 16B aligned");
    if (B == 0) return 0;
    SVRS_LAUNCH((reparam_bwd_kernel), ew_grid2((long long)B * Wd / 4), 256, 0, (cudaStream_t)stream, enc, eps, dz, dz_ld, denc, B, Wd, seed, stream_id, sample_offset, (const long long*)step_ptr);
    return check_launch("reparam_bwd");
}

extern "C" int svrs_philox_normal(float* out, int B, int Wd, uint64_t seed, uint32_t stream_id,
                                  uint64_t sample_offset, const int64_t* step_ptr, void* stream) {
    SVRS_CHECK_ARG(out && B >= 0 && Wd > 0 && Wd % 4 == 0 && al16(out), "philox_normal: bad args");
    if (B == 0) return 0;
    SVRS_LAUNCH((philox_normal_kernel), ew_grid2((long long)B * Wd / 4), 256, 0, (cudaStream_t)stream, out, B, Wd, seed, stream_id, sample_offset, (const long long*)step_ptr);
    return check_launch("philox_normal");
}

static int fill_elbo_args(ElboArgs& a, const void* recon_x, const void* x, int dt_x, int dt_tx, int64_t n_x,
                          const void* recon_y, const void* y, int dt_y, int dt_ty, int64_t n_y,
                          const float* mu1, const float* lv1, int64_t ld1, int W1,
                          const float* mu2, const float* lv2, int64_t ld2,
                          const float* mu3, const float* lv3, int64_t ld3, int W2, int B) {
    SVRS_CHECK_ARG(B > 0, "elbo: B must be > 0");
    SVRS_CHECK_ARG(n_x == 0 || (recon_x && x), "elbo: recon_x/x null");
    SVRS_CHECK_ARG(n_y == 0 || (recon_y && y), "elbo: recon_y/y null");
    SVRS_CHECK_ARG((dt_x == SVRS_F32 || dt_x == SVRS_BF16) && (dt_y == SVRS_F32 || dt_y == SVRS_BF16) &&
                   (dt_tx == SVRS_F32 || dt_tx == SVRS_BF16) && (dt_ty == SVRS_F32 || dt_ty == SVRS_BF16), "elbo: bad dtype");
    SVRS_CHECK_ARG(al16(recon_x) && al16(x) && al16(recon_y) && al16(y), "elbo: image pointers must be 16B aligned");
    if (mu1) {
        SVRS_CHECK_ARG(lv1 && W1 > 0 && W1 % 4 == 0 && ld1 % 4 == 0 && al16(mu1) && al16(lv1), "elbo: kl1 needs W1 > 0, W1,ld1 %% 4 == 0 and 16B alignment");
        SVRS_CHECK_ARG(ld1 >= W1, "elbo: kl1 row stride ld1 (%lld) < W1 (%d)", (long long)ld1, W1);
    }
    if (mu2) {
        SVRS_CHECK_ARG(lv2 && mu3 && lv3 && W2 > 0 && W2 % 4 == 0 && ld2 % 4 == 0 && ld3 % 4 == 0 && al16(mu2) && al16(lv2) && al16(mu3) && al16(lv3),
                       "elbo: kl23 needs W2 > 0, W2,ld2,ld3 %% 4 == 0 and 16B alignment");
        SVRS_CHECK_ARG(ld2 >= W2 && ld3 >= W2, "elbo: kl23 row strides ld2 (%lld) / ld3 (%lld) < W2 (%d)", (long long)ld2, (long long)ld3, W2);
    }
    a.rx = recon_x; a.x = x; a.ry = recon_y; a.y = y; a.dtx = dt_x; a.dty = dt_y; a.dttx = dt_tx; a.dtty = dt_ty; a.nx = n_x; a.ny = n_y;
    a.mu1 = mu1; a.lv1 = lv1; a.mu2 = mu2; a.lv2 = lv2; a.mu3 = mu3; a.lv3 = lv3;
    a.ld1 = ld1; a.ld2 = ld2; a.ld3 = ld3; a.W1 = W1; a.W2 = W2; a.B = B;
    return 0;
}

extern "C" int svrs_elbo_fwd(const void* recon_x, const void* x, int dt_x, int dt_tx, int64_t n_x,
                             const void* recon_y, const void* y, int dt_y, int dt_ty, int64_t n_y,
                             const float* mu1, const float* lv1, int64_t ld1, int W1,
                             const float* mu2, const float* lv2, int64_t ld2,
                             const float* mu3, const float* lv3, int64_t ld3, int W2,
                             int B, double* acc, void* stream) {
    SVRS_CHECK_ARG(acc, "elbo_fwd: acc null");
    ElboArgs a;
    int rc = fill_elbo_args(a, recon_x, x, dt_x, dt_tx, n_x, recon_y, y, dt_y, dt_ty, n_y, mu1, lv1, ld1, W1, mu2, lv2, ld2, mu3, lv3, ld3, W2, B);
    if (rc) return rc;
    long long work = (n_x > n_y ? n_x : n_y) / 4;
    long long w2 = (long long)B * (W2 > W1 ? W2 : W1) / 4;
    if (w2 > work) work = w2;
    SVRS_LAUNCH((elbo_fwd_kernel), ew_grid2(work), 256, 0, (cudaStream_t)stream, a, acc);
    return check_launch("elbo_fwd");
}

extern "C" int svrs_elbo_finalize(const double* acc, int64_t n_x, int64_t n_y, int B, const float* gammas,
                                  float* out5, void* stream) {
    SVRS_CHECK_ARG(acc && gammas && out5 && B > 0, "elbo_finalize: bad args");
    SVRS_LAUNCH((elbo_finalize_kernel), 1, 32, 0, (cudaStream_t)stream, acc, n_x, n_y, B, gammas, out5);
    return check_launch("elbo_finalize");
}

extern "C" int svrs_elbo_bwd(const void* recon_x, const void* x, int dt_x, int dt_tx, int64_t n_x, void* d_recon_x, int dt_dx,
                             const void* recon_y, const void* y, int dt_y, int dt_ty, int64_t n_y, void* d_recon_y, int dt_dy,
                             const float* mu1, const float* lv1, int64_t ld1, int W1, float* d_mu1, float* d_lv1, int64_t dld1,
                             const float* mu2, const float* lv2, int64_t ld2, float* d_mu2, float* d_lv2, int64_t dld2,
                             const float* mu3, const float* lv3, int64_t ld3, int W2, float* d_mu3, float* d_lv3, int64_t dld3,
                             int B, const double* acc, const float* gammas, const float* gout, float* d_gammas,
                             int act, void* stream) {
    SVRS_CHECK_ARG(acc && gammas && gout, "elbo_bwd: acc/gammas/gout null");
    SVRS_CHECK_ARG((dt_dx == SVRS_F32 || dt_dx == SVRS_BF16) && (dt_dy == SVRS_F32 || dt_dy == SVRS_BF16) &&
                   (act == SVRS_ACT_NONE || act == SVRS_ACT_SIGMOID), "elbo_bwd: bad gradient dtype / act");
    ElboBwdArgs a;
    int rc = fill_elbo_args(a.f, recon_x, x, dt_x, dt_tx, n_x, recon_y, y, dt_y, dt_ty, n_y, mu1, lv1, ld1, W1, mu2, lv2, ld2, mu3, lv3, ld3, W2, B);
    if (rc) return rc;
    SVRS_CHECK_ARG(al16(d_recon_x) && al16(d_recon_y) && al16(d_mu1) && al16(d_lv1) && al16(d_mu2) && al16(d_lv2) && al16(d_mu3) && al16(d_lv3),
                   "elbo_bwd: gradient pointers must be 16B aligned");
    SVRS_CHECK_ARG(dld1 % 4 == 0 && dld2 % 4 == 0 && dld3 % 4 == 0, "elbo_bwd: gradient strides %% 4");
    SVRS_CHECK_ARG(!mu1 || !(d_mu1 || d_lv1) || dld1 >= W1, "elbo_bwd: gradient row stride dld1 (%lld) < W1 (%d)", (long long)dld1, W1);
    SVRS_CHECK_ARG(!mu2 || !(d_mu2 || d_lv2) || dld2 >= W2, "elbo_bwd: gradient row stride dld2 (%lld) < W2 (%d)", (long long)dld2, W2);
    SVRS_CHECK_ARG(!mu2 || !(d_mu3 || d_lv3) || dld3 >= W2, "elbo_bwd: gradient row stride dld3 (%lld) < W2 (%d)", (long long)dld3, W2);
    a.drx = d_recon_x; a.dry = d_recon_y; a.dtdx = dt_dx; a.dtdy = dt_dy; a.act = act;
    a.dmu1 = d_mu1; a.dlv1 = d_lv1; a.dmu2 = d_mu2; a.dlv2 = d_lv2; a.dmu3 = d_mu3; a.dlv3 = d_lv3;
    a.dld1 = dld1; a.dld2 = dld2; a.dld3 = dld3;
    a.acc = acc; a.gammas = gammas; a.gout = gout; a.dgammas = d_gammas;
    long long work = (n_x > n_y ? n_x : n_y) / 4;
    long long w2 = (long long)B * (W2 > W1 ? W2 : W1) / 4;
    if (w2 > work) work = w2;
    SVRS_LAUNCH((elbo_bwd_kernel), ew_grid2(work), 256, 0, (cudaStream_t)stream, a);
    return check_launch("elbo_bwd");
}
