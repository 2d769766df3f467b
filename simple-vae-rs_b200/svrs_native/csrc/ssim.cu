// ssim.cu - mean structural similarity of image pairs, the Metrics/SSIM* values of evaluate() (cond_vae.py:387-525,
// vae.py:142-216): skimage.metrics.structural_similarity(a, b, win_size=win, data_range=R, channel_axis=0) with its defaults
// (uniform window, sample covariance, K1 = 0.01, K2 = 0.03), per image of an NCHW fp32 batch.
//   * ssim_kernel          : one CTA per band of SS_BAND output rows of one (n, c) plane.  The band's input rows of both planes
//                            are staged in shared memory (one contiguous range of the plane), the five window sums
//                            (a, b, a^2, b^2, ab) are built by a vertical running-sum pass over the staged rows followed by a
//                            horizontal running-sum pass over the vertical sums, and the band's SSIM values are summed in double
//                            into one partial per CTA.
//   * ssim_finalize_kernel : folds the partials of every image in a fixed order (no atomics: bitwise reproducible).
// Only interior positions are computed (every window fully inside the plane), as skimage crops (win-1)/2 from every edge.
// Precision: the window sums are fp32 over a - k, b - k with k = the plane's first pixel (the shift of bn.cu's bf16 statistics):
// near-saturated planes would otherwise lose the variance to cancellation in E[a^2] - E[a]^2; the running sums subtract exactly
// the value they added, and the SSIM formula itself runs in double.
#include "common.cuh"

namespace svrs {

constexpr int SS_THREADS = 256;
constexpr int SS_BAND = 16;       // output rows per CTA
constexpr int SS_VP = 18;         // pitch of a column of vertical sums: the horizontal pass reads 16 rows x 2 chunks per warp,
                                  // 18 * SS_HCOLS = 144 = 16 (mod 32) banks apart -> conflict-free
constexpr int SS_HCOLS = 8;       // output columns per thread of the horizontal pass
constexpr int SS_SMEM_MAX = 227 * 1024;

static inline long long ssim_smem_bytes(int W, int win) {
    return 4LL * W * (2LL * (SS_BAND + win - 1) + 5LL * SS_VP);
}

struct SsimArgs {
    const float* a;
    const float* b;
    double* part;      // [N*C*nbands]
    int H, W, win, nbands;
    double c1, c2, cov_norm;
};

__global__ void __launch_bounds__(SS_THREADS) ssim_kernel(const __grid_constant__ SsimArgs p) {
    pdl_entry();
    extern __shared__ __align__(16) float ss_smem[];
    const int H = p.H, W = p.W, win = p.win;
    const int OH = H - win + 1, OW = W - win + 1;
    const int band = blockIdx.x % p.nbands;
    const long long plane = blockIdx.x / p.nbands;
    const int oy0 = band * SS_BAND;
    const int nr = min(SS_BAND, OH - oy0);          // output rows of this band
    const int nin = nr + win - 1;                   // staged input rows
    float* sa = ss_smem;                            // [nin][W]   a - ka
    float* sb = sa + (SS_BAND + win - 1) * W;       // [nin][W]   b - kb
    float* vs = sb + (SS_BAND + win - 1) * W;       // [5][W][SS_VP] vertical window sums of a, b, a^2, b^2, ab

    const float* ga = p.a + plane * H * W;
    const float* gb = p.b + plane * H * W;
    const float ka = __ldg(ga), kb = __ldg(gb);
    ga += (long long)oy0 * W;
    gb += (long long)oy0 * W;
    const int n = nin * W;
    if (((reinterpret_cast<uintptr_t>(ga) | reinterpret_cast<uintptr_t>(gb)) & 15) == 0 && (W & 3) == 0) {   // sb 16-B aligned too
        for (int i = threadIdx.x; i < n / 4; i += SS_THREADS) {
            float4 u = __ldg(reinterpret_cast<const float4*>(ga) + i), v = __ldg(reinterpret_cast<const float4*>(gb) + i);
            u.x -= ka; u.y -= ka; u.z -= ka; u.w -= ka;
            v.x -= kb; v.y -= kb; v.z -= kb; v.w -= kb;
            reinterpret_cast<float4*>(sa)[i] = u;
            reinterpret_cast<float4*>(sb)[i] = v;
        }
    } else {
        for (int i = threadIdx.x; i < n; i += SS_THREADS) {
            sa[i] = __ldg(ga + i) - ka;
            sb[i] = __ldg(gb + i) - kb;
        }
    }
    __syncthreads();

    // vertical pass: item = (input column x, group of consecutive output rows); a running sum down the group
    const int ngroups = max(1, min(nr, SS_THREADS / W));
    const int rpg = (nr + ngroups - 1) / ngroups;
    for (int it = threadIdx.x; it < W * ngroups; it += SS_THREADS) {
        const int x = it % W, r0 = (it / W) * rpg, r1 = min(nr, r0 + rpg);
        if (r0 >= r1) continue;
        float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f, s4 = 0.f;
        for (int i = r0; i < r0 + win; ++i) {
            const float u = sa[i * W + x], v = sb[i * W + x];
            s0 += u; s1 += v; s2 = fmaf(u, u, s2); s3 = fmaf(v, v, s3); s4 = fmaf(u, v, s4);
        }
        float* o = vs + x * SS_VP;
        for (int r = r0;; ++r) {
            o[r] = s0;
            o[W * SS_VP + r] = s1;
            o[2 * W * SS_VP + r] = s2;
            o[3 * W * SS_VP + r] = s3;
            o[4 * W * SS_VP + r] = s4;
            if (r + 1 >= r1) break;
            const float u = sa[(r + win) * W + x], v = sb[(r + win) * W + x];     // row entering the window
            const float uo = sa[r * W + x], vo = sb[r * W + x];                   // row leaving it
            s0 = (s0 + u) - uo; s1 = (s1 + v) - vo;
            s2 = fmaf(-uo, uo, fmaf(u, u, s2));
            s3 = fmaf(-vo, vo, fmaf(v, v, s3));
            s4 = fmaf(-uo, vo, fmaf(u, v, s4));
        }
    }
    __syncthreads();

    // horizontal pass: item = (output row r, chunk of SS_HCOLS output columns); rows vary fastest within a warp
    const double inv_np = 1.0 / ((double)win * win);
    const double c1 = p.c1, c2 = p.c2, cn = p.cov_norm, dka = ka, dkb = kb;
    const int nchunks = (OW + SS_HCOLS - 1) / SS_HCOLS;
    double acc = 0.0;
    for (int it = threadIdx.x; it < SS_BAND * nchunks; it += SS_THREADS) {
        const int r = it % SS_BAND, x0 = (it / SS_BAND) * SS_HCOLS;
        if (r >= nr) continue;
        const int x1 = min(OW, x0 + SS_HCOLS);
        const float* v0 = vs + r;
        float s[5] = {0.f, 0.f, 0.f, 0.f, 0.f};
        for (int x = x0; x < x0 + win; ++x) {
#pragma unroll
            for (int q = 0; q < 5; ++q) s[q] += v0[(q * W + x) * SS_VP];
        }
        for (int x = x0;; ++x) {
            const double mx = s[0] * inv_np, my = s[1] * inv_np;                  // shifted means
            const double vx = cn * (s[2] * inv_np - mx * mx);
            const double vy = cn * (s[3] * inv_np - my * my);
            const double vxy = cn * (s[4] * inv_np - mx * my);
            const double ux = mx + dka, uy = my + dkb;
            acc += ((2.0 * ux * uy + c1) * (2.0 * vxy + c2)) / ((ux * ux + uy * uy + c1) * (vx + vy + c2));
            if (x + 1 >= x1) break;
#pragma unroll
            for (int q = 0; q < 5; ++q) s[q] = (s[q] + v0[(q * W + x + win) * SS_VP]) - v0[(q * W + x) * SS_VP];
        }
    }
    acc = warp_sum(acc);
    double* wsum = reinterpret_cast<double*>(ss_smem);     // the staged rows are dead since the vertical pass
    if ((threadIdx.x & 31) == 0) wsum[threadIdx.x >> 5] = acc;
    __syncthreads();
    if (threadIdx.x == 0) {
        double t = 0.0;
#pragma unroll
        for (int w = 0; w < SS_THREADS / 32; ++w) t += wsum[w];
        p.part[blockIdx.x] = t;
    }
}

// out[n] = mean over c of (sum of the plane's band partials) / interior positions
__global__ void __launch_bounds__(128) ssim_finalize_kernel(const double* __restrict__ part, double* __restrict__ out, int N, int C,
                                                             int nbands, double inv_pos) {
    pdl_entry();
    const int n = blockIdx.x * 128 + threadIdx.x;
    if (n >= N) return;
    const double* pp = part + (long long)n * C * nbands;
    double t = 0.0;
    for (int c = 0; c < C; ++c) {
        double s = 0.0;
        for (int k = 0; k < nbands; ++k) s += pp[c * nbands + k];
        t += s * inv_pos;
    }
    out[n] = t / C;
}

}  // namespace svrs

using namespace svrs;

static int ssim_check(int N, int C, int H, int W, int win) {
    SVRS_CHECK_ARG(N >= 0 && C > 0, "ssim: N >= 0 and C > 0 required (got N = %d, C = %d)", N, C);
    SVRS_CHECK_ARG(win >= 3 && win % 2 == 1, "ssim: win must be odd and >= 3 (got %d)", win);
    SVRS_CHECK_ARG(win <= H && win <= W, "ssim: win (%d) exceeds the image (%d x %d)", win, H, W);
    SVRS_CHECK_ARG(ssim_smem_bytes(W, win) <= SS_SMEM_MAX,
                   "ssim: W = %d at win = %d needs %lld bytes of shared memory (limit %d: 4 * W * (2 * (%d + win - 1) + %d))",
                   W, win, ssim_smem_bytes(W, win), SS_SMEM_MAX, SS_BAND, 5 * SS_VP);
    return 0;
}

extern "C" int64_t svrs_ssim_workspace_doubles(int N, int C, int H, int W, int win) {
    if (ssim_check(N, C, H, W, win)) return -1;
    return (int64_t)N * C * ((H - win + 1 + SS_BAND - 1) / SS_BAND);
}

extern "C" int svrs_ssim(const float* a, const float* b, int N, int C, int H, int W, int win, float data_range,
                         double* workspace, double* out, void* stream) {
    if (int rc = ssim_check(N, C, H, W, win)) return rc;
    if (N == 0) return 0;
    SVRS_CHECK_ARG(a && b && workspace && out, "ssim: null pointer");
    const int nbands = (H - win + 1 + SS_BAND - 1) / SS_BAND;
    const long long blocks = (long long)N * C * nbands;
    SVRS_CHECK_ARG(blocks < (1LL << 31), "ssim: too many planes (%lld CTAs)", blocks);
    static bool attr_set = false;
    if (!attr_set) {
        cudaError_t e = cudaFuncSetAttribute(ssim_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, SS_SMEM_MAX);
        if (e != cudaSuccess) { set_error("ssim: cudaFuncSetAttribute: %s", cudaGetErrorString(e)); return SVRS_E_CUDA; }
        attr_set = true;
    }
    SsimArgs p;
    p.a = a; p.b = b; p.part = workspace;
    p.H = H; p.W = W; p.win = win; p.nbands = nbands;
    const double np = (double)win * win, R = data_range;
    p.c1 = (0.01 * R) * (0.01 * R);
    p.c2 = (0.03 * R) * (0.03 * R);
    p.cov_norm = np / (np - 1.0);
    SVRS_LAUNCH(ssim_kernel, (unsigned)blocks, SS_THREADS, ssim_smem_bytes(W, win), (cudaStream_t)stream, p);
    int rc = check_launch("ssim_kernel");
    if (rc) return rc;
    SVRS_LAUNCH(ssim_finalize_kernel, (N + 127) / 128, 128, 0, (cudaStream_t)stream, (const double*)workspace, out, N, C, nbands,
                1.0 / ((double)(H - win + 1) * (W - win + 1)));
    return check_launch("ssim_finalize_kernel");
}
