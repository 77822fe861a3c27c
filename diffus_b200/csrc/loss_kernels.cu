// Image losses of the reference's training loops (SURVEY.md section 8 row f3), forward and backward:
//
//   masked MSE + 0.5 * edge L1   notebooks/[DEMO] Train MRI to Impedance MLP.ipynb cell 19 (UltrasoundSynthesisModel.loss,
//                                gradient_loss): mse(a[mask], b[mask]) + 0.5 * l1(|d_x a|[mask[:,1:]], |d_x b|[mask[:,1:]])
//   1 - SSIM                     notebooks/[DEMO] Train MRI to Impedance MLP - GPU.ipynb cell 16: the synthetic image is
//                                min-max normalised, then piq.ssim(synth, real, data_range=1.0).  piq is a third-party
//                                dependency absent from the reference tree (and from this image): the algorithm restated
//                                here is piq 0.8's `ssim` with its defaults (Wang et al. 2004): 11 x 11 Gaussian window,
//                                sigma 1.5, VALID convolution, k1 = 0.01, k2 = 0.03, mean over the map; images below
//                                384 pixels are not down-sampled.
//
// A B-mode image is 256 x 256: the reductions are single-CTA or fixed-order block partials (run-to-run identical).
#include "common.cuh"
#include "launch.h"

namespace diffus {

namespace {

__device__ __forceinline__ double block_sum_d(double v, double* sh) {
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) v += __shfl_xor_sync(FULL, v, d);
    if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = v;
    __syncthreads();
    double r = 0.0;
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) r += sh[w];
    __syncthreads();
    return r;
}
__device__ __forceinline__ float sgn(float v) { return v > 0.f ? 1.f : (v < 0.f ? -1.f : 0.f); }

}  // namespace

// ---------------------------------------------------------------------------------------
// masked MSE + edge
// stats (floats): [0] loss  [1] N1 = count(mask)  [2] N2 = count(mask[:, 1:])
// ---------------------------------------------------------------------------------------
__global__ void __launch_bounds__(1024) masked_mse_edge_fwd_kernel(const float* __restrict__ a, const float* __restrict__ b,
                                                                   const uint8_t* __restrict__ mask, int H, int W, float edge_weight,
                                                                   float* __restrict__ stats) {
    __shared__ double sh[32];
    double s1 = 0.0, s2 = 0.0, n1 = 0.0, n2 = 0.0;
    const int64_t n = (int64_t)H * W;
    for (int64_t t = threadIdx.x; t < n; t += blockDim.x) {
        if (!mask[t]) continue;
        const int j = (int)(t % W);
        const float d = a[t] - b[t];
        s1 += (double)d * d;
        n1 += 1.0;
        if (j >= 1) {
            const float e = fabsf(a[t] - a[t - 1]) - fabsf(b[t] - b[t - 1]);
            s2 += fabs((double)e);
            n2 += 1.0;
        }
    }
    s1 = block_sum_d(s1, sh); s2 = block_sum_d(s2, sh); n1 = block_sum_d(n1, sh); n2 = block_sum_d(n2, sh);
    if (threadIdx.x == 0) {
        stats[0] = (float)(s1 / n1 + (double)edge_weight * (s2 / n2));     // empty masks give NaN, like torch's mean of nothing
        stats[1] = (float)n1;
        stats[2] = (float)n2;
    }
}

__global__ void masked_mse_edge_bwd_kernel(const float* __restrict__ a, const float* __restrict__ b, const uint8_t* __restrict__ mask,
                                           int H, int W, float edge_weight, const float* __restrict__ stats,
                                           const float* __restrict__ grad_loss, float* __restrict__ ga) {
    const int64_t n = (int64_t)H * W;
    const float gl = grad_loss[0], n1 = stats[1], n2 = stats[2];
    for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < n; t += (int64_t)gridDim.x * blockDim.x) {
        const int j = (int)(t % W);
        float g = 0.f;
        if (mask[t]) {
            g = 2.f * (a[t] - b[t]) / n1;
            if (j >= 1) {                      // as the LEFT... the term in which a[t] is the minuend of d_x a
                const float da = a[t] - a[t - 1];
                g += edge_weight / n2 * sgn(fabsf(da) - fabsf(b[t] - b[t - 1])) * sgn(da);
            }
        }
        if (j + 1 < W && mask[t + 1]) {        // the term of the right neighbour, in which a[t] is the subtrahend
            const float da = a[t + 1] - a[t];
            g -= edge_weight / n2 * sgn(fabsf(da) - fabsf(b[t + 1] - b[t])) * sgn(da);
        }
        ga[t] = g * gl;
    }
}

cudaError_t launch_masked_mse_edge_fwd(const float* a, const float* b, const uint8_t* mask, int H, int W, float edge_weight,
                                       float* stats, cudaStream_t st) {
    return launch_kernel(masked_mse_edge_fwd_kernel, 1, 1024, 0, st, a, b, mask, H, W, edge_weight, stats);
}
cudaError_t launch_masked_mse_edge_bwd(const float* a, const float* b, const uint8_t* mask, int H, int W, float edge_weight,
                                       const float* stats, const float* grad_loss, float* ga, cudaStream_t st) {
    const int64_t n = (int64_t)H * W;
    return launch_kernel(masked_mse_edge_bwd_kernel, (unsigned)max((int64_t)1, min((int64_t)148 * 4, (n + 255) / 256)), 256, 0, st, 
        a, b, mask, H, W, edge_weight, stats, grad_loss, ga);
}

// ---------------------------------------------------------------------------------------
// 1 - SSIM
// workspace: header (16 floats): [0] min [1] max [2] ties of min [3] ties of max [4] 1/(max - min + 1e-8) or 1
//            block partials (3 doubles per forward / backward tile)
//            coefficient maps Ga, Gb, Gc (3 x Hout x Wout floats): dS/dE[x], dS/dE[x^2], dS/dE[xy] per window
//            gxn (H x W floats): gradient w.r.t. the normalised image
// ---------------------------------------------------------------------------------------
constexpr int SSIM_TILE = 16;
constexpr int SSIM_MAXK = 33;

struct SsimLayout {
    float* header;
    double* partials;
    float *ga, *gb, *gc, *gxn;
    int Ho, Wo, tiles_fwd, tiles_bwd;
    int64_t bytes;
};
static SsimLayout ssim_layout(void* base, int H, int W, int K) {
    SsimLayout L{};
    L.Ho = H - K + 1;
    L.Wo = W - K + 1;
    L.tiles_fwd = ((L.Ho + SSIM_TILE - 1) / SSIM_TILE) * ((L.Wo + SSIM_TILE - 1) / SSIM_TILE);
    L.tiles_bwd = ((H + SSIM_TILE - 1) / SSIM_TILE) * ((W + SSIM_TILE - 1) / SSIM_TILE);
    int64_t off = 0;
    char* p = (char*)base;
    L.header = (float*)(p + off); off += 256;
    L.partials = (double*)(p + off); off += ((int64_t)3 * max(L.tiles_fwd, L.tiles_bwd) * 8 + 255) / 256 * 256;
    const int64_t map = ((int64_t)L.Ho * L.Wo * 4 + 255) / 256 * 256;
    L.ga = (float*)(p + off); off += map;
    L.gb = (float*)(p + off); off += map;
    L.gc = (float*)(p + off); off += map;
    L.gxn = (float*)(p + off); off += ((int64_t)H * W * 4 + 255) / 256 * 256;
    L.bytes = off;
    return L;
}
int64_t ssim_workspace_bytes(int H, int W, int K) { return ssim_layout(nullptr, H, W, K).bytes; }

__global__ void __launch_bounds__(1024) ssim_minmax_kernel(const float* __restrict__ s, int64_t n, int normalize, float* __restrict__ header) {
    __shared__ float shf[32];
    __shared__ double shd[32];
    if (!normalize) {
        if (threadIdx.x == 0) { header[0] = 0.f; header[1] = 1.f; header[2] = header[3] = 1.f; header[4] = 1.f; }
        return;
    }
    float mn = FLT_MAX, mx = -FLT_MAX;
    for (int64_t i = threadIdx.x; i < n; i += blockDim.x) { mn = fminf(mn, s[i]); mx = fmaxf(mx, s[i]); }
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) { mn = fminf(mn, __shfl_xor_sync(FULL, mn, d)); mx = fmaxf(mx, __shfl_xor_sync(FULL, mx, d)); }
    if ((threadIdx.x & 31) == 0) shf[threadIdx.x >> 5] = mn;
    __syncthreads();
    float r = shf[0];
    for (int w = 1; w < 32; ++w) r = fminf(r, shf[w]);
    __syncthreads();
    mn = r;
    if ((threadIdx.x & 31) == 0) shf[threadIdx.x >> 5] = mx;
    __syncthreads();
    r = shf[0];
    for (int w = 1; w < 32; ++w) r = fmaxf(r, shf[w]);
    __syncthreads();
    mx = r;
    double cmn = 0.0, cmx = 0.0;
    for (int64_t i = threadIdx.x; i < n; i += blockDim.x) { cmn += (s[i] == mn); cmx += (s[i] == mx); }
    cmn = block_sum_d(cmn, shd);
    cmx = block_sum_d(cmx, shd);
    if (threadIdx.x == 0) {
        header[0] = mn; header[1] = mx; header[2] = (float)cmn; header[3] = (float)cmx;
        header[4] = 1.f / (mx - mn + 1e-8f);
    }
}

// 1-D window, normalised: the 2-D window of piq is its outer product
__device__ __forceinline__ void fill_window(float* win, int K, float sigma) {
    if (threadIdx.x == 0) {
        float sum = 0.f;
        for (int i = 0; i < K; ++i) {
            const float c = (float)i - (float)(K - 1) * 0.5f;
            win[i] = expf(-(c * c) / (2.f * sigma * sigma));
            sum += win[i];
        }
        for (int i = 0; i < K; ++i) win[i] /= sum;
    }
}

__global__ void __launch_bounds__(SSIM_TILE * SSIM_TILE) ssim_fwd_kernel(const float* __restrict__ s, const float* __restrict__ y, int H, int W,
                                                                         int K, float sigma, float c1, float c2, SsimLayout L) {
    extern __shared__ float sm[];
    const int IN = SSIM_TILE + K - 1;
    float* xs = sm;                       // IN x IN normalised synthetic tile
    float* ys = xs + IN * IN;
    float* rows = ys + IN * IN;           // 5 x IN x TILE row-filtered quantities
    float* win = rows + 5 * IN * SSIM_TILE;
    __shared__ double shd[32];
    const int tiles_x = (L.Wo + SSIM_TILE - 1) / SSIM_TILE;
    const int ty0 = (blockIdx.x / tiles_x) * SSIM_TILE, tx0 = (blockIdx.x % tiles_x) * SSIM_TILE;
    const float mn = L.header[0], inv = L.header[4];
    fill_window(win, K, sigma);
    for (int t = threadIdx.x; t < IN * IN; t += blockDim.x) {
        const int r = ty0 + t / IN, c = tx0 + t % IN;
        const bool ok = r < H && c < W;
        xs[t] = ok ? (s[(int64_t)r * W + c] - mn) * inv : 0.f;
        ys[t] = ok ? y[(int64_t)r * W + c] : 0.f;
    }
    __syncthreads();
    for (int t = threadIdx.x; t < IN * SSIM_TILE; t += blockDim.x) {
        const int r = t / SSIM_TILE, c = t % SSIM_TILE;
        float ex = 0.f, ey = 0.f, exx = 0.f, eyy = 0.f, exy = 0.f;
        for (int k = 0; k < K; ++k) {
            const float w = win[k], xv = xs[r * IN + c + k], yv = ys[r * IN + c + k];
            ex = fmaf(w, xv, ex); ey = fmaf(w, yv, ey);
            exx = fmaf(w, xv * xv, exx); eyy = fmaf(w, yv * yv, eyy); exy = fmaf(w, xv * yv, exy);
        }
        rows[t] = ex; rows[IN * SSIM_TILE + t] = ey; rows[2 * IN * SSIM_TILE + t] = exx;
        rows[3 * IN * SSIM_TILE + t] = eyy; rows[4 * IN * SSIM_TILE + t] = exy;
    }
    __syncthreads();
    const int r = threadIdx.x / SSIM_TILE, c = threadIdx.x % SSIM_TILE;
    const int orow = ty0 + r, ocol = tx0 + c;
    double contrib = 0.0;
    if (orow < L.Ho && ocol < L.Wo) {
        float ex = 0.f, ey = 0.f, exx = 0.f, eyy = 0.f, exy = 0.f;
        for (int k = 0; k < K; ++k) {
            const float w = win[k];
            const int idx = (r + k) * SSIM_TILE + c;
            ex = fmaf(w, rows[idx], ex); ey = fmaf(w, rows[IN * SSIM_TILE + idx], ey);
            exx = fmaf(w, rows[2 * IN * SSIM_TILE + idx], exx); eyy = fmaf(w, rows[3 * IN * SSIM_TILE + idx], eyy);
            exy = fmaf(w, rows[4 * IN * SSIM_TILE + idx], exy);
        }
        const float A1 = 2.f * ex * ey + c1, A2 = 2.f * (exy - ex * ey) + c2;
        const float B1 = ex * ex + ey * ey + c1, B2 = (exx - ex * ex) + (eyy - ey * ey) + c2;
        const float S = (A1 * A2) / (B1 * B2);
        contrib = (double)S;
        const int64_t o = (int64_t)orow * L.Wo + ocol;
        L.ga[o] = 2.f * ey * (A2 - A1) / (B1 * B2) - S * 2.f * ex * (1.f / B1 - 1.f / B2);
        L.gb[o] = -S / B2;
        L.gc[o] = 2.f * A1 / (B1 * B2);
    }
    const double tot = block_sum_d(contrib, shd);
    if (threadIdx.x == 0) L.partials[blockIdx.x] = tot;
}

__global__ void ssim_loss_final_kernel(SsimLayout L, float* __restrict__ loss) {
    if (threadIdx.x == 0) {
        double t = 0.0;
        for (int b = 0; b < L.tiles_fwd; ++b) t += L.partials[b];
        loss[0] = (float)(1.0 - t / ((double)L.Ho * (double)L.Wo));
    }
}

// gradient w.r.t. the NORMALISED image: the transpose of the VALID window filter (a full correlation) of the three
// coefficient maps, gxn(q) = -(1/N) [F(Ga) + 2 xn(q) F(Gb) + y(q) F(Gc)], plus block partials of sum gxn, sum gxn xn
__global__ void __launch_bounds__(SSIM_TILE * SSIM_TILE) ssim_bwd_kernel(const float* __restrict__ s, const float* __restrict__ y, int H, int W,
                                                                         int K, float sigma, SsimLayout L) {
    extern __shared__ float sm[];
    const int IN = SSIM_TILE + K - 1;
    float* ca = sm;                       // IN x IN tiles of the three coefficient maps (zero outside the map)
    float* cb = ca + IN * IN;
    float* cc = cb + IN * IN;
    float* rows = cc + IN * IN;           // 3 x IN x TILE
    float* win = rows + 3 * IN * SSIM_TILE;
    __shared__ double shd[32];
    const int tiles_x = (W + SSIM_TILE - 1) / SSIM_TILE;
    const int qy0 = (blockIdx.x / tiles_x) * SSIM_TILE, qx0 = (blockIdx.x % tiles_x) * SSIM_TILE;
    fill_window(win, K, sigma);
    // input pixel q receives from windows p = q - k, k = 0..K-1: map rows qy0 - (K-1) .. qy0 + TILE - 1
    for (int t = threadIdx.x; t < IN * IN; t += blockDim.x) {
        const int pr = qy0 - (K - 1) + t / IN, pc = qx0 - (K - 1) + t % IN;
        const bool ok = pr >= 0 && pr < L.Ho && pc >= 0 && pc < L.Wo;
        const int64_t o = (int64_t)pr * L.Wo + pc;
        ca[t] = ok ? L.ga[o] : 0.f;
        cb[t] = ok ? L.gb[o] : 0.f;
        cc[t] = ok ? L.gc[o] : 0.f;
    }
    __syncthreads();
    for (int t = threadIdx.x; t < IN * SSIM_TILE; t += blockDim.x) {
        const int r = t / SSIM_TILE, c = t % SSIM_TILE;
        float fa = 0.f, fb = 0.f, fc = 0.f;
        for (int k = 0; k < K; ++k) {      // window tap k pairs input column q with map column q - k: tile column c + (K-1) - k
            const float w = win[k];
            const int idx = r * IN + c + (K - 1) - k;
            fa = fmaf(w, ca[idx], fa); fb = fmaf(w, cb[idx], fb); fc = fmaf(w, cc[idx], fc);
        }
        rows[t] = fa; rows[IN * SSIM_TILE + t] = fb; rows[2 * IN * SSIM_TILE + t] = fc;
    }
    __syncthreads();
    const int r = threadIdx.x / SSIM_TILE, c = threadIdx.x % SSIM_TILE;
    const int qr = qy0 + r, qc = qx0 + c;
    double sg = 0.0, sgx = 0.0;
    if (qr < H && qc < W) {
        float fa = 0.f, fb = 0.f, fc = 0.f;
        for (int k = 0; k < K; ++k) {
            const float w = win[k];
            const int idx = (r + (K - 1) - k) * SSIM_TILE + c;
            fa = fmaf(w, rows[idx], fa); fb = fmaf(w, rows[IN * SSIM_TILE + idx], fb); fc = fmaf(w, rows[2 * IN * SSIM_TILE + idx], fc);
        }
        const int64_t q = (int64_t)qr * W + qc;
        const float xn = (s[q] - L.header[0]) * L.header[4];
        const float g = -(fa + 2.f * xn * fb + y[q] * fc) / ((float)L.Ho * (float)L.Wo);
        L.gxn[q] = g;
        sg = (double)g;
        sgx = (double)g * (double)xn;
    }
    sg = block_sum_d(sg, shd);
    sgx = block_sum_d(sgx, shd);
    if (threadIdx.x == 0) { L.partials[2 * blockIdx.x] = sg; L.partials[2 * blockIdx.x + 1] = sgx; }
}

// chain through xn = (s - min) / (max - min + 1e-8): the gradients of min() and max() are spread evenly over their ties
__global__ void ssim_bwd_final_kernel(const float* __restrict__ s, int64_t n, int normalize, SsimLayout L,
                                      const float* __restrict__ grad_loss, float* __restrict__ gs) {
    double sg = 0.0, sgx = 0.0;
    if (normalize)
        for (int b = 0; b < L.tiles_bwd; ++b) { sg += L.partials[2 * b]; sgx += L.partials[2 * b + 1]; }
    const float gl = grad_loss[0];
    const float mn = L.header[0], mx = L.header[1], inv = L.header[4];
    const float gmn = normalize ? (float)((-sg + sgx) * (double)inv / (double)L.header[2]) : 0.f;
    const float gmx = normalize ? (float)(-sgx * (double)inv / (double)L.header[3]) : 0.f;
    for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < n; t += (int64_t)gridDim.x * blockDim.x) {
        float g = L.gxn[t] * inv;
        if (normalize) {
            if (s[t] == mn) g += gmn;
            if (s[t] == mx) g += gmx;
        }
        gs[t] = g * gl;
    }
}

cudaError_t launch_ssim_fwd(const float* s, const float* y, int H, int W, int K, float sigma, float k1, float k2, int normalize,
                            float* loss, void* workspace, cudaStream_t st) {
    SsimLayout L = ssim_layout(workspace, H, W, K);
    cudaError_t e = launch_kernel(ssim_minmax_kernel, 1, 1024, 0, st, s, (int64_t)H * W, normalize, L.header);
    if (e != cudaSuccess) return e;
    const int IN = SSIM_TILE + K - 1;
    const size_t smem = (size_t)(2 * IN * IN + 5 * IN * SSIM_TILE + SSIM_MAXK + 3) * sizeof(float);
    e = launch_kernel(ssim_fwd_kernel, L.tiles_fwd, SSIM_TILE * SSIM_TILE, smem, st, s, y, H, W, K, sigma, k1 * k1, k2 * k2, L);
    if (e != cudaSuccess) return e;
    return launch_kernel(ssim_loss_final_kernel, 1, 32, 0, st, L, loss);
}

cudaError_t launch_ssim_bwd(const float* s, const float* y, int H, int W, int K, float sigma, int normalize, const float* grad_loss,
                            float* grad_s, void* workspace, cudaStream_t st) {
    SsimLayout L = ssim_layout(workspace, H, W, K);
    const int IN = SSIM_TILE + K - 1;
    const size_t smem = (size_t)(3 * IN * IN + 3 * IN * SSIM_TILE + SSIM_MAXK + 3) * sizeof(float);
    cudaError_t e = launch_kernel(ssim_bwd_kernel, L.tiles_bwd, SSIM_TILE * SSIM_TILE, smem, st, s, y, H, W, K, sigma, L);
    if (e != cudaSuccess) return e;
    const int64_t n = (int64_t)H * W;
    return launch_kernel(ssim_bwd_final_kernel, (unsigned)max((int64_t)1, min((int64_t)148 * 4, (n + 255) / 256)), 256, 0, st, s, n, normalize, L, grad_loss, grad_s);
}

}  // namespace diffus
