// Scan conversion: differentiable_splat (reference src/renderer.py:694-737), SURVEY row f1.
//
//   axes    the two coordinates of largest variance, descending (host syncs in the reference, device here)
//   scatter image[idx1, idx0] = intensity at the rounded, clamped pixel -- NON-accumulating: for duplicate
//           pixels the sample with the highest flat index wins (what the reference's sequential CPU
//           index_put_ does); done with one 64-bit atomicMax on (sample index, value bits)
//   blur    both the image and the hit mask with the normalised (int(6 sigma)|1)^2 Gaussian, zero padded
//   out     blurred_image / (blurred_mask + 1e-8), returned transposed (W, H)
#include "common.cuh"
#include "launch.h"

namespace diffus {

constexpr int SPLAT_MAX_K = 63;

struct SplatStats {       // workspace header
    double sum[3], sumsq[3];
    int axis0, axis1;
};

__global__ void splat_stats_kernel(const float* __restrict__ c0, const float* __restrict__ c1, const float* __restrict__ c2,
                                   int64_t n, SplatStats* st) {
    double s[3] = {0, 0, 0}, q[3] = {0, 0, 0};
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        double a = c0[i], b = c1[i], c = c2[i];
        s[0] += a; q[0] += a * a; s[1] += b; q[1] += b * b; s[2] += c; q[2] += c * c;
    }
#pragma unroll
    for (int k = 0; k < 3; ++k) {
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) {
            s[k] += __shfl_xor_sync(FULL, s[k], d);
            q[k] += __shfl_xor_sync(FULL, q[k], d);
        }
        if ((threadIdx.x & 31) == 0) {
            atomicAdd(&st->sum[k], s[k]);
            atomicAdd(&st->sumsq[k], q[k]);
        }
    }
}

__global__ void splat_axes_kernel(SplatStats* st, int64_t n) {
    double var[3];
    for (int k = 0; k < 3; ++k) {
        double mean = st->sum[k] / (double)n;
        var[k] = (st->sumsq[k] - (double)n * mean * mean) / (double)(n > 1 ? n - 1 : 1);
    }
    // sorted(range(3), key=-variance)[:2]: stable, so ties keep the lower axis first
    int order[3] = {0, 1, 2};
    for (int i = 1; i < 3; ++i)
        for (int j = i; j > 0 && var[order[j]] > var[order[j - 1]]; --j) { int t = order[j]; order[j] = order[j - 1]; order[j - 1] = t; }
    st->axis0 = order[0];
    st->axis1 = order[1];
}

__device__ __forceinline__ int splat_pixel(float c, int n) { return min(max(__float2int_rn(c), 0), n - 1); }

__global__ void splat_scatter_kernel(const float* __restrict__ c0, const float* __restrict__ c1, const float* __restrict__ c2,
                                     const float* __restrict__ val, int64_t n, int H, int W, const SplatStats* st,
                                     unsigned long long* __restrict__ keys) {
    const float* cs[3] = {c0, c1, c2};
    const float* ca = cs[st->axis0];
    const float* cb = cs[st->axis1];
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        int px = splat_pixel(ca[i], W), py = splat_pixel(cb[i], H);
        unsigned long long key = ((unsigned long long)(i + 1) << 32) | (unsigned long long)__float_as_uint(val[i]);
        atomicMax(keys + (int64_t)py * W + px, key);
    }
}

__device__ __forceinline__ void splat_kernel1d(float* k1, int K, float sigma) {
    // kernel_1d = exp(-0.5 (t / sigma)^2), t = -K/2..K/2, normalised by its sum (float32, like the reference)
    if (threadIdx.x < K) {
        float t = (float)((int)threadIdx.x - K / 2);
        float q = t / sigma;
        k1[threadIdx.x] = expf(-0.5f * q * q);
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        float s = 0.f;
        for (int i = 0; i < K; ++i) s += k1[i];
        for (int i = 0; i < K; ++i) k1[i] = k1[i] / s;
    }
    __syncthreads();
}

// MODE 0: out (W,H) = blur(img) / (blur(mask) + 1e-8)
// MODE 1: g2 (H,W)  = grad_out^T / (blur(mask) + 1e-8)                (backward, step 1)
// MODE 2: gimg (H,W) = blur(g2)                                       (backward, step 2)
template <int MODE>
__global__ void splat_blur_kernel(const unsigned long long* __restrict__ keys, const float* __restrict__ in, int H, int W,
                                  int K, float sigma, float* __restrict__ out) {
    __shared__ float k1[SPLAT_MAX_K + 1];
    splat_kernel1d(k1, K, sigma);
    const int half = K / 2;
    for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < (int64_t)H * W; t += (int64_t)gridDim.x * blockDim.x) {
        int r = (int)(t / W), c = (int)(t - (int64_t)r * W);
        float num = 0.f, den = 0.f;
        for (int dy = 0; dy < K; ++dy) {
            int rr = r + dy - half;
            if (rr < 0 || rr >= H) continue;
            for (int dx = 0; dx < K; ++dx) {
                int cc = c + dx - half;
                if (cc < 0 || cc >= W) continue;
                float w = k1[dy] * k1[dx];
                if (MODE == 2) {
                    num += w * in[(int64_t)rr * W + cc];
                } else {
                    unsigned long long key = keys[(int64_t)rr * W + cc];
                    if (key) {
                        den += w;
                        if (MODE == 0) num += w * __uint_as_float((unsigned)(key & 0xffffffffu));
                    }
                }
            }
        }
        if (MODE == 0) out[(int64_t)c * H + r] = num / (den + 1e-8f);
        if (MODE == 1) out[t] = in[(int64_t)c * H + r] / (den + 1e-8f);
        if (MODE == 2) out[t] = num;
    }
}

// every sample -- winners and overwritten duplicates alike -- receives its pixel's gradient (index_put_ backward)
__global__ void splat_gather_grad_kernel(const float* __restrict__ c0, const float* __restrict__ c1, const float* __restrict__ c2,
                                         int64_t n, int H, int W, const SplatStats* st, const float* __restrict__ gimg,
                                         float* __restrict__ gval) {
    const float* cs[3] = {c0, c1, c2};
    const float* ca = cs[st->axis0];
    const float* cb = cs[st->axis1];
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
        gval[i] = gimg[(int64_t)splat_pixel(cb[i], H) * W + splat_pixel(ca[i], W)];
}

int64_t splat_workspace_bytes(int H, int W) {
    return 256 + (int64_t)H * W * 8 + 2 * (int64_t)H * W * 4;
}

static unsigned grid_for(int64_t n) { return (unsigned)max((int64_t)1, min((int64_t)148 * 8, (n + 255) / 256)); }

static cudaError_t splat_prepare(const float* c0, const float* c1, const float* c2, const float* val, int64_t n, int H, int W,
                                 void* ws, cudaStream_t st) {
    SplatStats* stats = (SplatStats*)ws;
    unsigned long long* keys = (unsigned long long*)((char*)ws + 256);
    cudaError_t e = cudaMemsetAsync(ws, 0, 256 + (size_t)H * W * 8, st);
    if (e != cudaSuccess) return e;
    e = launch_kernel(splat_stats_kernel, grid_for(n), 256, 0, st, c0, c1, c2, n, stats);
    if (e != cudaSuccess) return e;
    e = launch_kernel(splat_axes_kernel, 1, 1, 0, st, stats, n);
    if (e != cudaSuccess) return e;
    return launch_kernel(splat_scatter_kernel, grid_for(n), 256, 0, st, c0, c1, c2, val, n, H, W, stats, keys);
}

cudaError_t launch_splat_fwd(const float* c0, const float* c1, const float* c2, const float* val, int64_t n, int H, int W,
                             float sigma, float* out, void* ws, cudaStream_t st) {
    int K = (int)(6.f * sigma) | 1;
    if (K > SPLAT_MAX_K) return cudaErrorInvalidValue;
    cudaError_t e = splat_prepare(c0, c1, c2, val, n, H, W, ws, st);
    if (e != cudaSuccess) return e;
    const unsigned long long* keys = (const unsigned long long*)((char*)ws + 256);
    return launch_kernel(splat_blur_kernel<0>, grid_for((int64_t)H * W), 256, 0, st, keys, nullptr, H, W, K, sigma, out);
}

cudaError_t launch_splat_bwd(const float* c0, const float* c1, const float* c2, const float* val, int64_t n, int H, int W,
                             float sigma, const float* grad_out, float* grad_val, void* ws, cudaStream_t st) {
    int K = (int)(6.f * sigma) | 1;
    if (K > SPLAT_MAX_K) return cudaErrorInvalidValue;
    cudaError_t e = splat_prepare(c0, c1, c2, val, n, H, W, ws, st);
    if (e != cudaSuccess) return e;
    const SplatStats* stats = (const SplatStats*)ws;
    const unsigned long long* keys = (const unsigned long long*)((char*)ws + 256);
    float* g2 = (float*)((char*)ws + 256 + (size_t)H * W * 8);
    float* gimg = g2 + (size_t)H * W;
    e = launch_kernel(splat_blur_kernel<1>, grid_for((int64_t)H * W), 256, 0, st, keys, grad_out, H, W, K, sigma, g2);
    if (e != cudaSuccess) return e;
    e = launch_kernel(splat_blur_kernel<2>, grid_for((int64_t)H * W), 256, 0, st, keys, g2, H, W, K, sigma, gimg);
    if (e != cudaSuccess) return e;
    return launch_kernel(splat_gather_grad_kernel, grid_for(n), 256, 0, st, c0, c1, c2, n, H, W, stats, gimg, grad_val);
}

}  // namespace diffus
