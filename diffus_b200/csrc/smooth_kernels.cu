// Isotropic 3-D Gaussian smoothing of a float32 volume: scipy.ndimage.gaussian_filter(v, sigma, mode='nearest',
// truncate=truncate).  The scale space that coarse-to-fine pose recovery (pose_recovery.recover_poses_coarse_to_fine)
// renders from.
//
// Separable, three out-of-place passes, p2 src -> dst, p1 dst -> scratch, p0 scratch -> dst.  Out-of-range taps clamp the
// index to the edge voxel (the renderer's own border rule, grid_sample 'border'): zero padding would put an impedance step
// at every face, which the renderer turns into a strong echo.  Each input element is read from global memory once per CTA
// into a shared-memory tile with its 2r halo; every output sums its taps in one fixed order in fp32, pairing the two taps of
// equal weight (the weights are symmetric) -- no atomics, bit-identical from run to run.
#include "common.cuh"
#include "launch.h"

namespace diffus {

struct BlurTaps {
    float w[BLUR_MAX_RADIUS + 1];     // w[t] = weight of the taps at -t and +t
};

// the weight of the centre tap, then the pairs outwards: acc = w0 x0 + sum_t w_t (x_-t + x_t), in that order
__device__ __forceinline__ float blur_sum(const BlurTaps& taps, int r, const float* x, int stride) {
    float acc = taps.w[0] * x[0];
    for (int t = 1; t <= r; ++t) acc = fmaf(taps.w[t], x[-t * stride] + x[t * stride], acc);
    return acc;
}

// ---------------------------------------------------------------------------------------
// p2 (contiguous) pass: a CTA takes a 256-voxel segment of one row plus its halo; each thread produces two outputs,
// 128 apart, so consecutive lanes read consecutive shared-memory words.
// ---------------------------------------------------------------------------------------
constexpr int P2_THREADS = 128, P2_RUN = 2, P2_SEG = P2_THREADS * P2_RUN;

__global__ void __launch_bounds__(P2_THREADS) blur_p2_kernel(const float* __restrict__ src, float* __restrict__ dst, int64_t rows,
                                                             int W, int r, const __grid_constant__ BlurTaps taps) {
    extern __shared__ float tile[];               // P2_SEG + 2r floats
    const int segs = (W + P2_SEG - 1) / P2_SEG;
    const int64_t ntiles = rows * segs;
    for (int64_t tl = blockIdx.x; tl < ntiles; tl += gridDim.x) {
        const int64_t row = tl / segs;
        const int seg0 = (int)(tl - row * segs) * P2_SEG;
        const float* in = src + row * W;
        __syncthreads();                          // the previous tile's reads are done
        for (int q = threadIdx.x; q < P2_SEG + 2 * r; q += P2_THREADS)
            tile[q] = in[min(max(seg0 + q - r, 0), W - 1)];
        __syncthreads();
#pragma unroll
        for (int k = 0; k < P2_RUN; ++k) {
            const int o = k * P2_THREADS + threadIdx.x;
            if (seg0 + o < W) dst[row * W + seg0 + o] = blur_sum(taps, r, tile + o + r, 1);
        }
    }
}

// ---------------------------------------------------------------------------------------
// Strided pass along an axis of length L with `inner` contiguous elements per step (p1: inner = W, outer = D; p0: inner =
// H W, outer = 1).  Lanes take consecutive inner elements, so every load is a 128-byte row; the 8 warps of a CTA each produce
// a run of SR_RUN consecutive outputs along the axis from a (SR_SEG + 2r) x 32 shared-memory tile.  A warp's lanes all read one
// tile row: no bank conflicts.
// ---------------------------------------------------------------------------------------
constexpr int SR_LANES = 32, SR_WARPS = 8, SR_RUN = 16, SR_SEG = SR_WARPS * SR_RUN;

__global__ void __launch_bounds__(SR_LANES * SR_WARPS) blur_strided_kernel(const float* __restrict__ src, float* __restrict__ dst,
                                                                          int64_t outer, int L, int64_t inner, int r,
                                                                          const __grid_constant__ BlurTaps taps) {
    extern __shared__ float tile[];               // (SR_SEG + 2r) rows x 32
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int64_t cols = (inner + SR_LANES - 1) / SR_LANES;
    const int segs = (L + SR_SEG - 1) / SR_SEG;
    const int64_t ntiles = outer * segs * cols;
    const int rows = SR_SEG + 2 * r;
    for (int64_t tl = blockIdx.x; tl < ntiles; tl += gridDim.x) {
        const int64_t c = tl % cols;
        const int64_t rest = tl / cols;
        const int seg0 = (int)(rest % segs) * SR_SEG;
        const int64_t o = rest / segs;
        const int64_t col = c * SR_LANES + lane;
        const bool live = col < inner;
        const float* in = src + o * L * inner + col;
        __syncthreads();
        for (int q = warp; q < rows; q += SR_WARPS)
            tile[q * SR_LANES + lane] = live ? in[(int64_t)min(max(seg0 + q - r, 0), L - 1) * inner] : 0.f;
        __syncthreads();
        if (!live) continue;
        float* out = dst + o * L * inner + col;
        const int a0 = warp * SR_RUN;
#pragma unroll 4
        for (int k = 0; k < SR_RUN; ++k) {
            const int a = seg0 + a0 + k;
            if (a < L) out[(int64_t)a * inner] = blur_sum(taps, r, tile + (a0 + k + r) * SR_LANES + lane, SR_LANES);
        }
    }
}

// scipy.ndimage._filters._gaussian_kernel1d(sigma, 0, radius): exp(-x^2 / (2 sigma^2)) over x = -r..r, normalised to sum 1,
// in float64, then rounded to float32
static BlurTaps gaussian_taps(double sigma, int r) {
    double phi[BLUR_MAX_RADIUS + 1];
    const double c = -0.5 / (sigma * sigma);
    for (int t = 0; t <= r; ++t) phi[t] = exp(c * (double)(t * t));
    double sum = phi[0];
    for (int t = 1; t <= r; ++t) sum += 2.0 * phi[t];
    BlurTaps taps{};
    for (int t = 0; t <= r; ++t) taps.w[t] = (float)(phi[t] / sum);
    return taps;
}

cudaError_t launch_gaussian_blur(const float* src, const int32_t dim[3], float sigma, int r, float* dst, float* scratch,
                                 cudaStream_t st) {
    const int64_t D = dim[0], H = dim[1], W = dim[2];
    if (r == 0)      // sigma <= 1e-15 (scipy skips the axis) or a single tap of weight 1: an exact copy
        return cudaMemcpyAsync(dst, src, (size_t)(D * H * W) * sizeof(float), cudaMemcpyDeviceToDevice, st);
    const BlurTaps taps = gaussian_taps((double)sigma, r);
    const int64_t max_ctas = (int64_t)148 * 32;
    const int64_t t2 = D * H * ((W + P2_SEG - 1) / P2_SEG);
    blur_p2_kernel<<<(unsigned)min(t2, max_ctas), P2_THREADS, (P2_SEG + 2 * r) * sizeof(float), st>>>(src, dst, D * H, (int)W, r,
                                                                                                         taps);
    const size_t smem = (size_t)(SR_SEG + 2 * r) * SR_LANES * sizeof(float);
    const int64_t t1 = D * ((H + SR_SEG - 1) / SR_SEG) * ((W + SR_LANES - 1) / SR_LANES);
    blur_strided_kernel<<<(unsigned)min(t1, max_ctas), SR_LANES * SR_WARPS, smem, st>>>(dst, scratch, D, (int)H, W, r, taps);
    const int64_t t0 = ((D + SR_SEG - 1) / SR_SEG) * ((H * W + SR_LANES - 1) / SR_LANES);
    blur_strided_kernel<<<(unsigned)min(t0, max_ctas), SR_LANES * SR_WARPS, smem, st>>>(scratch, dst, 1, (int)D, H * W, r, taps);
    return cudaGetLastError();
}

}  // namespace diffus
