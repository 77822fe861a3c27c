// MRI preprocessing in front of the impedance MLP (reference src/utils.py:12-39, used by
// ImpedanceEstimator.compute_impedance_volume, src/impedance.py:46-54), SURVEY row f4:
//   create_brain_mask : volume > threshold, then `iterations` binary dilations and `iterations` binary
//                       erosions with scipy's default 6-neighbour cross and border value 0
//   zscore_normalize  : (volume - mean) / (std + 1e-8) with mean / unbiased std over the masked voxels
#include "common.cuh"
#include "launch.h"

namespace diffus {

__global__ void threshold_kernel(const float* __restrict__ v, int64_t n, float thr, uint8_t* __restrict__ m) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) m[i] = v[i] > thr;
}

template <bool DILATE>
__global__ void morph_kernel(const uint8_t* __restrict__ in, uint8_t* __restrict__ out, int D, int H, int W) {
    const int64_t n = (int64_t)D * H * W;
    for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < n; t += (int64_t)gridDim.x * blockDim.x) {
        int k = (int)(t % W), j = (int)((t / W) % H), i = (int)(t / ((int64_t)W * H));
        // neighbours outside the volume count as 0 (scipy border_value=0): they never set a voxel when dilating
        // and always clear it when eroding
        uint8_t c = in[t];
        uint8_t xm = i > 0 ? in[t - (int64_t)H * W] : 0, xp = i < D - 1 ? in[t + (int64_t)H * W] : 0;
        uint8_t ym = j > 0 ? in[t - W] : 0, yp = j < H - 1 ? in[t + W] : 0;
        uint8_t zm = k > 0 ? in[t - 1] : 0, zp = k < W - 1 ? in[t + 1] : 0;
        out[t] = DILATE ? (c | xm | xp | ym | yp | zm | zp) : (c & xm & xp & ym & yp & zm & zp);
    }
}

struct ZStats {
    double sum, sumsq;
    unsigned long long count;
};

__global__ void masked_stats_kernel(const float* __restrict__ v, const uint8_t* __restrict__ m, int64_t n, ZStats* st) {
    double s = 0, q = 0;
    unsigned long long c = 0;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
        if (m[i]) { double x = v[i]; s += x; q += x * x; ++c; }
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) {
        s += __shfl_xor_sync(FULL, s, d);
        q += __shfl_xor_sync(FULL, q, d);
        c += __shfl_xor_sync(FULL, c, d);
    }
    if ((threadIdx.x & 31) == 0 && c) {
        atomicAdd(&st->sum, s);
        atomicAdd(&st->sumsq, q);
        atomicAdd(&st->count, c);
    }
}

__global__ void zscore_kernel(const float* __restrict__ v, int64_t n, const ZStats* st, float* __restrict__ out) {
    const double cnt = (double)st->count;
    const double mean = st->sum / cnt;
    const double var = (st->sumsq - cnt * mean * mean) / (cnt - 1.0);      // unbiased, like torch.std
    // Rounding can take the one-pass variance just below 0: clamp it, but let a NaN through (one masked voxel gives 0 / 0,
    // torch's std of a single value).  The mean is subtracted in double: rounded to float32 it would be off by up to
    // ulp(mean) / 2, 1e-4 of the std when mean / std is 1e4 (a bright, low-contrast MRI).
    const double scale = 1.0 / (sqrt(var < 0.0 ? 0.0 : var) + 1e-8);
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
        out[i] = (float)(((double)v[i] - mean) * scale);
}

static unsigned grid_for(int64_t n) { return (unsigned)max((int64_t)1, min((int64_t)148 * 16, (n + 255) / 256)); }

cudaError_t launch_brain_mask(const float* volume, const int32_t dim[3], float threshold, int iterations, uint8_t* mask,
                              uint8_t* scratch, cudaStream_t st) {
    const int64_t n = (int64_t)dim[0] * dim[1] * dim[2];
    uint8_t* a = mask;
    uint8_t* b = scratch;
    threshold_kernel<<<grid_for(n), 256, 0, st>>>(volume, n, threshold, a);
    for (int it = 0; it < 2 * iterations; ++it) {
        if (it < iterations) morph_kernel<true><<<grid_for(n), 256, 0, st>>>(a, b, dim[0], dim[1], dim[2]);
        else morph_kernel<false><<<grid_for(n), 256, 0, st>>>(a, b, dim[0], dim[1], dim[2]);
        uint8_t* t = a; a = b; b = t;
    }
    // an even number of passes ends in `mask`
    return cudaGetLastError();
}

cudaError_t launch_masked_zscore(const float* volume, const uint8_t* mask, int64_t n, float* out, void* ws, cudaStream_t st) {
    cudaError_t e = cudaMemsetAsync(ws, 0, sizeof(ZStats), st);
    if (e != cudaSuccess) return e;
    masked_stats_kernel<<<grid_for(n), 256, 0, st>>>(volume, mask, n, (ZStats*)ws);
    zscore_kernel<<<grid_for(n), 256, 0, st>>>(volume, n, (const ZStats*)ws, out);
    return cudaGetLastError();
}

}  // namespace diffus
