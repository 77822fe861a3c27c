// Small kernels of the training loop around the renderer (SURVEY.md section 8 row f3 / f1 epilogue):
//   - the Adam update of the 1 153 MLP weights (torch.optim.Adam as used by the reference's notebooks and
//     src/impedance.py:26-35), one launch for parameters, both moments and the step counter;
//   - one slice of a volume in / out of the gathered layout (ImpedanceLearner.training_forward's slice mode,
//     notebooks/[DEMO] Train MRI to Impedance MLP - GPU.ipynb cell 16);
//   - rotate_around_apex (src/renderer.py:655-692) as one element-wise launch;
//   - log compression: log1p(|.|) / max (notebooks/[DEMO] Renderer Alternatives.ipynb cell 14, process_rf_to_bmode),
//     on an image (differentiable) and on RF lines behind their Hilbert envelope.
#include "common.cuh"
#include "launch.h"

namespace diffus {

// ---------------------------------------------------------------------------------------
// Adam.  state = [exp_avg (n) | exp_avg_sq (n) | step (1 float)], zero-initialised by the caller.
// One CTA: every thread reads the step before any thread writes it back.
// ---------------------------------------------------------------------------------------
__global__ void __launch_bounds__(1024) adam_step_kernel(float* __restrict__ params, const float* __restrict__ grads,
                                                         float* __restrict__ state, int n, float lr, float beta1, float beta2,
                                                         float eps, float weight_decay, float grad_scale) {
    float* m = state;
    float* v = state + n;
    const float step = state[2 * n] + 1.f;
    __syncthreads();
    // torch: bias_correction = 1 - beta ** step (python floats = double); step_size = lr / bc1; denom = sqrt(v) / sqrt(bc2) + eps
    const double bc1 = 1.0 - pow((double)beta1, (double)step), bc2 = 1.0 - pow((double)beta2, (double)step);
    const float step_size = (float)((double)lr / bc1);
    const float bc2_sqrt = (float)sqrt(bc2);
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
        float p = params[i];
        float g = grads[i] * grad_scale;
        if (weight_decay != 0.f) g = fmaf(weight_decay, p, g);
        float mi = m[i], vi = v[i];
        mi = mi + (g - mi) * (1.f - beta1);                      // exp_avg.lerp_(grad, 1 - beta1)
        vi = fmaf(vi, beta2, (1.f - beta2) * g * g);             // exp_avg_sq.mul_(beta2).addcmul_(grad, grad, 1 - beta2)
        const float denom = sqrtf(vi) / bc2_sqrt + eps;
        params[i] = p - step_size * (mi / denom);                // param.addcdiv_(exp_avg, denom, value=-step_size)
        m[i] = mi;
        v[i] = vi;
    }
    if (threadIdx.x == 0) state[2 * n] = step;
}

cudaError_t launch_adam_step(float* params, const float* grads, float* state, int64_t n, float lr, float beta1, float beta2,
                             float eps, float weight_decay, float grad_scale, cudaStream_t st) {
    return launch_kernel(adam_step_kernel, 1, 1024, 0, st, params, grads, state, (int)n, lr, beta1, beta2, eps, weight_decay, grad_scale);
}

// ---------------------------------------------------------------------------------------
// one slice of a volume: slice[b][c] <-> volume[... index along `axis` ...], LINEAR or BRICK layout
// ---------------------------------------------------------------------------------------
template <int LAYOUT, bool SCATTER>
__global__ void volume_slice_kernel(float* __restrict__ vol, VolumeView v, int axis, int index, float* __restrict__ slice, int nb, int nc) {
    const int64_t n = (int64_t)nb * nc;
    for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < n; t += (int64_t)gridDim.x * blockDim.x) {
        const int b = (int)(t / nc), c = (int)(t - (int64_t)b * nc);
        int i, j, k;
        if (axis == 0) { i = index; j = b; k = c; }
        else if (axis == 1) { i = b; j = index; k = c; }
        else { i = b; j = c; k = index; }
        const uint32_t off = voxel_offset<LAYOUT>(v, i, j, k);
        if (SCATTER) vol[off] = slice[t];
        else slice[t] = vol[off];
    }
}

cudaError_t launch_volume_slice(float* vol, const int32_t dim[3], int layout, int axis, int index, float* slice, bool scatter,
                                cudaStream_t st) {
    VolumeView v{};
    v.data = vol;
    v.D = dim[0]; v.H = dim[1]; v.W = dim[2];
    if (layout == DIFFUS_LAYOUT_BRICK) {
        const uint32_t nbj = (v.H + BRICK_J - 1) / BRICK_J, nbk = (v.W + BRICK_K - 1) / BRICK_K;
        v.sy = nbk * 32;
        v.sx = nbj * nbk * 32;
    } else {
        v.sy = (uint32_t)v.W;
        v.sx = (uint32_t)v.H * (uint32_t)v.W;
    }
    const int nb = axis == 0 ? dim[1] : dim[0], nc = axis == 2 ? dim[1] : dim[2];
    const int64_t n = (int64_t)nb * nc;
    const unsigned grid = (unsigned)max((int64_t)1, min((int64_t)148 * 8, (n + 255) / 256));
    if (layout == DIFFUS_LAYOUT_BRICK) {
        if (scatter) return launch_kernel(volume_slice_kernel<DIFFUS_LAYOUT_BRICK, true>, grid, 256, 0, st, vol, v, axis, index, slice, nb, nc);
        return launch_kernel(volume_slice_kernel<DIFFUS_LAYOUT_BRICK, false>, grid, 256, 0, st, vol, v, axis, index, slice, nb, nc);
    }
    if (scatter) return launch_kernel(volume_slice_kernel<DIFFUS_LAYOUT_LINEAR, true>, grid, 256, 0, st, vol, v, axis, index, slice, nb, nc);
    return launch_kernel(volume_slice_kernel<DIFFUS_LAYOUT_LINEAR, false>, grid, 256, 0, st, vol, v, axis, index, slice, nb, nc);
}

// ---------------------------------------------------------------------------------------
// rotate_around_apex (src/renderer.py:655-692): x_rot = cos (x - shift) - sin z + apex0, z_rot = sin (x - shift) + cos z + apex1
// with torch's one-rounding-per-op arithmetic spelled out
// ---------------------------------------------------------------------------------------
__global__ void rotate_apex_kernel(const float* __restrict__ x, const float* __restrict__ z, int64_t n, float cos_a, float sin_a,
                                   float shift, float apex0, float apex1, float* __restrict__ xr, float* __restrict__ zr) {
    for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < n; t += (int64_t)gridDim.x * blockDim.x) {
        const float xs = __fsub_rn(x[t], shift), zs = z[t];
        xr[t] = __fadd_rn(__fsub_rn(__fmul_rn(cos_a, xs), __fmul_rn(sin_a, zs)), apex0);
        zr[t] = __fadd_rn(__fadd_rn(__fmul_rn(sin_a, xs), __fmul_rn(cos_a, zs)), apex1);
    }
}

cudaError_t launch_rotate_apex(const float* x, const float* z, int64_t n, float cos_a, float sin_a, float shift, float apex0,
                               float apex1, float* xr, float* zr, cudaStream_t st) {
    const unsigned grid = (unsigned)max((int64_t)1, min((int64_t)148 * 8, (n + 255) / 256));
    return launch_kernel(rotate_apex_kernel, grid, 256, 0, st, x, z, n, cos_a, sin_a, shift, apex0, apex1, xr, zr);
}

// ---------------------------------------------------------------------------------------
// log compression of an image: out = log1p(|x|) / max(log1p(|x|)).  One CTA (a B-mode image is 256 x 256).
// Backward with the maximum's gradient spread evenly over its ties (torch's rule for a full-reduction max).
// ---------------------------------------------------------------------------------------
__device__ __forceinline__ float block_max(float v, float* sh) {
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) v = fmaxf(v, __shfl_xor_sync(FULL, v, d));
    if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = v;
    __syncthreads();
    float r = sh[0];
    for (int w = 1; w < (int)(blockDim.x >> 5); ++w) r = fmaxf(r, sh[w]);
    __syncthreads();
    return r;
}
__device__ __forceinline__ double block_sum(double v, double* sh) {
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) v += __shfl_xor_sync(FULL, v, d);
    if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = v;
    __syncthreads();
    double r = 0.0;
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) r += sh[w];
    __syncthreads();
    return r;
}

__global__ void __launch_bounds__(1024) log_compress_fwd_kernel(const float* __restrict__ x, int64_t n, float* __restrict__ out,
                                                                float* __restrict__ max_out) {
    __shared__ float sh[32];
    float m = 0.f;
    for (int64_t i = threadIdx.x; i < n; i += blockDim.x) m = fmaxf(m, log1pf(fabsf(x[i])));
    m = block_max(m, sh);
    for (int64_t i = threadIdx.x; i < n; i += blockDim.x) out[i] = log1pf(fabsf(x[i])) / m;
    if (threadIdx.x == 0 && max_out) max_out[0] = m;
}

__global__ void __launch_bounds__(1024) log_compress_bwd_kernel(const float* __restrict__ x, const float* __restrict__ gout, int64_t n,
                                                                float* __restrict__ gx) {
    __shared__ float sh[32];
    __shared__ double shd[32];
    float m = 0.f;
    for (int64_t i = threadIdx.x; i < n; i += blockDim.x) m = fmaxf(m, log1pf(fabsf(x[i])));
    m = block_max(m, sh);
    double acc = 0.0, cnt = 0.0;
    for (int64_t i = threadIdx.x; i < n; i += blockDim.x) {
        const float L = log1pf(fabsf(x[i]));
        acc += (double)gout[i] * (double)L;
        cnt += (L == m) ? 1.0 : 0.0;
    }
    const double gl = block_sum(acc, shd);                  // sum_i g_i L_i
    const double ties = block_sum(cnt, shd);
    const float gm = (float)(-gl / ((double)m * (double)m) / ties);      // d loss / d max, per tied element
    for (int64_t i = threadIdx.x; i < n; i += blockDim.x) {
        const float xi = x[i], L = log1pf(fabsf(xi));
        const float dL = (xi > 0.f ? 1.f : (xi < 0.f ? -1.f : 0.f)) / (1.f + fabsf(xi));
        gx[i] = (gout[i] / m + (L == m ? gm : 0.f)) * dL;
    }
}

cudaError_t launch_log_compress_fwd(const float* x, int64_t n, float* out, float* max_out, cudaStream_t st) {
    return launch_kernel(log_compress_fwd_kernel, 1, 1024, 0, st, x, n, out, max_out);
}
cudaError_t launch_log_compress_bwd(const float* x, const float* gout, int64_t n, float* gx, cudaStream_t st) {
    return launch_kernel(log_compress_bwd_kernel, 1, 1024, 0, st, x, gout, n, gx);
}

// ---------------------------------------------------------------------------------------
// process_rf_to_bmode: envelope = |analytic signal| per RF line (scipy.signal.hilbert along the samples), log1p, / max.
// The imaginary part of the analytic signal is the circular convolution of the line with g = Im(ifft(h)), h the
// one-sided spectrum weights scipy uses; the host passes g (n_samples floats).  One CTA per line, O(S^2) MACs per line
// out of shared memory (a 128 x 512 frame is 33 M MACs).  The frame maximum is taken with an integer atomicMax on the
// (non-negative) float bits; a second launch divides.
// ---------------------------------------------------------------------------------------
__global__ void rf_envelope_kernel(const float* __restrict__ rf, int S, const float* __restrict__ g, float* __restrict__ out,
                                   unsigned* __restrict__ max_bits) {
    extern __shared__ float sm[];
    float* x = sm;
    float* gk = sm + S;
    const float* row = rf + (int64_t)blockIdx.x * S;
    for (int i = threadIdx.x; i < S; i += blockDim.x) { x[i] = row[i]; gk[i] = g[i]; }
    __syncthreads();
    float local_max = 0.f;
    for (int n = threadIdx.x; n < S; n += blockDim.x) {
        float acc = 0.f;
        int k = n;                                           // g index (n - m) mod S, walking m upwards
        for (int m = 0; m < S; ++m) {
            acc = fmaf(x[m], gk[k], acc);
            k = (k == 0) ? S - 1 : k - 1;
        }
        const float env = sqrtf(fmaf(x[n], x[n], acc * acc));
        const float b = log1pf(env);
        out[(int64_t)blockIdx.x * S + n] = b;
        local_max = fmaxf(local_max, b);
    }
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) local_max = fmaxf(local_max, __shfl_xor_sync(FULL, local_max, d));
    if ((threadIdx.x & 31) == 0) atomicMax(max_bits, __float_as_uint(local_max));
}

__global__ void rf_normalise_kernel(float* __restrict__ out, int64_t n, const unsigned* __restrict__ max_bits) {
    const float m = __uint_as_float(*max_bits);
    for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < n; t += (int64_t)gridDim.x * blockDim.x) out[t] = out[t] / m;
}

// ---------------------------------------------------------------------------------------
// compute_gaussian_pulse's F.conv1d (src/renderer.py:476): every row cross-correlated with one short kernel,
//     out[b][o] = sum_t w[t] in[b][o + t - pad]        (zero outside the row), o = 0 .. n_out - 1.
// The backward w.r.t. the rows is the same kernel with w flipped and pad' = L - 1 - pad.
// ---------------------------------------------------------------------------------------
constexpr int CONV_MAX_TAPS = 128;

__global__ void __launch_bounds__(256) conv1d_rows_kernel(const float* __restrict__ in, int64_t rows, int n_in, const float* __restrict__ w,
                                                          int taps, int pad, int flip, float* __restrict__ out, int n_out) {
    __shared__ float ws[CONV_MAX_TAPS];
    for (int t = threadIdx.x; t < taps; t += blockDim.x) ws[t] = __ldg(w + (flip ? taps - 1 - t : t));
    __syncthreads();
    const int64_t total = rows * n_out;
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
        const int64_t b = e / n_out;
        const int o = (int)(e - b * n_out);
        const float* row = in + b * n_in;
        float acc = 0.f;
        const int lo = max(0, pad - o), hi = min(taps, n_in + pad - o);       // taps whose sample lies inside the row
        for (int t = lo; t < hi; ++t) acc = fmaf(ws[t], __ldg(row + o + t - pad), acc);
        out[e] = acc;
    }
}

cudaError_t launch_conv1d_rows(const float* in, int64_t rows, int n_in, const float* w, int taps, int pad, int flip, float* out,
                               int n_out, cudaStream_t st) {
    const int64_t total = rows * n_out;
    const unsigned grid = (unsigned)max((int64_t)1, min((total + 255) / 256, (int64_t)148 * 8));
    return launch_kernel(conv1d_rows_kernel, grid, 256, 0, st, in, rows, n_in, w, taps, pad, flip, out, n_out);
}

__global__ void zero_word_kernel(unsigned* w) { *w = 0u; }

cudaError_t launch_rf_to_bmode(const float* rf, int64_t n_rays, int S, const float* g, float* out, void* workspace, cudaStream_t st) {
    unsigned* max_bits = (unsigned*)workspace;
    cudaError_t e = launch_kernel(zero_word_kernel, 1, 1, 0, st, max_bits);
    if (e != cudaSuccess) return e;
    const size_t smem = (size_t)2 * S * sizeof(float);
    if (smem > 48 * 1024) {
        e = ensure_smem(rf_envelope_kernel, smem);
        if (e != cudaSuccess) return e;
    }
    e = launch_kernel(rf_envelope_kernel, (unsigned)n_rays, 256, smem, st, rf, S, g, out, max_bits);
    if (e != cudaSuccess) return e;
    const int64_t n = n_rays * S;
    return launch_kernel(rf_normalise_kernel, (unsigned)max((int64_t)1, min((int64_t)148 * 8, (n + 255) / 256)), 256, 0, st, out, n, max_bits);
}

}  // namespace diffus
