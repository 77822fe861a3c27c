// Small kernels around the march: start>0 median, index/value outputs, reductions, fans, bricks.
#include "common.cuh"
#include "launch.h"

namespace diffus {

// ---------------------------------------------------------------------------------------
// start > 0: the first kept reflection coefficient of every ray of a pose is replaced by
// the LOWER median over the pose's rays (torch.median), reference src/renderer.py:241-244.
// One CTA per pose.  The median is found by a 4-pass radix select over the rays' coefficients
// held in shared memory (O(R) per pass; the first version ranked by counting, O(R^2)).
// Besides the median the kernel records how many rays TIE with it: torch's backward of
// `median()` spreads the gradient evenly over the tied elements (evenly_distribute_backward),
// and ties are the common case -- a near field outside the volume clamps to the border and
// gives r = 0 exactly on most rays.
// ---------------------------------------------------------------------------------------
__device__ __forceinline__ float first_reflection(float z0, float z1) { return (z1 - z0) / (z0 + z1); }

// monotone map float -> uint32 (total order; -0 sorts below +0, which only decides which zero is returned)
__device__ __forceinline__ uint32_t radix_key(float v) {
    uint32_t b = __float_as_uint(v);
    return b ^ ((b >> 31) ? 0xffffffffu : 0x80000000u);
}

template <int SAMPLER, int LAYOUT, bool POSE64>
__global__ void first_refl_median_kernel(const RenderParams p, float* __restrict__ median, int32_t* __restrict__ tie_count) {
    extern __shared__ float vals[];
    __shared__ unsigned hist[256];
    __shared__ unsigned sel_prefix, sel_rank, any_nan, ties;
    const int64_t pose = blockIdx.x;
    const int R = (int)p.n_rays;
    if (threadIdx.x == 0) { sel_prefix = 0u; sel_rank = (unsigned)((R - 1) / 2); any_nan = 0u; ties = 0u; }
    __syncthreads();
    for (int ray = threadIdx.x; ray < R; ray += blockDim.x) {
        RaySetup<POSE64> rs;
        rs.load(p.sources, p.directions, pose, ray, p.src_pose_stride, p.src_ray_stride, p.dir_pose_stride, p.product_f32);
        float g[3];
        int k = p.start;
        float z0 = sample_volume<SAMPLER, LAYOUT, false>(p.vol, rs.coord(0, k), rs.coord(1, k), rs.coord(2, k), g);
        float z1 = sample_volume<SAMPLER, LAYOUT, false>(p.vol, rs.coord(0, k + 1), rs.coord(1, k + 1), rs.coord(2, k + 1), g);
        float v = first_reflection(z0, z1);
        vals[ray] = v;
        if (v != v) any_nan = 1u;             // torch.median propagates NaN
    }
    __syncthreads();
    if (any_nan) {
        if (threadIdx.x == 0) { median[pose] = __int_as_float(0x7fc00000); tie_count[pose] = 0; }
        return;
    }
    uint32_t mask = 0u;
    for (int pass = 3; pass >= 0; --pass) {
        for (int b = threadIdx.x; b < 256; b += blockDim.x) hist[b] = 0u;
        __syncthreads();
        const uint32_t prefix = sel_prefix;
        for (int i = threadIdx.x; i < R; i += blockDim.x) {
            uint32_t key = radix_key(vals[i]);
            if ((key & mask) == prefix) atomicAdd(&hist[(key >> (8 * pass)) & 255u], 1u);
        }
        __syncthreads();
        if (threadIdx.x == 0) {               // 256 bins: a serial walk is shorter than a scan's barriers
            unsigned rank = sel_rank, d = 0;
            while (hist[d] <= rank) { rank -= hist[d]; ++d; }
            sel_rank = rank;
            sel_prefix = prefix | (d << (8 * pass));
        }
        mask |= 0xffu << (8 * pass);
        __syncthreads();
    }
    const uint32_t key = sel_prefix;
    const uint32_t bits = (key >> 31) ? (key ^ 0x80000000u) : ~key;
    const float med = __uint_as_float(bits);
    unsigned mine = 0;
    for (int i = threadIdx.x; i < R; i += blockDim.x) mine += (vals[i] == med);
    if (mine) atomicAdd(&ties, mine);
    __syncthreads();
    if (threadIdx.x == 0) { median[pose] = med; tie_count[pose] = (int32_t)ties; }
}

cudaError_t launch_first_refl_median(const RenderParams& p, int sampler, int layout, int pose64, float* median,
                                     int32_t* tie_count, cudaStream_t st) {
    int threads = (int)min((int64_t)256, ((p.n_rays + 31) / 32) * 32);
    size_t smem = (size_t)p.n_rays * sizeof(float);
    DIFFUS_DISPATCH(auto k = first_refl_median_kernel<S_, L_, P64_>;
                    if (smem > 40 * 1024) { cudaError_t e = ensure_smem(k, smem); if (e != cudaSuccess) return e; }
                    return launch_kernel(k, (unsigned)p.n_poses, threads, smem, st, p, median, tie_count))
    return cudaErrorInvalidValue;
}

// Gradient of the median replacement: the summed d loss / d r_1 of a pose flows back through
// `median()` -- evenly onto every ray whose own first coefficient equals the median (one ray when
// there is no tie) -- and from there into the two impedances of that ray's first interface.
// One warp per pose, each lane its own rays; runs after the main backward kernel and before the ray reduction.
template <int SAMPLER, int LAYOUT, bool POSE64, bool POSE_GRAD, bool VOL_GRAD>
__global__ void median_backward_kernel(const RenderParams p, const int32_t* __restrict__ tie_count) {
    const int64_t pose = blockIdx.x;
    const int lane = threadIdx.x;
    float acc = 0.f;
    for (int64_t ray = lane; ray < p.n_rays; ray += 32) acc += p.first_rbar[pose * p.n_rays + ray];
    acc = warp_sum(acc);
    const int ties = tie_count[pose];
    if (ties <= 0) return;                   // NaN median: no element equals it, nothing flows
    const float med = p.median[pose];
    acc /= (float)ties;
    const int k = p.start;
    for (int64_t m = lane; m < p.n_rays; m += 32) {
        const int64_t ray = pose * p.n_rays + m;
        RaySetup<POSE64> rs;
        rs.load(p.sources, p.directions, pose, m, p.src_pose_stride, p.src_ray_stride, p.dir_pose_stride, p.product_f32);
        float g0[3], g1[3];
        float z0 = sample_volume<SAMPLER, LAYOUT, POSE_GRAD>(p.vol, rs.coord(0, k), rs.coord(1, k), rs.coord(2, k), g0);
        float z1 = sample_volume<SAMPLER, LAYOUT, POSE_GRAD>(p.vol, rs.coord(0, k + 1), rs.coord(1, k + 1), rs.coord(2, k + 1), g1);
        if (!(first_reflection(z0, z1) == med)) continue;
        float sum = z0 + z1;
        float zb0 = -acc * 2.f * z1 / (sum * sum), zb1 = acc * 2.f * z0 / (sum * sum);
        if (!(zb0 == zb0)) zb0 = 0.f;
        if (!(zb1 == zb1)) zb1 = 0.f;
        if (POSE_GRAD) {
#pragma unroll
            for (int a = 0; a < 3; ++a) {
                p.grad_src_partial[ray * 3 + a] += zb0 * g0[a] + zb1 * g1[a];
                p.grad_dir[ray * 3 + a] += (float)k * zb0 * g0[a] + (float)(k + 1) * zb1 * g1[a];
            }
        }
        if (VOL_GRAD) {
            for (int which = 0; which < 2; ++which) {
                int kk = k + which;
                float zb = which ? zb1 : zb0;
                float p0 = rs.coord(0, kk), p1 = rs.coord(1, kk), p2 = rs.coord(2, kk);
                if (SAMPLER == DIFFUS_SAMPLER_NEAREST) {
                    int i = nearest_index(p0, p.vol.D), j = nearest_index(p1, p.vol.H), l = nearest_index(p2, p.vol.W);
                    atomicAdd(p.grad_volume + grad_offset<LAYOUT>(p.vol, i, j, l), zb);
                } else {
                    TriCell c;
                    tri_axis(p0, p.vol.D, c.i0[0], c.i1[0], c.f[0]);
                    tri_axis(p1, p.vol.H, c.i0[1], c.i1[1], c.f[1]);
                    tri_axis(p2, p.vol.W, c.i0[2], c.i1[2], c.f[2]);
                    uint32_t off[8];
                    tri_offsets<GradLayout<LAYOUT>::value>(p.vol, c, off);
                    for (int q = 0; q < 8; ++q) {
                        float w = ((q & 4) ? c.f[0] : 1.f - c.f[0]) * ((q & 2) ? c.f[1] : 1.f - c.f[1]) * ((q & 1) ? c.f[2] : 1.f - c.f[2]);
                        if (w != 0.f) atomicAdd(p.grad_volume + off[q], w * zb);
                    }
                }
            }
        }
    }
}

cudaError_t launch_median_backward(const RenderParams& p, int sampler, int layout, int pose64,
                                   const int32_t* tie_count, bool pose_grad, bool vol_grad, cudaStream_t st) {
    if (sampler == DIFFUS_SAMPLER_NEAREST) pose_grad = false;
    if (!pose_grad && !vol_grad) return cudaSuccess;      // loss / frame only: no gradient flows through the median
#define DIFFUS_MB(PG, VG) launch_kernel(median_backward_kernel<S_, L_, P64_, PG, VG>, (unsigned)p.n_poses, 32, 0, st, p, tie_count)
    DIFFUS_DISPATCH(if (pose_grad && vol_grad) return DIFFUS_MB(true, true); if (pose_grad) return DIFFUS_MB(true, false);
                    return DIFFUS_MB(false, true))
#undef DIFFUS_MB
    return cudaErrorInvalidValue;
}

// ---------------------------------------------------------------------------------------
// x, y, z index outputs (src/renderer.py:754-756) and raw sampled values (trace_ray)
// ---------------------------------------------------------------------------------------
template <bool POSE64>
__global__ void ray_indices_kernel(const RenderParams p, int64_t* __restrict__ x, int64_t* __restrict__ y, int64_t* __restrict__ z) {
    const int64_t n = p.total_rays * p.Sout;
    for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < n; t += (int64_t)gridDim.x * blockDim.x) {
        int64_t ray = t / p.Sout;
        int c = (int)(t - ray * p.Sout);
        int64_t pose = ray / p.n_rays;
        RaySetup<POSE64> rs;
        rs.load(p.sources, p.directions, pose, ray - pose * p.n_rays, p.src_pose_stride, p.src_ray_stride, p.dir_pose_stride, p.product_f32);
        int k = p.start + c;
        x[t] = nearest_index(rs.coord(0, k), p.vol.D);
        y[t] = nearest_index(rs.coord(1, k), p.vol.H);
        z[t] = nearest_index(rs.coord(2, k), p.vol.W);
    }
}

cudaError_t launch_ray_indices(const RenderParams& p, int pose64, int64_t* x, int64_t* y, int64_t* z, cudaStream_t st) {
    int64_t n = p.total_rays * p.Sout;
    unsigned grid = (unsigned)min((int64_t)148 * 16, (n + 255) / 256);
    if (pose64) return launch_kernel(ray_indices_kernel<true>, grid, 256, 0, st, p, x, y, z);
    return launch_kernel(ray_indices_kernel<false>, grid, 256, 0, st, p, x, y, z);
}

template <int SAMPLER, int LAYOUT, bool POSE64>
__global__ void trace_values_kernel(const RenderParams p, float* __restrict__ out) {
    const int64_t n = p.total_rays * p.S;
    for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < n; t += (int64_t)gridDim.x * blockDim.x) {
        int64_t ray = t / p.S;
        int k = (int)(t - ray * p.S);
        int64_t pose = ray / p.n_rays;
        RaySetup<POSE64> rs;
        rs.load(p.sources, p.directions, pose, ray - pose * p.n_rays, p.src_pose_stride, p.src_ray_stride, p.dir_pose_stride, p.product_f32);
        float g[3];
        out[t] = sample_volume<SAMPLER, LAYOUT, false>(p.vol, rs.coord(0, k), rs.coord(1, k), rs.coord(2, k), g);
    }
}

cudaError_t launch_trace_values(const RenderParams& p, int sampler, int layout, int pose64, float* out, cudaStream_t st) {
    int64_t n = p.total_rays * p.S;
    unsigned grid = (unsigned)min((int64_t)148 * 16, (n + 255) / 256);
    DIFFUS_DISPATCH(return launch_kernel(trace_values_kernel<S_, L_, P64_>, grid, 256, 0, st, p, out))
    return cudaErrorInvalidValue;
}

// custom_nearest_sampler on explicit points (reference src/renderer.py:741-819): points (n,3) in voxel
// coordinates -> clamped nearest-voxel indices and the sampled values (nearest or trilinear).
template <int SAMPLER, int LAYOUT>
__global__ void sample_points_kernel(const VolumeView vol, const float* __restrict__ pts, int64_t n, float* __restrict__ val,
                                     int64_t* __restrict__ x, int64_t* __restrict__ y, int64_t* __restrict__ z) {
    for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < n; t += (int64_t)gridDim.x * blockDim.x) {
        float p0 = pts[t * 3], p1 = pts[t * 3 + 1], p2 = pts[t * 3 + 2];
        if (x) {
            x[t] = nearest_index(p0, vol.D);
            y[t] = nearest_index(p1, vol.H);
            z[t] = nearest_index(p2, vol.W);
        }
        float g[3];
        val[t] = sample_volume<SAMPLER, LAYOUT, false>(vol, p0, p1, p2, g);
    }
}

cudaError_t launch_sample_points(const RenderParams& p, int sampler, int layout, const float* pts, int64_t n, float* val,
                                 int64_t* x, int64_t* y, int64_t* z, cudaStream_t st) {
    unsigned grid = (unsigned)max((int64_t)1, min((int64_t)148 * 16, (n + 255) / 256));
    const int pose64 = 0;
    DIFFUS_DISPATCH((void)P64_; return launch_kernel(sample_points_kernel<S_, L_>, grid, 256, 0, st, p.vol, pts, n, val, x, y, z))
    return cudaErrorInvalidValue;
}

// Backward of trace_values (what autograd does through the reference's sampler): the gradient of every
// sampled impedance is scattered into the volume (same layout as the gathers) and, for the trilinear
// sampler, contracted with the spatial gradient into per-ray pose partials.  One warp per ray.
template <int SAMPLER, int LAYOUT, bool POSE64, bool POSE_GRAD, bool VOL_GRAD>
__global__ void trace_values_bwd_kernel(const RenderParams p, const float* __restrict__ gval) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int64_t ray = (int64_t)blockIdx.x * (blockDim.x >> 5) + warp;
    if (ray >= p.total_rays) return;
    const int64_t pose = ray / p.n_rays;
    RaySetup<POSE64> rs;
    rs.load(p.sources, p.directions, pose, ray - pose * p.n_rays, p.src_pose_stride, p.src_ray_stride, p.dir_pose_stride, p.product_f32);
    float acc_s[3] = {0.f, 0.f, 0.f}, acc_d[3] = {0.f, 0.f, 0.f};
    for (int k = lane; k < p.S; k += 32) {
        float g = __ldg(gval + ray * (int64_t)p.S + k);
        float p0 = rs.coord(0, k), p1 = rs.coord(1, k), p2 = rs.coord(2, k);
        if (SAMPLER == DIFFUS_SAMPLER_NEAREST) {
            if (VOL_GRAD && g != 0.f) {
                int i = nearest_index(p0, p.vol.D), j = nearest_index(p1, p.vol.H), l = nearest_index(p2, p.vol.W);
                atomicAdd(p.grad_volume + grad_offset<LAYOUT>(p.vol, i, j, l), g);
            }
        } else {
            TriCell c;
            tri_axis(p0, p.vol.D, c.i0[0], c.i1[0], c.f[0]);
            tri_axis(p1, p.vol.H, c.i0[1], c.i1[1], c.f[1]);
            tri_axis(p2, p.vol.W, c.i0[2], c.i1[2], c.f[2]);
            uint32_t off[8];
            tri_offsets<GradLayout<LAYOUT>::value>(p.vol, c, off);
            if (POSE_GRAD) {
                float dzv[3];
                sample_volume<SAMPLER, LAYOUT, true>(p.vol, p0, p1, p2, dzv);
#pragma unroll
                for (int a = 0; a < 3; ++a) { acc_s[a] += g * dzv[a]; acc_d[a] += (float)k * g * dzv[a]; }
            }
            if (VOL_GRAD && g != 0.f) {
#pragma unroll
                for (int q = 0; q < 8; ++q) {
                    float w = ((q & 4) ? c.f[0] : 1.f - c.f[0]) * ((q & 2) ? c.f[1] : 1.f - c.f[1]) * ((q & 1) ? c.f[2] : 1.f - c.f[2]);
                    if (w != 0.f) atomicAdd(p.grad_volume + off[q], w * g);
                }
            }
        }
    }
    if (POSE_GRAD) {
#pragma unroll
        for (int a = 0; a < 3; ++a) {
            float ss = warp_sum(acc_s[a]), dd = warp_sum(acc_d[a]);
            if (lane == 0) { p.grad_src_partial[ray * 3 + a] = ss; p.grad_dir[ray * 3 + a] = dd; }
        }
    }
}

cudaError_t launch_trace_values_bwd(const RenderParams& p, int sampler, int layout, int pose64, const float* gval,
                                    bool pose_grad, bool vol_grad, cudaStream_t st) {
    if (sampler == DIFFUS_SAMPLER_NEAREST) pose_grad = false;
    if (!pose_grad && !vol_grad) return cudaSuccess;      // nothing requested: nothing to write
    unsigned grid = (unsigned)((p.total_rays + 3) / 4);
#define DIFFUS_TB(PG, VG) launch_kernel(trace_values_bwd_kernel<S_, L_, P64_, PG, VG>, grid, 128, 0, st, p, gval)
    DIFFUS_DISPATCH(if (pose_grad && vol_grad) return DIFFUS_TB(true, true); if (pose_grad) return DIFFUS_TB(true, false);
                    return DIFFUS_TB(false, true))
#undef DIFFUS_TB
    return cudaErrorInvalidValue;
}

// ---------------------------------------------------------------------------------------
// per-ray source partials -> per-pose gradient (atomic-free, fixed order)
// ---------------------------------------------------------------------------------------
__global__ void reduce_rays_kernel(const float* __restrict__ partial, int64_t n_poses, int64_t n_rays, float* __restrict__ out) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int64_t pose = (int64_t)blockIdx.x * (blockDim.x >> 5) + warp;
    if (pose >= n_poses) return;
    float a0 = 0.f, a1 = 0.f, a2 = 0.f;
    const float* src = partial + pose * n_rays * 3;
    for (int64_t r = lane; r < n_rays; r += 32) { a0 += src[r * 3]; a1 += src[r * 3 + 1]; a2 += src[r * 3 + 2]; }
    a0 = warp_sum(a0); a1 = warp_sum(a1); a2 = warp_sum(a2);
    if (lane == 0) { out[pose * 3] = a0; out[pose * 3 + 1] = a1; out[pose * 3 + 2] = a2; }
}

cudaError_t launch_reduce_rays(const float* partial, int64_t n_poses, int64_t n_rays, float* out, cudaStream_t st) {
    unsigned grid = (unsigned)((n_poses + 3) / 4);
    return launch_kernel(reduce_rays_kernel, grid, 128, 0, st, partial, n_poses, n_rays, out);
}

// ---------------------------------------------------------------------------------------
// fans for a batch of poses (src/cone.py:242-259 per pose)
// ---------------------------------------------------------------------------------------
__global__ void cone_directions_kernel(const double* __restrict__ median, int64_t n_poses, int64_t n_rays, double angle,
                                       float* __restrict__ out) {
    const int64_t n = n_poses * n_rays;
    for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < n; t += (int64_t)gridDim.x * blockDim.x) {
        int64_t pose = t / n_rays, i = t - pose * n_rays;
        double dx = median[pose * 2], dy = median[pose * 2 + 1];
        double nrm = sqrt(__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)));
        dx /= nrm; dy /= nrm;
        double lo = -angle / 2, hi = angle / 2;
        double a = lo;                                   // numpy.linspace: start + i*step, endpoint pinned
        if (n_rays > 1) {
            double step = (hi - lo) / (double)(n_rays - 1);
            a = (i == n_rays - 1) ? hi : __dadd_rn(__dmul_rn((double)i, step), lo);
        }
        double ca = cos(a), sa = sin(a);
        out[t * 3 + 0] = (float)__dadd_rn(__dmul_rn(ca, dx), __dmul_rn(sa, -dy));
        out[t * 3 + 1] = (float)__dadd_rn(__dmul_rn(ca, dy), __dmul_rn(sa, dx));
        out[t * 3 + 2] = 0.f;
    }
}

cudaError_t launch_cone_directions(const double* median, int64_t n_poses, int64_t n_rays, double opening_angle,
                                   float* out, cudaStream_t st) {
    int64_t n = n_poses * n_rays;
    unsigned grid = (unsigned)min((int64_t)148 * 8, (n + 127) / 128);
    return launch_kernel(cone_directions_kernel, grid, 128, 0, st, median, n_poses, n_rays, opening_angle, out);
}

// ---------------------------------------------------------------------------------------
// LINEAR <-> BRICK (4x4x2 voxels = one 128-byte line)
// ---------------------------------------------------------------------------------------
template <bool TO_BRICKS>
__global__ void brick_copy_kernel(const float* __restrict__ src, float* __restrict__ dst, int D, int H, int W, int nbi,
                                  int nbj, int nbk) {
    const int64_t n = (int64_t)nbi * nbj * nbk * 32;
    for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < n; t += (int64_t)gridDim.x * blockDim.x) {
        int e = (int)(t & 31);
        int64_t b = t >> 5;
        int bk = (int)(b % nbk);
        int bj = (int)((b / nbk) % nbj);
        int bi = (int)(b / ((int64_t)nbk * nbj));
        int i = bi * BRICK_I + (e >> 3), j = bj * BRICK_J + ((e >> 1) & 3), k = bk * BRICK_K + (e & 1);
        bool ok = i < D && j < H && k < W;
        int64_t lin = ((int64_t)i * H + j) * W + k;
        if (TO_BRICKS) dst[t] = ok ? src[lin] : 0.f;
        else if (ok) dst[lin] = src[t];
    }
}

static void brick_counts(const int32_t dim[3], int& nbi, int& nbj, int& nbk) {
    nbi = (dim[0] + BRICK_I - 1) / BRICK_I;
    nbj = (dim[1] + BRICK_J - 1) / BRICK_J;
    nbk = (dim[2] + BRICK_K - 1) / BRICK_K;
}

cudaError_t launch_to_bricks(const float* linear, const int32_t dim[3], float* bricks, cudaStream_t st) {
    int nbi, nbj, nbk;
    brick_counts(dim, nbi, nbj, nbk);
    int64_t n = (int64_t)nbi * nbj * nbk * 32;
    unsigned grid = (unsigned)min((int64_t)148 * 32, (n + 255) / 256);
    return launch_kernel(brick_copy_kernel<true>, grid, 256, 0, st, linear, bricks, dim[0], dim[1], dim[2], nbi, nbj, nbk);
}

cudaError_t launch_from_bricks(const float* bricks, const int32_t dim[3], float* linear, cudaStream_t st) {
    int nbi, nbj, nbk;
    brick_counts(dim, nbi, nbj, nbk);
    int64_t n = (int64_t)nbi * nbj * nbk * 32;
    unsigned grid = (unsigned)min((int64_t)148 * 32, (n + 255) / 256);
    return launch_kernel(brick_copy_kernel<false>, grid, 256, 0, st, bricks, linear, dim[0], dim[1], dim[2], nbi, nbj, nbk);
}

// ---------------------------------------------------------------------------------------
// LINEAR -> QUAD: element (i, j, k) = (Z[i,j,k], Z[i,j+1,k], Z[i,j,k+1], Z[i,j+1,k+1]) with +1 clamped at the faces
// (the i1 = min(i0 + 1, n - 1) rule of the sampler); 2x2x2 elements per 128-byte line, the i-pair in one sector.
// ---------------------------------------------------------------------------------------
__global__ void quad_copy_kernel(const float* __restrict__ src, float4* __restrict__ dst, int D, int H, int W, int nqi,
                                 int nqj, int nqk) {
    const int64_t n = (int64_t)nqi * nqj * nqk * 8;
    for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < n; t += (int64_t)gridDim.x * blockDim.x) {
        int e = (int)(t & 7);
        int64_t b = t >> 3;
        int bk = (int)(b % nqk);
        int bj = (int)((b / nqk) % nqj);
        int bi = (int)(b / ((int64_t)nqk * nqj));
        int i = bi * QUAD_B + (e & 1), k = bk * QUAD_B + ((e >> 1) & 1), j = bj * QUAD_B + ((e >> 2) & 1);
        float4 q = make_float4(0.f, 0.f, 0.f, 0.f);
        if (i < D && j < H && k < W) {
            const int j1 = min(j + 1, H - 1), k1 = min(k + 1, W - 1);
            const float* slab = src + (int64_t)i * H * W;
            q = make_float4(slab[(int64_t)j * W + k], slab[(int64_t)j1 * W + k], slab[(int64_t)j * W + k1], slab[(int64_t)j1 * W + k1]);
        }
        dst[t] = q;
    }
}

cudaError_t launch_to_quads(const float* linear, const int32_t dim[3], float* quads, cudaStream_t st) {
    int nqi = (dim[0] + QUAD_B - 1) / QUAD_B, nqj = (dim[1] + QUAD_B - 1) / QUAD_B, nqk = (dim[2] + QUAD_B - 1) / QUAD_B;
    int64_t n = (int64_t)nqi * nqj * nqk * 8;
    unsigned grid = (unsigned)min((int64_t)148 * 32, (n + 255) / 256);
    return launch_kernel(quad_copy_kernel, grid, 256, 0, st, linear, (float4*)quads, dim[0], dim[1], dim[2], nqi, nqj, nqk);
}

// ---------------------------------------------------------------------------------------
// roofline probe: random 32-byte-sector reads (measurement aid, include/diffus_b200.h)
// ---------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) gather_probe_kernel(const float* __restrict__ buf, uint32_t n_sectors, int reads,
                                                           uint32_t seed, float* __restrict__ sink) {
    const uint32_t tid = blockIdx.x * blockDim.x + threadIdx.x;
    uint32_t h = (tid + 1u) * 2654435761u ^ seed;
    float acc[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    for (int r = 0; r < reads; r += 8) {
#pragma unroll
        for (int u = 0; u < 8; ++u) {                    // eight independent loads in flight per thread
            h ^= h << 13; h ^= h >> 17; h ^= h << 5;     // xorshift32
            const uint32_t sector = (uint32_t)(((uint64_t)h * n_sectors) >> 32);
            acc[u] += __ldg(buf + (size_t)sector * 8 + (h & 7u));
        }
    }
    sink[tid] = ((acc[0] + acc[1]) + (acc[2] + acc[3])) + ((acc[4] + acc[5]) + (acc[6] + acc[7]));
}

cudaError_t launch_gather_probe(const float* buf, int64_t n_floats, int reads, int64_t n_threads, uint32_t seed, float* sink,
                                cudaStream_t st) {
    return launch_kernel(gather_probe_kernel, (unsigned)(n_threads / 256), 256, 0, st, buf, (uint32_t)(n_floats / 8), reads, seed, sink);
}

// ---------------------------------------------------------------------------------------
// fans in an arbitrary plane for a batch of poses, from pose PARAMETERS (north_star: "source position and
// direction, cone aperture and ray count in"): ray i = cos(a_i) m^ + sin(a_i) u^, a = linspace(-angle/2, angle/2, R),
// m^ = median / |median|, u^ = the normal hint made orthogonal to m^ and normalised -- generate_cone_directions
// (src/cone.py:242-259) generalised from the z = 0 plane, float64 arithmetic and a float32 result like the reference.
// The backward takes d loss / d directions (P,R,3) to d loss / d median and d loss / d hint.
// ---------------------------------------------------------------------------------------
struct FanFrame {
    double m[3], u[3], nm, nu, hm;       // unit median, unit in-plane axis, |median|, |hint - (hint.m^) m^|, hint.m^
};
__device__ __forceinline__ FanFrame fan_frame(const float* median, const float* hint) {
    FanFrame f;
    double mx = median[0], my = median[1], mz = median[2], hx = hint[0], hy = hint[1], hz = hint[2];
    f.nm = sqrt(mx * mx + my * my + mz * mz);
    f.m[0] = mx / f.nm; f.m[1] = my / f.nm; f.m[2] = mz / f.nm;
    f.hm = hx * f.m[0] + hy * f.m[1] + hz * f.m[2];
    double ux = hx - f.hm * f.m[0], uy = hy - f.hm * f.m[1], uz = hz - f.hm * f.m[2];
    f.nu = sqrt(ux * ux + uy * uy + uz * uz);
    f.u[0] = ux / f.nu; f.u[1] = uy / f.nu; f.u[2] = uz / f.nu;
    return f;
}
__device__ __forceinline__ double fan_angle(int64_t i, int64_t n_rays, double angle) {
    const double lo = -angle / 2, hi = angle / 2;
    if (n_rays <= 1) return lo;
    return (i == n_rays - 1) ? hi : (double)i * ((hi - lo) / (double)(n_rays - 1)) + lo;
}

// d loss / d m^ and d loss / d u^ (as independent vectors) -> d loss / d median and d loss / d hint (3 floats each, overwritten)
// through the normalisations and the Gram-Schmidt step of fan_frame
__device__ __forceinline__ void fan_frame_bwd(const float* median, const float* hint, int64_t pose, const double gm[3],
                                              const double gu[3], float* grad_median, float* grad_hint) {
    const FanFrame f = fan_frame(median + pose * 3, hint + pose * 3);
    // u^ = u / |u|
    double gud = gu[0] * f.u[0] + gu[1] * f.u[1] + gu[2] * f.u[2], gv[3];
#pragma unroll
    for (int a = 0; a < 3; ++a) gv[a] = (gu[a] - gud * f.u[a]) / f.nu;              // d loss / d u
    // u = h - (h.m^) m^
    const double gvm = gv[0] * f.m[0] + gv[1] * f.m[1] + gv[2] * f.m[2];
    double gmt[3];
#pragma unroll
    for (int a = 0; a < 3; ++a) {
        const double h = (double)hint[pose * 3 + a];
        grad_hint[pose * 3 + a] = (float)(gv[a] - gvm * f.m[a]);
        gmt[a] = gm[a] - f.hm * gv[a] - gvm * h;                                        // total d loss / d m^
    }
    // m^ = m / |m|
    const double gmd = gmt[0] * f.m[0] + gmt[1] * f.m[1] + gmt[2] * f.m[2];
#pragma unroll
    for (int a = 0; a < 3; ++a) grad_median[pose * 3 + a] = (float)((gmt[a] - gmd * f.m[a]) / f.nm);
}

__global__ void fan_directions_kernel(const float* __restrict__ median, const float* __restrict__ hint, int64_t n_poses,
                                      int64_t n_rays, double angle, float* __restrict__ out) {
    const int64_t pose = blockIdx.x;
    const FanFrame f = fan_frame(median + pose * 3, hint + pose * 3);
    for (int64_t i = threadIdx.x; i < n_rays; i += blockDim.x) {
        double sa, ca;
        sincos(fan_angle(i, n_rays, angle), &sa, &ca);
        float* o = out + (pose * n_rays + i) * 3;
#pragma unroll
        for (int a = 0; a < 3; ++a) o[a] = (float)(ca * f.m[a] + sa * f.u[a]);
    }
}

__global__ void fan_directions_bwd_kernel(const float* __restrict__ median, const float* __restrict__ hint,
                                          const float* __restrict__ grad_dirs, int64_t n_poses, int64_t n_rays, double angle,
                                          float* __restrict__ grad_median, float* __restrict__ grad_hint) {
    const int64_t pose = blockIdx.x;                       // one warp per pose
    const int lane = threadIdx.x;
    double gm[3] = {0, 0, 0}, gu[3] = {0, 0, 0};           // d loss / d m^ and d loss / d u^ (as independent vectors)
    for (int64_t i = lane; i < n_rays; i += 32) {
        double sa, ca;
        sincos(fan_angle(i, n_rays, angle), &sa, &ca);
        const float* g = grad_dirs + (pose * n_rays + i) * 3;
#pragma unroll
        for (int a = 0; a < 3; ++a) { gm[a] += ca * (double)g[a]; gu[a] += sa * (double)g[a]; }
    }
#pragma unroll
    for (int a = 0; a < 3; ++a)
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) {
            gm[a] += __shfl_xor_sync(FULL, gm[a], d);
            gu[a] += __shfl_xor_sync(FULL, gu[a], d);
        }
    if (lane != 0) return;
    fan_frame_bwd(median, hint, pose, gm, gu, grad_median, grad_hint);
}

cudaError_t launch_fan_directions(const float* median, const float* hint, int64_t n_poses, int64_t n_rays, double angle,
                                  float* out, cudaStream_t st) {
    return launch_kernel(fan_directions_kernel, (unsigned)n_poses, 128, 0, st, median, hint, n_poses, n_rays, angle, out);
}

cudaError_t launch_fan_directions_bwd(const float* median, const float* hint, const float* grad_dirs, int64_t n_poses,
                                      int64_t n_rays, double angle, float* grad_median, float* grad_hint, cudaStream_t st) {
    return launch_kernel(fan_directions_bwd_kernel, (unsigned)n_poses, 32, 0, st, median, hint, grad_dirs, n_poses, n_rays, angle, grad_median,
                                                                grad_hint);
}


// ---------------------------------------------------------------------------------------
// array probes from pose PARAMETERS (centre, median, hint; m^ and u^ as in the fan above), one origin per ray:
//   convex (opening angle, radius rho >= 0): d_i = cos a_i m^ + sin a_i u^ exactly as fan_directions_kernel forms it, and
//          origin_i = c + rho d_i on the arc, in double -- rho = 0 gives the sector probe's rays bit for bit;
//   linear (width w > 0): d_i = m^ for every ray, origin_i = c + t_i u^ with t_i spread over [-w/2, w/2] by fan_angle's rule.
// The backward maps d loss / d origins and d loss / d directions (P,R,3 each) to d loss / d centre, median and hint (P,3 each).
// ---------------------------------------------------------------------------------------
__global__ void probe_rays_kernel(int kind, const float* __restrict__ centre, const float* __restrict__ median,
                                  const float* __restrict__ hint, int64_t n_rays, double angle, double radius, double width,
                                  float* __restrict__ origins, float* __restrict__ dirs) {
    const int64_t pose = blockIdx.x;
    const FanFrame f = fan_frame(median + pose * 3, hint + pose * 3);
    const double c[3] = {(double)centre[pose * 3], (double)centre[pose * 3 + 1], (double)centre[pose * 3 + 2]};
    for (int64_t i = threadIdx.x; i < n_rays; i += blockDim.x) {
        float* o = origins + (pose * n_rays + i) * 3;
        float* d = dirs + (pose * n_rays + i) * 3;
        if (kind == DIFFUS_PROBE_CONVEX) {
            double sa, ca;
            sincos(fan_angle(i, n_rays, angle), &sa, &ca);
#pragma unroll
            for (int a = 0; a < 3; ++a) {
                const double w = ca * f.m[a] + sa * f.u[a];
                d[a] = (float)w;
                o[a] = (float)(c[a] + radius * w);
            }
        } else {
            const double t = fan_angle(i, n_rays, width);
#pragma unroll
            for (int a = 0; a < 3; ++a) {
                d[a] = (float)f.m[a];
                o[a] = (float)(c[a] + t * f.u[a]);
            }
        }
    }
}

__global__ void probe_rays_bwd_kernel(int kind, const float* __restrict__ median, const float* __restrict__ hint,
                                      const float* __restrict__ grad_origins, const float* __restrict__ grad_dirs, int64_t n_rays,
                                      double angle, double radius, double width, float* __restrict__ grad_centre,
                                      float* __restrict__ grad_median, float* __restrict__ grad_hint) {
    const int64_t pose = blockIdx.x;                       // one warp per pose
    const int lane = threadIdx.x;
    double gc[3] = {0, 0, 0}, gm[3] = {0, 0, 0}, gu[3] = {0, 0, 0};
    for (int64_t i = lane; i < n_rays; i += 32) {
        const float* go = grad_origins + (pose * n_rays + i) * 3;
        const float* gd = grad_dirs + (pose * n_rays + i) * 3;
        if (kind == DIFFUS_PROBE_CONVEX) {
            double sa, ca;
            sincos(fan_angle(i, n_rays, angle), &sa, &ca);
#pragma unroll
            for (int a = 0; a < 3; ++a) {
                const double g = (double)gd[a] + radius * (double)go[a];      // d_i and the arc point both follow the fan ray
                gm[a] += ca * g;
                gu[a] += sa * g;
                gc[a] += (double)go[a];
            }
        } else {
            const double t = fan_angle(i, n_rays, width);
#pragma unroll
            for (int a = 0; a < 3; ++a) {
                gm[a] += (double)gd[a];
                gu[a] += t * (double)go[a];
                gc[a] += (double)go[a];
            }
        }
    }
#pragma unroll
    for (int a = 0; a < 3; ++a)
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) {
            gc[a] += __shfl_xor_sync(FULL, gc[a], d);
            gm[a] += __shfl_xor_sync(FULL, gm[a], d);
            gu[a] += __shfl_xor_sync(FULL, gu[a], d);
        }
    if (lane != 0) return;
#pragma unroll
    for (int a = 0; a < 3; ++a) grad_centre[pose * 3 + a] = (float)gc[a];
    fan_frame_bwd(median, hint, pose, gm, gu, grad_median, grad_hint);
}

cudaError_t launch_probe_rays(int kind, const float* centre, const float* median, const float* hint, int64_t n_poses, int64_t n_rays,
                              double angle, double radius, double width, float* origins, float* dirs, cudaStream_t st) {
    return launch_kernel(probe_rays_kernel, (unsigned)n_poses, 128, 0, st, kind, centre, median, hint, n_rays, angle, radius, width, origins, dirs);
}

cudaError_t launch_probe_rays_bwd(int kind, const float* centre, const float* median, const float* hint, const float* grad_origins,
                                  const float* grad_dirs, int64_t n_poses, int64_t n_rays, double angle, double radius, double width,
                                  float* grad_centre, float* grad_median, float* grad_hint, cudaStream_t st) {
    (void)centre;                                          // the centre enters the origins linearly
    return launch_kernel(probe_rays_bwd_kernel, (unsigned)n_poses, 32, 0, st, kind, median, hint, grad_origins, grad_dirs, n_rays, angle, radius, width,
                                                            grad_centre, grad_median, grad_hint);
}

}  // namespace diffus
