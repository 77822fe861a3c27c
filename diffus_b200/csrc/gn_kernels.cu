// Gauss-Newton system of the frame residual w.r.t. a rigid twist of each pose, in one forward-mode pass (sm_100a).
//
// A pose update is the twist xi = (v, w) about the current pose, rotating about the source: p_k(xi) = (s + v) + k Rot(w) d_i,
// so every sample's impedance has the tangent dZ_k / dxi = (grad Z_k, k (d_i x grad Z_k)) -- the spatial gradient the trilinear
// gather already forms for the pose-gradient kernels.  With one origin s_i per ray (array probes) the probe turns about its
// pivot c, the float64 mean of the pose's origins: p_k(xi) = c + v + Rot(w) (s_i - c + k d_i), tangent (grad Z_k,
// (o_i + k d_i) x grad Z_k) with the lever o_i = s_i - c (the GN_LEVER_POSE instantiations; the per-pose ones are unchanged).  A
// tracked sweep shares ONE twist and one pivot c among all poses (GN_LEVER_SWEEP): the lever is o_i = s_i - c with s_i the pose's
// source or the ray's own origin, and the per-ray partials of every pose are summed into one system (gn_sweep_sum_kernel).
// The transfer-matrix prefix is carried as a DUAL pair (P, Pdot_1..6):
// (P, Pdot) (M, Mdot) = (P M, Pdot M + P Mdot) is associative, so the march keeps the structure of the forward kernel --
// lane-local chunk products, one warp scan, a second sweep -- with no reverse sweep and no prefix pre-pass.  Per column
//     rdot  = ((Zdot_c - Zdot_{c-1}) - r (Zdot_{c-1} + Zdot_c)) / (Z_{c-1} + Z_c)      (d of (Z_c - Z_{c-1}) / (Z_{c-1} + Z_c))
//     Mdot  = rdot [[-4 r, 1], [-1, 0]]
//     edot  = (Pdot[0][1] - e Pdot[1][1]) / P[1][1],    J = att edot
// and each ray leaves its share of loss = sum res^2, Jtr = sum J res and the 21 entries of JtJ = sum J J^T (res = frame - target)
// as one per-ray partial; a second launch adds the partials of a pose in a fixed order (no atomics: run-to-run identical).
// DESIGN.md section 4 states the math and the NaN / median rules.
#include "common.cuh"
#include "launch.h"

namespace diffus {

constexpr int GN_ROW = FwdGeo::OBUF;          // one padded row of a 512-column pass
// rows of the per-warp shared-memory block: r, rdot_0..5, attenuation, target
constexpr int GN_R = 0, GN_RD = 1, GN_ATT = 7, GN_TGT = 8, GN_ROWS = 9;
constexpr int GN_CARRY = 28;                  // the dual prefix entering the pass (written by lane 31)
constexpr int GN_SMEM_PER_WARP = GN_ROWS * GN_ROW + GN_CARRY + 4;

// dual 2x2 matrix: value and its six tangents
struct D2 {
    M2 v;
    M2 t[6];
};

__device__ __forceinline__ D2 d2_identity() {
    D2 x;
    x.v = m2_identity();
#pragma unroll
    for (int j = 0; j < 6; ++j) x.t[j] = m2_zero();
    return x;
}

__device__ __forceinline__ D2 d2_mul(const D2& x, const D2& y) {
    D2 z;
    z.v = m2_mul(x.v, y.v);
#pragma unroll
    for (int j = 0; j < 6; ++j) z.t[j] = m2_add(m2_mul(x.t[j], y.v), m2_mul(x.v, y.t[j]));
    return z;
}

// x <- x (M(r), rdot dM/dr)
__device__ __forceinline__ void d2_mul_interface(D2& x, float r, const float rd[6]) {
    const float2 q0 = __ffma2_rn(x.v.c0, bcast(-4.f * r), make_float2(-x.v.c1.x, -x.v.c1.y));   // P dM/dr, column 0
    const float2 q1 = x.v.c0;                                                                    //          column 1
#pragma unroll
    for (int j = 0; j < 6; ++j) {
        M2 t = m2_mul_interface(x.t[j], r);
        t.c0 = __ffma2_rn(q0, bcast(rd[j]), t.c0);
        t.c1 = __ffma2_rn(q1, bcast(rd[j]), t.c1);
        x.t[j] = t;
    }
    x.v = m2_mul_interface(x.v, r);
}

__device__ __forceinline__ D2 d2_shfl_up(const D2& x, int d) {
    D2 y;
    y.v = m2_shfl_up(x.v, d);
#pragma unroll
    for (int j = 0; j < 6; ++j) y.t[j] = m2_shfl_up(x.t[j], d);
    return y;
}
__device__ __forceinline__ D2 d2_shfl(const D2& x, int src) {
    D2 y;
    y.v = m2_shfl(x.v, src);
#pragma unroll
    for (int j = 0; j < 6; ++j) y.t[j] = m2_shfl(x.t[j], src);
    return y;
}
__device__ __forceinline__ void d2_store(float* s, const D2& x) {
    s[0] = x.v.a(); s[1] = x.v.b(); s[2] = x.v.c(); s[3] = x.v.d();
#pragma unroll
    for (int j = 0; j < 6; ++j) {
        s[4 + 4 * j] = x.t[j].a(); s[5 + 4 * j] = x.t[j].b(); s[6 + 4 * j] = x.t[j].c(); s[7 + 4 * j] = x.t[j].d();
    }
}
__device__ __forceinline__ D2 d2_load(const float* s) {
    D2 x;
    x.v = m2_make(s[0], s[1], s[2], s[3]);
#pragma unroll
    for (int j = 0; j < 6; ++j) x.t[j] = m2_make(s[4 + 4 * j], s[5 + 4 * j], s[6 + 4 * j], s[7 + 4 * j]);
    return x;
}

// the lane's sample tangent (grad Z, k (d x grad Z)); with a pivot: (grad Z, (o + k d) x grad Z) with the ray's lever o
template <int LEVER>
__device__ __forceinline__ void sample_tangent(const float d[3], const float o[3], const float g[3], float kf, float t[6]) {
    t[0] = g[0]; t[1] = g[1]; t[2] = g[2];
    if (LEVER != GN_LEVER_SOURCE) {
        const float a0 = fmaf(kf, d[0], o[0]), a1 = fmaf(kf, d[1], o[1]), a2 = fmaf(kf, d[2], o[2]);
        t[3] = a1 * g[2] - a2 * g[1];
        t[4] = a2 * g[0] - a0 * g[2];
        t[5] = a0 * g[1] - a1 * g[0];
    } else {
        t[3] = kf * (d[1] * g[2] - d[2] * g[1]);
        t[4] = kf * (d[2] * g[0] - d[0] * g[2]);
        t[5] = kf * (d[0] * g[1] - d[1] * g[0]);
    }
}

// the ray's lever o = s_i - c about its pose's pivot, or about the sweep's one pivot (float64 difference, one rounding)
template <int LEVER>
__device__ __forceinline__ void ray_lever(const RaySetup<false>& rs, const double* __restrict__ pivot, int64_t pose, float o[3]) {
#pragma unroll
    for (int a = 0; a < 3; ++a) {
        if (LEVER == GN_LEVER_POSE) o[a] = (float)((double)rs.s[a] - __ldg(pivot + pose * 3 + a));
        else if (LEVER == GN_LEVER_SWEEP) o[a] = (float)((double)rs.s[a] - __ldg(pivot + a));
        else o[a] = 0.f;
    }
}

__device__ __forceinline__ int64_t gn_pose_of_ray(int64_t ray, const RenderParams& p) {
    if (p.total_rays <= 0xffffffffLL) return (int64_t)((uint32_t)ray / (uint32_t)p.n_rays);
    return ray / p.n_rays;
}

// One warp per ray, passes of 512 columns.  Gather phase (lane = consecutive column): Z and grad Z of the sample, its tangent,
// the neighbour's by one shuffle, and the column's r, rdot, attenuation and target parked in shared memory.  Chunk phase (lane =
// 16 consecutive columns): the dual chunk product, one warp scan, the second sweep forming e, J and the accumulators.  The dual
// prefix entering the next pass goes through shared memory, so it is not live during the gathers.
template <int LAYOUT, int LEVER>
__global__ void __launch_bounds__(128) render_gn_kernel(const RenderParams p, const float* __restrict__ med_tan,
                                                        const double* __restrict__ pivot, float* __restrict__ partial) {
    using G = FwdGeo;
    constexpr int CH = G::CHUNK;
    extern __shared__ __align__(16) float smem[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int64_t ray = (int64_t)blockIdx.x * (blockDim.x >> 5) + warp;
    if (ray >= p.total_rays) return;
    float* rows = smem + warp * GN_SMEM_PER_WARP;
    float* carry_s = rows + GN_ROWS * GN_ROW;
    const int64_t pose = gn_pose_of_ray(ray, p);
    RaySetup<false> rs;
    rs.load(p.sources, p.directions, pose, ray - pose * p.n_rays, p.src_pose_stride, p.src_ray_stride, p.dir_pose_stride, 0);
    float lever[3];
    ray_lever<LEVER>(rs, pivot, pose, lever);
    const bool has_med = p.median != nullptr;
    const float med = has_med ? __ldg(p.median + pose) : 0.f;
    float mt[6];
#pragma unroll
    for (int j = 0; j < 6; ++j) mt[j] = has_med ? __ldg(med_tan + pose * 6 + j) : 0.f;
    const float* tgt = p.target + ray * (int64_t)p.Sout;
    if (lane == 0) d2_store(carry_s, d2_identity());

    float zc_prev = 0.f, tc_prev[6] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f};    // the sample before the current tile
    float acc[28];
#pragma unroll
    for (int q = 0; q < 28; ++q) acc[q] = 0.f;

    constexpr int GB = LAYOUT == DIFFUS_LAYOUT_TEXTURE ? 4 : 2;          // tiles of gathers in flight
    for (int c0 = 0; c0 < p.Sout; c0 += G::SEG) {
        const int ncol = min(G::SEG, p.Sout - c0);
        const int ntile = (ncol + 31) >> 5;
        for (int t0 = 0; t0 < ntile; t0 += GB) {
            Fetch<DIFFUS_SAMPLER_TRILINEAR, LAYOUT> fe[GB];
#pragma unroll
            for (int u = 0; u < GB; ++u) {
                const int idx = (t0 + u) * 32 + lane;
                if (t0 + u < ntile && idx < ncol) {
                    const int k = p.start + c0 + idx;
                    fe[u].template issue<true>(p.vol, rs.coord(0, k), rs.coord(1, k), rs.coord(2, k));
                }
            }
#pragma unroll
            for (int u = 0; u < GB; ++u) {
                if (t0 + u >= ntile) break;                                  // warp-uniform
                const int idx = (t0 + u) * 32 + lane;
                const bool ok = idx < ncol;
                const int c = c0 + idx;
                float g[3] = {0.f, 0.f, 0.f};
                float z = 0.f;
                if (ok) z = fe[u].template finish<true>(g);
                float tz[6];
                sample_tangent<LEVER>(rs.d, lever, g, (float)(p.start + c), tz);
                float zp = __shfl_up_sync(FULL, z, 1);
                float tp[6];
#pragma unroll
                for (int j = 0; j < 6; ++j) tp[j] = __shfl_up_sync(FULL, tz[j], 1);
                if (lane == 0) {
                    zp = zc_prev;
#pragma unroll
                    for (int j = 0; j < 6; ++j) tp[j] = tc_prev[j];
                }
                zc_prev = __shfl_sync(FULL, z, 31);
#pragma unroll
                for (int j = 0; j < 6; ++j) tc_prev[j] = __shfl_sync(FULL, tz[j], 31);
                const float inv = fast_rcp(__fadd_rn(zp, z));
                float r = __fmul_rn(__fsub_rn(z, zp), inv);                   // reflection() of the render kernels
                float rd[6];
#pragma unroll
                for (int j = 0; j < 6; ++j) rd[j] = ((tz[j] - tp[j]) - r * (tp[j] + tz[j])) * inv;
                if (c == 1 && has_med) {                                     // the pose's median replaces column 1
                    r = med;
#pragma unroll
                    for (int j = 0; j < 6; ++j) rd[j] = mt[j];
                }
                if (c == 0 || !ok) {                                         // column 0 owns no interface
                    r = 0.f;
#pragma unroll
                    for (int j = 0; j < 6; ++j) rd[j] = 0.f;
                }
                const int s = G::pad(idx);
                rows[GN_R * GN_ROW + s] = r;
#pragma unroll
                for (int j = 0; j < 6; ++j) rows[(GN_RD + j) * GN_ROW + s] = rd[j];
                rows[GN_ATT * GN_ROW + s] = expf(-p.alpha * (float)c);
                rows[GN_TGT * GN_ROW + s] = ok ? __ldg(tgt + c) : 0.f;
            }
        }
        __syncwarp();

        // chunk phase
        const int lc = lane * CH;
        auto load_col = [&](int i, float& r, float rd[6]) {
            const int s = G::pad(lc + i);
            const bool ok = lc + i < ncol;                                    // columns beyond the pass: identity
            r = ok ? rows[GN_R * GN_ROW + s] : 0.f;
#pragma unroll
            for (int j = 0; j < 6; ++j) rd[j] = ok ? rows[(GN_RD + j) * GN_ROW + s] : 0.f;
        };
        D2 P = d2_identity();
#pragma unroll 4
        for (int i = 0; i < CH; ++i) {
            float r, rd[6];
            load_col(i, r, rd);
            d2_mul_interface(P, r, rd);
        }
        // exclusive scan of the chunk products, then the prefix entering the pass on the left
#pragma unroll 1
        for (int d = 1; d < 32; d <<= 1) {
            const D2 left = d2_shfl_up(P, d);
            if (lane >= d) P = d2_mul(left, P);
        }
        {
            D2 exc = d2_shfl_up(P, 1);
            if (lane == 0) exc = d2_identity();
            P = d2_mul(d2_load(carry_s), exc);
        }
#pragma unroll 2
        for (int i = 0; i < CH; ++i) {
            float r, rd[6];
            load_col(i, r, rd);
            d2_mul_interface(P, r, rd);
            if (lc + i < ncol) {
                const int s = G::pad(lc + i);
                const float att = rows[GN_ATT * GN_ROW + s];
                const float inv = fast_rcp(P.v.d());
                const float e = echo_of(P.v.b(), inv);
                const bool finite = fabsf(e) <= FLT_MAX;                     // NaN rule of the fused MSE kernel: no tangent
                const float res = __fmul_rn(nan_to_num(e), att) - rows[GN_TGT * GN_ROW + s];
                float J[6];
#pragma unroll
                for (int j = 0; j < 6; ++j) J[j] = finite ? (P.t[j].b() - e * P.t[j].d()) * inv * att : 0.f;
                acc[0] = fmaf(res, res, acc[0]);
#pragma unroll
                for (int j = 0; j < 6; ++j) acc[1 + j] = fmaf(J[j], res, acc[1 + j]);
                int q = 7;
#pragma unroll
                for (int a = 0; a < 6; ++a)
#pragma unroll
                    for (int b = a; b < 6; ++b) { acc[q] = fmaf(J[a], J[b], acc[q]); ++q; }
            }
        }
        __syncwarp();
        if (lane == 31) d2_store(carry_s, P);                                // prefix through the pass's last column
        __syncwarp();
    }
    // the ray's 28 sums: four transposing reductions of eight values
    float* out = partial + ray * 32;
#pragma unroll
    for (int g = 0; g < 4; ++g) {
        float v[8];
#pragma unroll
        for (int q = 0; q < 8; ++q) v[q] = 8 * g + q < 28 ? acc[8 * g + q] : 0.f;
        const float t = warp_sum8(v, lane);
        if (lane < 8) out[8 * g + warp_sum8_index(lane)] = t;
    }
}

// Per pose: the 32-float partials of its rays summed in a fixed order in double -> loss, Jtr (6) and the symmetric JtJ (6x6).
__global__ void __launch_bounds__(128) gn_reduce_kernel(const float* __restrict__ partial, int64_t n_rays, float* __restrict__ loss,
                                                        float* __restrict__ jtr, float* __restrict__ jtj) {
    __shared__ double part[4][32];
    const int64_t pose = blockIdx.x;
    const int t = threadIdx.x & 31, grp = threadIdx.x >> 5;
    const float* src = partial + pose * n_rays * 32 + t;
    double a0 = 0.0, a1 = 0.0;
    int64_t r = grp;
    for (; r + 4 < n_rays; r += 8) { a0 += (double)__ldg(src + r * 32); a1 += (double)__ldg(src + (r + 4) * 32); }
    if (r < n_rays) a0 += (double)__ldg(src + r * 32);
    part[grp][t] = a0 + a1;
    __syncthreads();
    if (threadIdx.x >= 28) return;
    const float v = (float)((part[0][t] + part[1][t]) + (part[2][t] + part[3][t]));
    if (t == 0) {
        loss[pose] = v;
    } else if (t < 7) {
        jtr[pose * 6 + t - 1] = v;
    } else {
        int q = t - 7, a = 0;
        while (q >= 6 - a) { q -= 6 - a; ++a; }
        const int b = a + q;
        jtj[pose * 36 + a * 6 + b] = v;
        jtj[pose * 36 + b * 6 + a] = v;
    }
}

// start > 0: the tangent of the median-replaced coefficient of each pose -- torch's forward-mode rule for a full median(): the
// mean of the tangents of the rays tied with it (tie_count from first_refl_median_kernel; a NaN median has no tangent).  The
// coefficient is formed exactly like first_refl_median_kernel does (same expression, IEEE division), so the ties it counted are
// the ties found here.  One warp per pose.
template <int LAYOUT, int LEVER>
__global__ void gn_median_tangent_kernel(const RenderParams p, const int32_t* __restrict__ tie_count, const double* __restrict__ pivot,
                                         float* __restrict__ med_tan) {
    const int64_t pose = blockIdx.x;
    const int lane = threadIdx.x;
    const float med = p.median[pose];
    const int ties = tie_count[pose];
    const int k = p.start;
    float acc[6] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    for (int64_t m = lane; m < p.n_rays && ties > 0; m += 32) {
        RaySetup<false> rs;
        rs.load(p.sources, p.directions, pose, m, p.src_pose_stride, p.src_ray_stride, p.dir_pose_stride, 0);
        float g0[3], g1[3];
        const float z0 = sample_volume<DIFFUS_SAMPLER_TRILINEAR, LAYOUT, true>(p.vol, rs.coord(0, k), rs.coord(1, k), rs.coord(2, k), g0);
        const float z1 = sample_volume<DIFFUS_SAMPLER_TRILINEAR, LAYOUT, true>(p.vol, rs.coord(0, k + 1), rs.coord(1, k + 1),
                                                                               rs.coord(2, k + 1), g1);
        if (!((z1 - z0) / (z0 + z1) == med)) continue;
        float lever[3], t0[6], t1[6];
        ray_lever<LEVER>(rs, pivot, pose, lever);
        sample_tangent<LEVER>(rs.d, lever, g0, (float)k, t0);
        sample_tangent<LEVER>(rs.d, lever, g1, (float)(k + 1), t1);
        const float sum = z0 + z1;
        const float w = 2.f / (sum * sum);
#pragma unroll
        for (int j = 0; j < 6; ++j) acc[j] += w * (z0 * t1[j] - z1 * t0[j]);
    }
#pragma unroll
    for (int j = 0; j < 6; ++j) {
        const float s = warp_sum(acc[j]);
        if (lane == 0) med_tan[pose * 6 + j] = ties > 0 ? s / (float)ties : 0.f;
    }
}

// Per-ray origins: the pivot of each pose, the mean of its R origins in double (lane-strided sums, then a butterfly: the same
// order on every run).  One warp per pose.
__global__ void __launch_bounds__(128) gn_pivot_kernel(const float* __restrict__ src, int64_t n_poses, int64_t n_rays,
                                                       double* __restrict__ pivot) {
    const int lane = threadIdx.x & 31;
    const int64_t pose = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (pose >= n_poses) return;
    const float* s = src + pose * n_rays * 3;
    double a[3] = {0.0, 0.0, 0.0};
    for (int64_t r = lane; r < n_rays; r += 32)
#pragma unroll
        for (int j = 0; j < 3; ++j) a[j] += (double)__ldg(s + r * 3 + j);
#pragma unroll
    for (int j = 0; j < 3; ++j) {
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) a[j] += __shfl_xor_sync(FULL, a[j], d);
        if (lane == 0) pivot[pose * 3 + j] = a[j] / (double)n_rays;
    }
}

// Tracked sweeps.  A sum over all P*R rows is split into contiguous ranges whose length follows from the row count alone
// (gn_sweep_range_rows), each range summed by one CTA in a fixed order, then the range sums by one CTA in a fixed order: no
// atomics, the same additions in the same order on every run and every device.
constexpr int SWEEP_THREADS = 256;
constexpr int64_t SWEEP_MAX_RANGES = 512;

static int64_t gn_sweep_range_rows(int64_t rows) {
    const int64_t len = (rows + SWEEP_MAX_RANGES - 1) / SWEEP_MAX_RANGES;
    return len > 64 ? len : 64;
}

int64_t gn_sweep_ranges(int64_t rows) {
    const int64_t len = gn_sweep_range_rows(rows);
    return (rows + len - 1) / len;
}

// column sums of n rows of 32 values in double: eight row groups of 32 lanes (one lane per column), two chains each, then the
// groups in a fixed tree.  The result is valid in threads 0..31.
template <typename T>
__device__ __forceinline__ double sweep_sum_columns(const T* __restrict__ rows, int64_t n, double (*part)[32]) {
    const int t = threadIdx.x & 31, grp = threadIdx.x >> 5;
    const T* src = rows + t;
    double a0 = 0.0, a1 = 0.0;
    int64_t r = grp;
#pragma unroll 4
    for (; r + 8 < n; r += 16) { a0 += (double)__ldg(src + r * 32); a1 += (double)__ldg(src + (r + 8) * 32); }
    if (r < n) a0 += (double)__ldg(src + r * 32);
    part[grp][t] = a0 + a1;
    __syncthreads();
    return ((part[0][t] + part[1][t]) + (part[2][t] + part[3][t])) + ((part[4][t] + part[5][t]) + (part[6][t] + part[7][t]));
}

// stage 1: CTA b sums the 32-float per-ray partials of rays [b len, (b + 1) len)
__global__ void __launch_bounds__(SWEEP_THREADS) gn_sweep_range_kernel(const float* __restrict__ partial, int64_t n_rows, int64_t len,
                                                                       double* __restrict__ range_sum) {
    __shared__ double part[SWEEP_THREADS / 32][32];
    const int64_t lo = (int64_t)blockIdx.x * len;
    const double v = sweep_sum_columns(partial + lo * 32, n_rows - lo < len ? n_rows - lo : len, part);
    if (threadIdx.x < 32) range_sum[(int64_t)blockIdx.x * 32 + threadIdx.x] = v;
}

// stage 2 (one CTA): the range sums -> loss, Jtr (6) and the symmetric JtJ (6x6), all double
__global__ void __launch_bounds__(SWEEP_THREADS) gn_sweep_sum_kernel(const double* __restrict__ range_sum, int64_t n_ranges,
                                                                     double* __restrict__ loss, double* __restrict__ jtr,
                                                                     double* __restrict__ jtj) {
    __shared__ double part[SWEEP_THREADS / 32][32];
    const double v = sweep_sum_columns(range_sum, n_ranges, part);
    const int t = threadIdx.x;
    if (t == 0) {
        loss[0] = v;
    } else if (t < 7) {
        jtr[t - 1] = v;
    } else if (t < 28) {
        int q = t - 7, a = 0;
        while (q >= 6 - a) { q -= 6 - a; ++a; }
        const int b = a + q;
        jtj[a * 6 + b] = v;
        jtj[b * 6 + a] = v;
    }
}

// The sweep's pivot: the mean of n_rows origins (3 floats each) in double.  Stage 1 (FINAL = false) writes the three sums of
// rows [b len, (b + 1) len) per CTA, stage 2 (FINAL, one CTA) sums those and divides by `count`.  Thread i takes rows i, i + 256,
// ...; each warp folds by a butterfly and the eight warps in a fixed tree.
template <typename T, bool FINAL>
__global__ void __launch_bounds__(SWEEP_THREADS) gn_sweep_pivot_kernel(const T* __restrict__ rows, int64_t n_rows, int64_t len,
                                                                       int64_t count, double* __restrict__ out) {
    __shared__ double part[SWEEP_THREADS / 32][3];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int64_t lo = (int64_t)blockIdx.x * len, hi = lo + len < n_rows ? lo + len : n_rows;
    double a[3] = {0.0, 0.0, 0.0};
    for (int64_t r = lo + threadIdx.x; r < hi; r += SWEEP_THREADS)
#pragma unroll
        for (int j = 0; j < 3; ++j) a[j] += (double)__ldg(rows + r * 3 + j);
#pragma unroll
    for (int j = 0; j < 3; ++j) {
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) a[j] += __shfl_xor_sync(FULL, a[j], d);
        if (lane == 0) part[warp][j] = a[j];
    }
    __syncthreads();
    if (threadIdx.x >= 3) return;
    const int j = threadIdx.x;
    const double s = ((part[0][j] + part[1][j]) + (part[2][j] + part[3][j])) + ((part[4][j] + part[5][j]) + (part[6][j] + part[7][j]));
    out[(int64_t)blockIdx.x * 3 + j] = FINAL ? s / (double)count : s;
}

cudaError_t launch_gn_sweep_pivot(const float* origins, int64_t n_rows, double* range_ws, double* pivot, cudaStream_t st) {
    const int64_t len = gn_sweep_range_rows(n_rows), g = (n_rows + len - 1) / len;
    cudaError_t e = launch_kernel(gn_sweep_pivot_kernel<float, false>, (unsigned)g, SWEEP_THREADS, 0, st, origins, n_rows, len, n_rows,
                                  range_ws);
    if (e != cudaSuccess) return e;
    return launch_kernel(gn_sweep_pivot_kernel<double, true>, 1, SWEEP_THREADS, 0, st, range_ws, g, g, n_rows, pivot);
}

cudaError_t launch_gn_pivot(const float* sources, int64_t n_poses, int64_t n_rays, double* pivot, cudaStream_t st) {
    return launch_kernel(gn_pivot_kernel, (unsigned)((n_poses + 3) / 4), 128, 0, st, sources, n_poses, n_rays, pivot);
}

static int gn_warps_per_block(int64_t total_rays) {
    if (total_rays >= 4 * 148 * 4) return 4;
    if (total_rays >= 2 * 148 * 2) return 2;
    return 1;
}

#define DIFFUS_GN_LAYOUTS(...)                                                   \
    switch (layout) {                                                             \
        case DIFFUS_LAYOUT_LINEAR: { constexpr int L_ = DIFFUS_LAYOUT_LINEAR; __VA_ARGS__; } \
        case DIFFUS_LAYOUT_BRICK: { constexpr int L_ = DIFFUS_LAYOUT_BRICK; __VA_ARGS__; }   \
        case DIFFUS_LAYOUT_QUAD: { constexpr int L_ = DIFFUS_LAYOUT_QUAD; __VA_ARGS__; }     \
        case DIFFUS_LAYOUT_TEXTURE: { constexpr int L_ = DIFFUS_LAYOUT_TEXTURE; __VA_ARGS__; } \
    }

#define DIFFUS_GN_LEVERS(...)                                                                      \
    switch (lever) {                                                                                \
        case GN_LEVER_SOURCE: { constexpr int V_ = GN_LEVER_SOURCE; DIFFUS_GN_LAYOUTS(__VA_ARGS__) break; } \
        case GN_LEVER_POSE: { constexpr int V_ = GN_LEVER_POSE; DIFFUS_GN_LAYOUTS(__VA_ARGS__) break; }     \
        case GN_LEVER_SWEEP: { constexpr int V_ = GN_LEVER_SWEEP; DIFFUS_GN_LAYOUTS(__VA_ARGS__) break; }   \
    }

cudaError_t launch_gn_median_tangent(const RenderParams& p, int layout, int lever, const int32_t* tie_count, const double* pivot,
                                     float* med_tan, cudaStream_t st) {
    DIFFUS_GN_LEVERS(return launch_kernel(gn_median_tangent_kernel<L_, V_>, (unsigned)p.n_poses, 32, 0, st, p, tie_count, pivot, med_tan))
    return cudaErrorInvalidValue;
}

// the march: one 32-float partial per ray
static cudaError_t launch_gn_march(const RenderParams& p, int layout, int lever, const float* med_tan, const double* pivot,
                                   float* partial, cudaStream_t st) {
    const int wpb = gn_warps_per_block(p.total_rays);
    const size_t smem = (size_t)wpb * GN_SMEM_PER_WARP * sizeof(float);
    const unsigned grid = (unsigned)((p.total_rays + wpb - 1) / wpb);
    DIFFUS_GN_LEVERS(auto k = render_gn_kernel<L_, V_>; cudaError_t e = ensure_smem(k, smem); if (e != cudaSuccess) return e;
                     return launch_kernel(k, grid, wpb * 32, smem, st, p, med_tan, pivot, partial))
    return cudaErrorInvalidValue;
}

cudaError_t launch_render_gn(const RenderParams& p, int layout, const float* med_tan, const double* pivot, float* partial, float* loss,
                             float* jtr, float* jtj, cudaStream_t st) {
    cudaError_t e = launch_gn_march(p, layout, pivot ? GN_LEVER_POSE : GN_LEVER_SOURCE, med_tan, pivot, partial, st);
    if (e != cudaSuccess) return e;
    return launch_kernel(gn_reduce_kernel, (unsigned)p.n_poses, 128, 0, st, partial, p.n_rays, loss, jtr, jtj);
}

cudaError_t launch_render_gn_sweep(const RenderParams& p, int layout, const float* med_tan, const double* pivot, float* partial,
                                   double* range_ws, double* loss, double* jtr, double* jtj, cudaStream_t st) {
    cudaError_t e = launch_gn_march(p, layout, GN_LEVER_SWEEP, med_tan, pivot, partial, st);
    if (e != cudaSuccess) return e;
    const int64_t len = gn_sweep_range_rows(p.total_rays), g = (p.total_rays + len - 1) / len;
    e = launch_kernel(gn_sweep_range_kernel, (unsigned)g, SWEEP_THREADS, 0, st, partial, p.total_rays, len, range_ws);
    if (e != cudaSuccess) return e;
    return launch_kernel(gn_sweep_sum_kernel, 1, SWEEP_THREADS, 0, st, range_ws, g, loss, jtr, jtj);
}

#undef DIFFUS_GN_LEVERS
#undef DIFFUS_GN_LAYOUTS

}  // namespace diffus
