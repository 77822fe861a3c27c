// Gauss-Newton system of the frame residual w.r.t. a rigid twist of each pose, in one forward-mode pass (sm_100a).
//
// A pose update is the twist xi = (v, w) about the current pose, rotating about the source: p_k(xi) = (s + v) + k Rot(w) d_i,
// so every sample's impedance has the tangent dZ_k / dxi = (grad Z_k, k (d_i x grad Z_k)) -- the spatial gradient the trilinear
// gather already forms for the pose-gradient kernels.  The transfer-matrix prefix is carried as a DUAL pair (P, Pdot_1..6):
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

// the lane's sample tangent (grad Z, k (d x grad Z))
__device__ __forceinline__ void sample_tangent(const float d[3], const float g[3], float kf, float t[6]) {
    t[0] = g[0]; t[1] = g[1]; t[2] = g[2];
    t[3] = kf * (d[1] * g[2] - d[2] * g[1]);
    t[4] = kf * (d[2] * g[0] - d[0] * g[2]);
    t[5] = kf * (d[0] * g[1] - d[1] * g[0]);
}

__device__ __forceinline__ int64_t gn_pose_of_ray(int64_t ray, const RenderParams& p) {
    if (p.total_rays <= 0xffffffffLL) return (int64_t)((uint32_t)ray / (uint32_t)p.n_rays);
    return ray / p.n_rays;
}

// One warp per ray, passes of 512 columns.  Gather phase (lane = consecutive column): Z and grad Z of the sample, its tangent,
// the neighbour's by one shuffle, and the column's r, rdot, attenuation and target parked in shared memory.  Chunk phase (lane =
// 16 consecutive columns): the dual chunk product, one warp scan, the second sweep forming e, J and the accumulators.  The dual
// prefix entering the next pass goes through shared memory, so it is not live during the gathers.
template <int LAYOUT>
__global__ void __launch_bounds__(128) render_gn_kernel(const RenderParams p, const float* __restrict__ med_tan,
                                                        float* __restrict__ partial) {
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
    rs.load(p.sources, p.directions, pose, ray - pose * p.n_rays, p.n_rays, p.dir_pose_stride, 0);
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
                sample_tangent(rs.d, g, (float)(p.start + c), tz);
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
template <int LAYOUT>
__global__ void gn_median_tangent_kernel(const RenderParams p, const int32_t* __restrict__ tie_count, float* __restrict__ med_tan) {
    const int64_t pose = blockIdx.x;
    const int lane = threadIdx.x;
    const float med = p.median[pose];
    const int ties = tie_count[pose];
    const int k = p.start;
    float acc[6] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    for (int64_t m = lane; m < p.n_rays && ties > 0; m += 32) {
        RaySetup<false> rs;
        rs.load(p.sources, p.directions, pose, m, p.n_rays, p.dir_pose_stride, 0);
        float g0[3], g1[3];
        const float z0 = sample_volume<DIFFUS_SAMPLER_TRILINEAR, LAYOUT, true>(p.vol, rs.coord(0, k), rs.coord(1, k), rs.coord(2, k), g0);
        const float z1 = sample_volume<DIFFUS_SAMPLER_TRILINEAR, LAYOUT, true>(p.vol, rs.coord(0, k + 1), rs.coord(1, k + 1),
                                                                               rs.coord(2, k + 1), g1);
        if (!((z1 - z0) / (z0 + z1) == med)) continue;
        float t0[6], t1[6];
        sample_tangent(rs.d, g0, (float)k, t0);
        sample_tangent(rs.d, g1, (float)(k + 1), t1);
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

cudaError_t launch_gn_median_tangent(const RenderParams& p, int layout, const int32_t* tie_count, float* med_tan, cudaStream_t st) {
    DIFFUS_GN_LAYOUTS(gn_median_tangent_kernel<L_><<<(unsigned)p.n_poses, 32, 0, st>>>(p, tie_count, med_tan); return cudaGetLastError())
    return cudaErrorInvalidValue;
}

cudaError_t launch_render_gn(const RenderParams& p, int layout, const float* med_tan, float* partial, float* loss, float* jtr,
                             float* jtj, cudaStream_t st) {
    const int wpb = gn_warps_per_block(p.total_rays);
    const size_t smem = (size_t)wpb * GN_SMEM_PER_WARP * sizeof(float);
    const unsigned grid = (unsigned)((p.total_rays + wpb - 1) / wpb);
    cudaError_t e = cudaErrorInvalidValue;
    DIFFUS_GN_LAYOUTS(auto k = render_gn_kernel<L_>; e = ensure_smem(k, smem); if (e != cudaSuccess) return e;
                      k<<<grid, wpb * 32, smem, st>>>(p, med_tan, partial); e = cudaGetLastError(); break)
    if (e != cudaSuccess) return e;
    gn_reduce_kernel<<<(unsigned)p.n_poses, 128, 0, st>>>(partial, p.n_rays, loss, jtr, jtj);
    return cudaGetLastError();
}

#undef DIFFUS_GN_LAYOUTS

}  // namespace diffus
