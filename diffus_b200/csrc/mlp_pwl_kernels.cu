// The impedance MLP as the piecewise-linear function it is (sm_100a).
//
// ImpedanceEstimator (reference src/impedance.py:6-17) is Linear(1,32)-ReLU-Linear(32,32)-ReLU-Linear(32,1) applied to ONE
// scalar per voxel.  A ReLU network of a scalar input is a continuous piecewise-linear function of that scalar: between two
// consecutive points where some unit switches, every activation mask is fixed and
//         mlp(x) = P_r x + Q_r                                            (region r)
// The layer-1 units switch at x = -b1_i / w1_i (<= 32 points); inside each of the <= 33 intervals they leave, a layer-2
// pre-activation is affine, s_j(x) = p_j x + q_j, and switches at most once, at -q_j / p_j.  So there are at most
// 32 + 33 * 32 = 1088 breakpoints (55 - 75 for freshly initialised weights), and:
//   forward   out[v] = P_r x_v + Q_r with r found by a binary search over the sorted breakpoints: one pass over the volume at
//             HBM speed instead of 2 176 flop per voxel (no dense contraction is left for the tensor cores to do);
//   backward  d loss / d theta = sum_v g_v d mlp(x_v) / d theta, and inside a region d mlp / d theta is affine in x, so the
//             whole weight gradient follows from TWO moments per region, G0_r = sum g_v and G1_r = sum g_v x_v.  The pass
//             over the volume only bins (g, g x) by region; a second, tiny kernel assembles the 1 153 gradients per region.
// The table (breakpoints, masks at the region midpoints, P_r, Q_r) is built in float64 by every CTA in shared memory from
// the 1 153 parameters (a few microseconds), so the entry points stay stateless.  Against the float64 oracle this is MORE
// accurate than evaluating the layers in float32: the only rounding is the final P x + Q, and the difference of two
// impedances of the same region -- what a reflection coefficient is made of -- carries no layer rounding noise at all.
// A voxel within one float32 ulp of a breakpoint may be assigned to the neighbouring region; the function is continuous
// there, so values move by O(ulp) (the layered float32 evaluation has the same ambiguity in its ReLU gates).
// Weights with more than PWL_MAXR regions fall back to the layered evaluation (forward: inline; backward: the gated
// CUDA-core kernels of mlp_kernels.cu).
#include <math.h>

#include "common.cuh"
#include "launch.h"

namespace diffus {

namespace {

constexpr int HID = 32;
constexpr int OFF_W1 = 0, OFF_B1 = 32, OFF_W2 = 64, OFF_B2 = 64 + 1024, OFF_W3 = OFF_B2 + 32, OFF_B3 = OFF_W3 + 32;
constexpr int NP = DIFFUS_MLP_NPARAMS;
constexpr int PWL_MAXR = 256;                      // regions this path handles (binary search of 8 steps, 4 KB of bins per warp)
constexpr int PWL_MAXC = HID + (HID + 1) * HID;    // candidate breakpoints
constexpr int PWL_THREADS = 256, PWL_WARPS = PWL_THREADS / 32;
constexpr double DINF = __builtin_huge_val();

struct PwlTable {                    // what the voxel loops read
    double P[PWL_MAXR], Q[PWL_MAXR], xm[PWL_MAXR];     // per region: mlp(x) = P x + Q; midpoint (where the masks are taken)
    float bpf[PWL_MAXR];             // breakpoints as float32, +inf padded: the search array
    float prm[NP + 3];
    int n1, nbp, nreg, nsearch, count;
};
struct PwlScratch {                  // only while the table is built (the backward's bins reuse the space)
    double cand[PWL_MAXC];           // candidate breakpoints (+inf = none)
    double2 pq[(HID + 1) * HID];     // layer-2 pre-activations per layer-1 interval e and unit j: s_j(x) = pq[e][j].x x + pq[e][j].y
    double sorted1[HID];             // layer-1 breakpoints, ascending, +inf padded
    double bpd[PWL_MAXR];            // all breakpoints, ascending
    int unit1[HID];                  // the layer-1 unit that switches at sorted1[k]
};

__device__ __forceinline__ double pwl_mid(double a, double b) {
    const bool ia = !(a > -DINF), ib = !(b < DINF);
    if (ia && ib) return 0.0;
    if (ia) return b - 1.0 - fabs(b);
    if (ib) return a + 1.0 + fabs(a);
    return 0.5 * (a + b);
}

// layer-2 pre-activation of unit j as an affine function of x under the layer-1 mask taken at xm (direct evaluation)
__device__ __forceinline__ void pwl_affine(const float* prm, double xm, int j, double& p, double& q) {
    p = 0.0;
    q = (double)prm[OFF_B2 + j];
#pragma unroll 8
    for (int i = 0; i < HID; ++i) {
        const double w = (double)prm[OFF_W1 + i], b = (double)prm[OFF_B1 + i];
        if (w * xm + b > 0.0) {
            const double w2 = (double)prm[OFF_W2 + j * HID + i];
            p += w2 * w;
            q += w2 * b;
        }
    }
}

__device__ __forceinline__ double warp_sum_f64(double v) {
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) v += __shfl_xor_sync(FULL, v, d);
    return v;
}

// Every thread of the CTA takes part (blockDim.x >= 64).  On return S.nreg is the region count; if it exceeds PWL_MAXR
// nothing else is valid.  Cost: a few thousand warp instructions -- the layer-2 pre-activations are carried from one layer-1
// interval to the next (one unit switches at a time) instead of being re-evaluated per interval.
__device__ void pwl_build(PwlTable& S, PwlScratch& W, const float* __restrict__ params) {
    const int tid = threadIdx.x, nt = blockDim.x, warp = tid >> 5, lane = tid & 31, nw = nt >> 5;
    for (int i = tid; i < NP; i += nt) S.prm[i] = __ldg(params + i);
    if (tid == 0) S.count = 0;
    __syncthreads();
    if (tid < HID) {
        const double w = (double)S.prm[OFF_W1 + tid], b = (double)S.prm[OFF_B1 + tid];
        double t = (w != 0.0) ? -b / w : DINF;
        if (!(fabs(t) < DINF)) t = DINF;                 // NaN / infinite: the unit never switches
        W.cand[tid] = t;
    }
    __syncthreads();
    if (tid < HID) {                                     // rank sort of 32 (value, unit) pairs
        const double t = W.cand[tid];
        int rank = 0;
        for (int k = 0; k < HID; ++k) {
            const double u = W.cand[k];
            rank += (u < t) || (u == t && k < tid);
        }
        W.sorted1[rank] = t;
        W.unit1[rank] = tid;
        const unsigned fin = __ballot_sync(FULL, t < DINF);
        if (tid == 0) S.n1 = __popc(fin);
    }
    __syncthreads();
    const int n1 = S.n1;
    const int ncand = HID + (n1 + 1) * HID;
    if (warp == 0) {                                     // lane = layer-2 unit j; walk the layer-1 intervals left to right
        const int j = lane;
        double p = 0.0, q = (double)S.prm[OFF_B2 + j];
        for (int i = 0; i < HID; ++i) {                  // x -> -inf: unit i is on iff w1_i < 0 (or constant and positive)
            const double w = (double)S.prm[OFF_W1 + i], b = (double)S.prm[OFF_B1 + i];
            if (w < 0.0 || (w == 0.0 && b > 0.0)) {
                const double w2 = (double)S.prm[OFF_W2 + j * HID + i];
                p += w2 * w;
                q += w2 * b;
            }
        }
        for (int e = 0; e <= n1; ++e) {
            const double a = e == 0 ? -DINF : W.sorted1[e - 1], b = e == n1 ? DINF : W.sorted1[e];
            W.pq[e * HID + j] = make_double2(p, q);
            double r = DINF;
            if (a < b && p != 0.0) {
                const double t = -q / p;
                if (t > a && t < b) r = t;
            }
            W.cand[HID + e * HID + j] = r;
            if (e < n1) {                                // unit i switches at b: on if its slope is positive, off otherwise
                const int i = W.unit1[e];
                const double w = (double)S.prm[OFF_W1 + i], bb = (double)S.prm[OFF_B1 + i];
                const double w2 = (double)S.prm[OFF_W2 + j * HID + i];
                const double sg = w > 0.0 ? 1.0 : -1.0;
                p += sg * (w2 * w);
                q += sg * (w2 * bb);
            }
        }
    }
    __syncthreads();
    {
        int mine = 0;
        for (int k = tid; k < ncand; k += nt) mine += W.cand[k] < DINF;
        if (mine) atomicAdd(&S.count, mine);
    }
    __syncthreads();
    const int nbp = S.count;
    __syncthreads();
    if (tid == 0) {
        S.nbp = nbp;
        S.nreg = nbp + 1;
        S.count = 0;
        int ns = 1;
        while (ns < nbp + 1) ns <<= 1;
        S.nsearch = ns;
    }
    __syncthreads();
    if (nbp + 1 > PWL_MAXR) return;                      // (uniform) too many regions for this path
    for (int k = tid; k < ncand; k += nt) {              // compact (any order), then rank sort: S.P is scratch here
        const double c = W.cand[k];
        if (c < DINF) S.P[atomicAdd(&S.count, 1)] = c;
    }
    __syncthreads();
    for (int k = tid; k < nbp; k += nt) {
        const double c = S.P[k];
        int rank = 0;
        for (int m = 0; m < nbp; ++m) {
            const double u = S.P[m];
            rank += (u < c) || (u == c && m < k);
        }
        W.bpd[rank] = c;
    }
    __syncthreads();
    for (int k = tid; k < PWL_MAXR; k += nt) S.bpf[k] = k < nbp ? (float)W.bpd[k] : __int_as_float(0x7f800000);
    const double b3 = (double)S.prm[OFF_B3];
    const double t1 = W.sorted1[lane];
    for (int r = warp; r <= nbp; r += nw) {              // a warp per region, a lane per layer-2 unit: masks at the midpoint
        const double a = r == 0 ? -DINF : W.bpd[r - 1], b = r == nbp ? DINF : W.bpd[r];
        const double xm = pwl_mid(a, b);
        const int e = __popc(__ballot_sync(FULL, t1 <= xm));           // the layer-1 interval the midpoint lies in
        const double2 pq = W.pq[e * HID + lane];
        const bool on = pq.x * xm + pq.y > 0.0;
        const double w3 = (double)S.prm[OFF_W3 + lane];
        const double cp = warp_sum_f64(on ? w3 * pq.x : 0.0), cq = warp_sum_f64(on ? w3 * pq.y : 0.0);
        if (lane == 0) {
            S.P[r] = cp;
            S.Q[r] = cq + b3;
            S.xm[r] = xm;
        }
    }
    __syncthreads();
}

constexpr size_t PWL_TABLE_BYTES = (sizeof(PwlTable) + 15) & ~(size_t)15;
constexpr size_t PWL_BINS_BYTES = sizeof(double2) * PWL_WARPS * PWL_MAXR;
static_assert(sizeof(PwlScratch) <= PWL_BINS_BYTES, "the backward's bins reuse the build scratch");

// number of breakpoints <= x  (= region index); bpf is +inf padded up to nsearch - 1 entries
__device__ __forceinline__ int pwl_region(const float* bpf, int nsearch, float x) {
    int lo = 0;
    for (int s = nsearch >> 1; s > 0; s >>= 1) lo += (bpf[lo + s - 1] <= x) ? s : 0;
    return lo;
}

// the reference's own evaluation order in float32 (fallback when the weights have more than PWL_MAXR regions)
__device__ float mlp_layered(const float* prm, float x) {
    float h1[HID];
#pragma unroll
    for (int i = 0; i < HID; ++i) h1[i] = fmaxf(fmaf(prm[OFF_W1 + i], x, prm[OFF_B1 + i]), 0.f);
    float out = prm[OFF_B3];
    for (int j = 0; j < HID; ++j) {
        float s = prm[OFF_B2 + j];
#pragma unroll
        for (int i = 0; i < HID; ++i) s = fmaf(prm[OFF_W2 + j * HID + i], h1[i], s);
        out = fmaf(prm[OFF_W3 + j], fmaxf(s, 0.f), out);
    }
    return out;
}

__device__ __forceinline__ float pwl_eval(const PwlTable& S, int nsearch, float x) {
    const int r = pwl_region(S.bpf, nsearch, x);
    return (float)fma(S.P[r], (double)x, S.Q[r]);        // one rounding to float32 of the exact affine value
}

}  // namespace

__global__ void __launch_bounds__(PWL_THREADS) mlp_pwl_fwd_kernel(const float* __restrict__ params, const float* __restrict__ x,
                                                                 const uint8_t* __restrict__ mask, int64_t n, float out_scale,
                                                                 float fill, float* __restrict__ out) {
    extern __shared__ __align__(16) unsigned char pwl_smem[];
    PwlTable& S = *reinterpret_cast<PwlTable*>(pwl_smem);
    pwl_build(S, *reinterpret_cast<PwlScratch*>(pwl_smem + PWL_TABLE_BYTES), params);
    const int64_t gtid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x, gstride = (int64_t)gridDim.x * blockDim.x;
    if (S.nreg > PWL_MAXR) {
        for (int64_t i = gtid; i < n; i += gstride) out[i] = (mask && !mask[i]) ? fill : out_scale * mlp_layered(S.prm, __ldg(x + i));
        return;
    }
    const int nsearch = S.nsearch;
    const bool vec = ((((uintptr_t)x) | ((uintptr_t)out)) & 15u) == 0 && (!mask || (((uintptr_t)mask) & 3u) == 0);
    const int64_t n4 = vec ? n >> 2 : 0;
    // four 16-byte loads in flight per thread (one per trip left the stream at 1.1 TB/s: a DRAM round trip per 16 bytes per thread)
    constexpr int PF = 4;
    int64_t i0 = gtid;
    for (; i0 + (PF - 1) * gstride < n4; i0 += PF * gstride) {
        float4 xv[PF];
        uchar4 mv[PF];
#pragma unroll
        for (int u = 0; u < PF; ++u) {
            xv[u] = __ldg((const float4*)x + i0 + u * gstride);
            if (mask) mv[u] = __ldg((const uchar4*)mask + i0 + u * gstride);
        }
#pragma unroll
        for (int u = 0; u < PF; ++u) {
            float4 o;
            o.x = out_scale * pwl_eval(S, nsearch, xv[u].x);
            o.y = out_scale * pwl_eval(S, nsearch, xv[u].y);
            o.z = out_scale * pwl_eval(S, nsearch, xv[u].z);
            o.w = out_scale * pwl_eval(S, nsearch, xv[u].w);
            if (mask) {
                if (!mv[u].x) o.x = fill;
                if (!mv[u].y) o.y = fill;
                if (!mv[u].z) o.z = fill;
                if (!mv[u].w) o.w = fill;
            }
            ((float4*)out)[i0 + u * gstride] = o;
        }
    }
    for (int64_t i = i0; i < n4; i += gstride) {
        const float4 xv = __ldg((const float4*)x + i);
        float4 o;
        o.x = out_scale * pwl_eval(S, nsearch, xv.x);
        o.y = out_scale * pwl_eval(S, nsearch, xv.y);
        o.z = out_scale * pwl_eval(S, nsearch, xv.z);
        o.w = out_scale * pwl_eval(S, nsearch, xv.w);
        if (mask) {
            const uchar4 m = __ldg((const uchar4*)mask + i);
            if (!m.x) o.x = fill;
            if (!m.y) o.y = fill;
            if (!m.z) o.z = fill;
            if (!m.w) o.w = fill;
        }
        ((float4*)out)[i] = o;
    }
    for (int64_t i = (n4 << 2) + gtid; i < n; i += gstride)
        out[i] = (mask && !mask[i]) ? fill : out_scale * pwl_eval(S, nsearch, __ldg(x + i));
}

// d out / d x: the slope of the region (the input gradient nn.Sequential gives the reference's callers)
__global__ void __launch_bounds__(PWL_THREADS) mlp_pwl_dx_kernel(const float* __restrict__ params, const float* __restrict__ x,
                                                                const uint8_t* __restrict__ mask, const float* __restrict__ grad_out,
                                                                int64_t n, float out_scale, float* __restrict__ grad_x) {
    extern __shared__ __align__(16) unsigned char pwl_smem[];
    PwlTable& S = *reinterpret_cast<PwlTable*>(pwl_smem);
    pwl_build(S, *reinterpret_cast<PwlScratch*>(pwl_smem + PWL_TABLE_BYTES), params);
    const int64_t gtid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x, gstride = (int64_t)gridDim.x * blockDim.x;
    const bool table = S.nreg <= PWL_MAXR;
    const int nsearch = S.nsearch;
    for (int64_t i = gtid; i < n; i += gstride) {
        const float xv = __ldg(x + i);
        float slope;
        if (table) {
            slope = (float)S.P[pwl_region(S.bpf, nsearch, xv)];
        } else {                                             // layered: sum_j w3_j [s_j > 0] sum_i W2[j][i] [h1_i > 0] w1_i
            const float* prm = S.prm;
            float h1[HID];
#pragma unroll
            for (int k = 0; k < HID; ++k) h1[k] = fmaf(prm[OFF_W1 + k], xv, prm[OFF_B1 + k]);
            slope = 0.f;
            for (int j = 0; j < HID; ++j) {
                float sj = prm[OFF_B2 + j], dj = 0.f;
#pragma unroll
                for (int k = 0; k < HID; ++k) {
                    const float w2 = prm[OFF_W2 + j * HID + k];
                    sj = fmaf(w2, fmaxf(h1[k], 0.f), sj);
                    dj = h1[k] > 0.f ? fmaf(w2, prm[OFF_W1 + k], dj) : dj;
                }
                if (sj > 0.f) slope = fmaf(prm[OFF_W3 + j], dj, slope);
            }
        }
        grad_x[i] = (mask && !mask[i]) ? 0.f : __ldg(grad_out + i) * out_scale * slope;
    }
}

// ---------------------------------------------------------------------------------------------------------------------
// backward
// workspace (8-byte aligned): [hdr: 4 x int32 {nreg, overflow, -, -}] [xm: PWL_MAXR doubles]
//                             [partial: blocks x PWL_MAXR x 2 doubles] [scratch: PWL_MAXR x NP doubles]
//                             [dense fallback: its block partials, floats]
// ---------------------------------------------------------------------------------------------------------------------
namespace {

// Adds (g, g x) of the warp's voxels (up to four per lane) to the warp's bins: one pair of warp reductions per DISTINCT
// region among them (neighbouring voxels are mostly the same tissue), the bin itself in float64 with a single writer --
// no atomics, run-to-run identical.
__device__ __forceinline__ void pwl_accumulate4(double2* wb, const int r[4], const float g[4], const float x[4], int lane) {
    unsigned pend = (g[0] != 0.f ? 1u : 0u) | (g[1] != 0.f ? 2u : 0u) | (g[2] != 0.f ? 4u : 0u) | (g[3] != 0.f ? 8u : 0u);
    const float gx[4] = {g[0] * x[0], g[1] * x[1], g[2] * x[2], g[3] * x[3]};
    for (;;) {
        const unsigned todo = __ballot_sync(FULL, pend != 0u);
        if (!todo) break;
        const int leader = __ffs(todo) - 1;
        const int mine = (pend & 1u) ? r[0] : (pend & 2u) ? r[1] : (pend & 4u) ? r[2] : r[3];
        const int rr = __shfl_sync(FULL, mine, leader);
        float s0 = 0.f, s1 = 0.f;
#pragma unroll
        for (int k = 0; k < 4; ++k)
            if (((pend >> k) & 1u) && r[k] == rr) {
                s0 += g[k];
                s1 += gx[k];
                pend &= ~(1u << k);
            }
        s0 = warp_sum(s0);
        s1 = warp_sum(s1);
        if (lane == 0) {
            double2 b = wb[rr];
            b.x += (double)s0;
            b.y += (double)s1;
            wb[rr] = b;
        }
    }
}

}  // namespace

__global__ void __launch_bounds__(PWL_THREADS) mlp_pwl_bwd_kernel(const float* __restrict__ params, const float* __restrict__ x,
                                                                 const uint8_t* __restrict__ mask,
                                                                 const float* __restrict__ grad_out, int64_t n, float out_scale,
                                                                 int* __restrict__ hdr, double* __restrict__ ws_xm,
                                                                 double* __restrict__ partial) {
    extern __shared__ __align__(16) unsigned char pwl_smem[];
    PwlTable& S = *reinterpret_cast<PwlTable*>(pwl_smem);
    double2* bins = reinterpret_cast<double2*>(pwl_smem + PWL_TABLE_BYTES);     // [PWL_WARPS][PWL_MAXR], after the build scratch is dead
    pwl_build(S, *reinterpret_cast<PwlScratch*>(pwl_smem + PWL_TABLE_BYTES), params);
    __syncthreads();
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    if (blockIdx.x == 0 && tid == 0) {
        hdr[0] = S.nreg;
        hdr[1] = S.nreg > PWL_MAXR;
    }
    if (S.nreg > PWL_MAXR) return;
    const int nreg = S.nreg, nsearch = S.nsearch;
    if (blockIdx.x == 0)
        for (int r = tid; r < nreg; r += blockDim.x) ws_xm[r] = S.xm[r];
    for (int k = tid; k < PWL_WARPS * PWL_MAXR; k += blockDim.x) bins[k] = make_double2(0.0, 0.0);
    __syncthreads();
    double2* wb = bins + warp * PWL_MAXR;
    const bool vec = ((((uintptr_t)x) | ((uintptr_t)grad_out)) & 15u) == 0 && (!mask || (((uintptr_t)mask) & 3u) == 0);
    const int64_t n4 = vec ? n >> 2 : 0;
    const int64_t wstride = (int64_t)gridDim.x * blockDim.x;
    // the loads of the next trip are issued before this trip's voxels are binned (the binning is a chain of warp votes and
    // reductions: with one trip in flight the stream ran at 0.75 TB/s)
    auto fetch = [&](int64_t i, float4& xv, float4& gv) {
        xv = make_float4(0.f, 0.f, 0.f, 0.f);
        gv = xv;
        if (i < n4) {
            xv = __ldg((const float4*)x + i);
            gv = __ldg((const float4*)grad_out + i);
            if (mask) {
                const uchar4 m = __ldg((const uchar4*)mask + i);
                if (!m.x) gv.x = 0.f;
                if (!m.y) gv.y = 0.f;
                if (!m.z) gv.z = 0.f;
                if (!m.w) gv.w = 0.f;
            }
        }
    };
    float4 xn, gn;
    fetch((int64_t)blockIdx.x * blockDim.x + warp * 32 + lane, xn, gn);
    for (int64_t base = (int64_t)blockIdx.x * blockDim.x + warp * 32; base < n4; base += wstride) {      // warp-uniform trip count
        const float4 xv = xn, gv = gn;
        fetch(base + wstride + lane, xn, gn);
        if (!__any_sync(FULL, gv.x != 0.f || gv.y != 0.f || gv.z != 0.f || gv.w != 0.f)) continue;      // voxels no ray touched
        const int r[4] = {pwl_region(S.bpf, nsearch, xv.x), pwl_region(S.bpf, nsearch, xv.y), pwl_region(S.bpf, nsearch, xv.z),
                          pwl_region(S.bpf, nsearch, xv.w)};
        const float g[4] = {gv.x * out_scale, gv.y * out_scale, gv.z * out_scale, gv.w * out_scale};
        const float xs[4] = {xv.x, xv.y, xv.z, xv.w};
        pwl_accumulate4(wb, r, g, xs, lane);
    }
    for (int64_t base = (n4 << 2) + (int64_t)blockIdx.x * blockDim.x + warp * 32; base < n; base += wstride) {   // scalar tail / unaligned
        const int64_t i = base + lane;
        float xs[4] = {0.f, 0.f, 0.f, 0.f}, g[4] = {0.f, 0.f, 0.f, 0.f};
        if (i < n) {
            xs[0] = __ldg(x + i);
            g[0] = (mask && !mask[i]) ? 0.f : __ldg(grad_out + i) * out_scale;
        }
        const int r[4] = {pwl_region(S.bpf, nsearch, xs[0]), 0, 0, 0};
        pwl_accumulate4(wb, r, g, xs, lane);
    }
    __syncthreads();
    double* dst = partial + (int64_t)blockIdx.x * PWL_MAXR * 2;
    for (int r = tid; r < nreg; r += blockDim.x) {        // the CTA's warps, in fixed order
        double s0 = 0.0, s1 = 0.0;
#pragma unroll
        for (int w = 0; w < PWL_WARPS; ++w) {
            s0 += bins[w * PWL_MAXR + r].x;
            s1 += bins[w * PWL_MAXR + r].y;
        }
        dst[2 * r] = s0;
        dst[2 * r + 1] = s1;
    }
}

// one CTA per region: its two moments (blocks summed in a fixed order) -> its contribution to each of the 1 153 gradients
__global__ void __launch_bounds__(128) mlp_pwl_assemble_kernel(const float* __restrict__ params, const int* __restrict__ hdr,
                                                              const double* __restrict__ ws_xm, const double* __restrict__ partial,
                                                              int nblocks, double* __restrict__ scratch) {
    const int r = blockIdx.x, tid = threadIdx.x;
    if (hdr[1] || r >= hdr[0]) return;
    __shared__ double red0[128], red1[128], sp[HID], sq[HID], su[HID];
    __shared__ int m1s[HID], m2s[HID];
    __shared__ float prm[NP];
    for (int i = tid; i < NP; i += 128) prm[i] = __ldg(params + i);
    double a0 = 0.0, a1 = 0.0;
    for (int b = tid; b < nblocks; b += 128) {
        a0 += partial[((int64_t)b * PWL_MAXR + r) * 2];
        a1 += partial[((int64_t)b * PWL_MAXR + r) * 2 + 1];
    }
    red0[tid] = a0;
    red1[tid] = a1;
    __syncthreads();
    for (int s = 64; s > 0; s >>= 1) {
        if (tid < s) {
            red0[tid] += red0[tid + s];
            red1[tid] += red1[tid + s];
        }
        __syncthreads();
    }
    const double G0 = red0[0], G1 = red1[0], xm = ws_xm[r];
    if (tid < HID) {
        m1s[tid] = (double)prm[OFF_W1 + tid] * xm + (double)prm[OFF_B1 + tid] > 0.0;
        double p, q;
        pwl_affine(prm, xm, tid, p, q);
        sp[tid] = p;
        sq[tid] = q;
        m2s[tid] = p * xm + q > 0.0;
    }
    __syncthreads();
    if (tid < HID) {                                      // d out / d h1_i under both masks
        double u = 0.0;
        for (int j = 0; j < HID; ++j)
            if (m2s[j]) u += (double)prm[OFF_W2 + j * HID + tid] * (double)prm[OFF_W3 + j];
        su[tid] = m1s[tid] ? u : 0.0;
    }
    __syncthreads();
    for (int k = tid; k < NP; k += 128) {
        double c;
        if (k < OFF_B1) c = su[k] * G1;                                                    // d W1_i = sum g dh1_i x
        else if (k < OFF_W2) c = su[k - OFF_B1] * G0;                                      // d b1_i
        else if (k < OFF_B2) {
            const int j = (k - OFF_W2) / HID, i = (k - OFF_W2) % HID;                      // d W2[j][i] = w3_j sum g h1_i
            c = (m2s[j] && m1s[i]) ? (double)prm[OFF_W3 + j] * ((double)prm[OFF_W1 + i] * G1 + (double)prm[OFF_B1 + i] * G0) : 0.0;
        } else if (k < OFF_W3) c = m2s[k - OFF_B2] ? (double)prm[OFF_W3 + (k - OFF_B2)] * G0 : 0.0;          // d b2_j
        else if (k < OFF_B3) c = m2s[k - OFF_W3] ? sp[k - OFF_W3] * G1 + sq[k - OFF_W3] * G0 : 0.0;          // d W3_j = sum g h2_j
        else c = G0;                                                                       // d b3
        scratch[(int64_t)r * NP + k] = c;
    }
}

__global__ void mlp_pwl_finish_kernel(const int* __restrict__ hdr, const double* __restrict__ scratch, float* __restrict__ grad_params) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= NP || hdr[1]) return;
    const int nreg = hdr[0];
    double s = 0.0;
#pragma unroll 8
    for (int r = 0; r < nreg; ++r) s += scratch[(int64_t)r * NP + k];      // regions in index order: run-to-run identical
    grad_params[k] += (float)s;
}

static size_t pwl_fwd_smem() { return PWL_TABLE_BYTES + sizeof(PwlScratch); }
static size_t pwl_bwd_smem() { return PWL_TABLE_BYTES + PWL_BINS_BYTES; }
static int pwl_blocks(int64_t n) {
    const int64_t want = (n / 4 + PWL_THREADS - 1) / PWL_THREADS;
    return (int)max((int64_t)1, min(want, (int64_t)148 * 4));
}
static constexpr int64_t PWL_HDR_BYTES = 16;

int64_t mlp_pwl_bwd_workspace_bytes(int64_t n) {
    return PWL_HDR_BYTES + (int64_t)sizeof(double) * (PWL_MAXR + (int64_t)pwl_blocks(n) * PWL_MAXR * 2 + (int64_t)PWL_MAXR * NP);
}

cudaError_t launch_mlp_pwl_fwd(const float* params, const float* x, const uint8_t* mask, int64_t n, float out_scale, float fill,
                               float* out, cudaStream_t st) {
    const size_t smem = pwl_fwd_smem();
    cudaError_t e = cudaFuncSetAttribute(mlp_pwl_fwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    return launch_kernel(mlp_pwl_fwd_kernel, pwl_blocks(n), PWL_THREADS, smem, st, params, x, mask, n, out_scale, fill, out);
}

cudaError_t launch_mlp_pwl_dx(const float* params, const float* x, const uint8_t* mask, const float* grad_out, int64_t n,
                              float out_scale, float* grad_x, cudaStream_t st) {
    const size_t smem = pwl_fwd_smem();
    cudaError_t e = cudaFuncSetAttribute(mlp_pwl_dx_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    const int64_t want = (n + PWL_THREADS - 1) / PWL_THREADS;
    return launch_kernel(mlp_pwl_dx_kernel, (unsigned)max((int64_t)1, min(want, (int64_t)148 * 4)), PWL_THREADS, smem, st, params, x, mask, grad_out, n,
                                                                                                      out_scale, grad_x);
}

// `workspace` holds mlp_pwl_bwd_workspace_bytes(n) bytes followed by the dense fallback's block partials
cudaError_t launch_mlp_pwl_bwd(const float* params, const float* x, const uint8_t* mask, const float* grad_out, int64_t n,
                               float out_scale, float* grad_params, void* workspace, cudaStream_t st) {
    const size_t smem = pwl_bwd_smem();
    cudaError_t e = cudaFuncSetAttribute(mlp_pwl_bwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    const int blocks = pwl_blocks(n);
    int* hdr = (int*)workspace;
    double* ws_xm = (double*)((char*)workspace + PWL_HDR_BYTES);
    double* partial = ws_xm + PWL_MAXR;
    double* scratch = partial + (int64_t)blocks * PWL_MAXR * 2;
    e = launch_kernel(mlp_pwl_bwd_kernel, blocks, PWL_THREADS, smem, st, params, x, mask, grad_out, n, out_scale, hdr, ws_xm, partial);
    if (e != cudaSuccess) return e;
    e = launch_kernel(mlp_pwl_assemble_kernel, PWL_MAXR, 128, 0, st, params, hdr, ws_xm, partial, blocks, scratch);
    if (e != cudaSuccess) return e;
    e = launch_kernel(mlp_pwl_finish_kernel, (NP + 127) / 128, 128, 0, st, hdr, scratch, grad_params);
    if (e != cudaSuccess) return e;
    // more than PWL_MAXR regions: the layered CUDA-core kernels run instead (they return at once when hdr[1] == 0)
    void* dense_ws = (char*)workspace + mlp_pwl_bwd_workspace_bytes(n);
    return launch_mlp_bwd(params, x, mask, grad_out, n, out_scale, grad_params, dense_ws, hdr + 1, st);
}

}  // namespace diffus
