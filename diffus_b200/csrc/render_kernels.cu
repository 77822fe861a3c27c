// Fused per-ray march, forward and backward (sm_100a).  See common.cuh for the layout.
//
// forward  : replaces plot_beam_frame's numeric core (reference src/renderer.py:201-275)
// backward : what torch autograd derives from it (SURVEY.md 3.2), written as a reverse
//            affine scan of 2x2 matrices; per-ray gradient partials are written once
//            (no atomics) and only the volume gradient uses red.global.add.f32, mirroring
//            index_put_(accumulate=True).  With a target frame the backward kernel also
//            evaluates the forward and the MSE loss itself, so one launch is a whole
//            pose-recovery step (fused forward + loss + backward, one gather pass).
#include <cuda_pipeline.h>

#include <type_traits>

#include "common.cuh"
#include "launch.h"

namespace diffus {

// ---------------------------------------------------------------------------------------
// chunk-phase building blocks shared by the render and the echo-only kernels
// ---------------------------------------------------------------------------------------

// exclusive prefix of the lanes' chunk products, left-multiplied by the segment carry
__device__ __forceinline__ M2 warp_exclusive_prefix(const M2& chunk_total, const M2& carry, int lane) {
    M2 inc = chunk_total;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        M2 left = m2_shfl_up(inc, d);
        if (lane >= d) inc = m2_mul(left, inc);
    }
    M2 exc = m2_shfl_up(inc, 1);
    if (lane == 0) exc = m2_identity();
    return m2_mul(carry, exc);
}

// Forward chunk phase for one segment.  `r[i]` must hold the coefficient of column
// c0 + lane*CH + i (0 for columns that do not exist).  Writes echo (NaN -> 0) to obuf and
// returns the updated carry (prefix through the last column of the segment).
template <class G>
__device__ __forceinline__ M2 forward_chunk(const float r[G::CHUNK], M2 carry, float* obuf, int lane) {
    M2 T = m2_identity();
#pragma unroll
    for (int i = 0; i < G::CHUNK; ++i) T = m2_mul_interface(T, r[i]);
    M2 P = warp_exclusive_prefix(T, carry, lane);
#pragma unroll
    for (int i = 0; i < G::CHUNK; ++i) {
        P = m2_mul_interface(P, r[i]);
        obuf[G::pad(lane * G::CHUNK) + i] = nan_to_num(echo_of(P.b(), fast_rcp(P.d())));   // i < CHUNK stays inside one 32-column block
    }
    return m2_shfl(P, 31);
}

// What the upstream gradient of a column is made of.
//   LOSS_GRAD : gbuf holds d loss / d frame                               -> ebar = g * att
//   LOSS_MSE  : gbuf holds the target frame; the kernel forms frame = echo * att,
//               diff = frame - target, ebar = grad_scale * diff * att, accumulates diff^2
//               and (optionally) stores the frame
constexpr int LOSS_GRAD = 0, LOSS_MSE = 1;
constexpr int WIDE_CTAS = 4;     // resident 4-warp CTA equivalents per SM of the WIDE kernels (4: 128 registers, 5: 96 and spills)
constexpr int FWD_GB = 1;        // tiles per gather batch of the forward kernel (trilinear)
constexpr int TEX_GB = 2;        // tiles of tld4 gathers in flight per warp in the fused backward (TEXTURE layout)
constexpr int TEX_GB_WIDE = 4;   // the same in the WIDE kernels (128 registers; the multi-pass kernel spills 620 bytes with 4: config 5 14.4 -> 15.8 ms)
constexpr int BWD_DZ_STRIDE = FwdGeo::OBUF;   // floats between the per-axis rows of the spatial-gradient buffer

// What the render kernels add to the plain echo backward: the impedances around the lane's columns, so that the
// reverse sweep goes all the way to d loss / d Z per column and (pose gradient) to the lane's share of
// d loss / d source and d loss / d direction -- no separate pass over the columns afterwards.
struct ZTail {
    const float* zbuf;     // padded; slot s = impedance of the sample before pass-column s
    const float* dz;       // padded rows (BWD_DZ floats per axis): spatial gradient of Z per pass-column
    int lane_col;          // first pass-column of this lane's chunk
    float kbase;           // sample index of that column
    unsigned skip_mask;    // bit i: column i has no direct Z dependence (column 0, or the median-replaced one)
    float* rbar1;          // if not null, lane 0 stores rbar of its column 1 there (the median's gradient)
    float w_after;         // weight w of the column after the segment's last one (later segment / pass), 0 if none
    float w_first;         // out: w of the segment's first column (all lanes)
    float2 acc[3];         // per axis: (d loss / d source, d loss / d direction) partial sums of this lane
    float* xch;            // COOP: the CTA's exchange area (CoopXch), else unused
};

// COOP (rays of two to four passes, one pass per warp of the CTA -- see render_bwd_kernel): what the warps of a ray tell each
// other through shared memory, in floats from the start of the exchange area
struct CoopXch {
    static constexpr int TOTAL = 0;      // [4][4] transfer product of each pass
    static constexpr int MAP_A = 16;     // [4][4] \ the pass's reverse sweep as the affine map
    static constexpr int MAP_B = 32;     // [4][4] /  V -> V A + B of the adjoint entering it
    static constexpr int W_FIRST = 48;   // [4]    weight w of each pass's first column
    static constexpr int OUT = 52;       // [4][8] per-pass partial sums of the pose gradient and the loss
    static constexpr int FLOATS = 96;
};
__device__ __forceinline__ void xch_store(float* x, const M2& m) { x[0] = m.a(); x[1] = m.b(); x[2] = m.c(); x[3] = m.d(); }
__device__ __forceinline__ M2 xch_load(const float* x) { return m2_make(x[0], x[1], x[2], x[3]); }

// Backward chunk phase for one segment.
//   r[i]        coefficient of column c0 + lane*CH + i (0 where the column does not exist)
//   gbuf        see above; on return gbuf holds d loss / d r per column (ZMODE: d loss / d Z when STORE_ZBAR)
//   att_lane    attenuation of this lane's columns (padded table), or null for 1
//   frame_lane  where this lane's columns of the frame go (global), or null
//   zt          ZMODE only.  With w_c = 2 rbar_c / (Z_{c-1} + Z_c)^2 (0 for skipped / missing columns),
//               d loss / d Z_c = w_c Z_{c-1} - w_{c+1} Z_{c+1}; the lane's last column takes w_{c+1} from the
//               next lane (one shuffle after the sweep)
//   carry       forward prefix P through the column before the segment
//   vin         adjoint flowing into the segment's last column from later segments
//   ncol_lane   number of existing columns in this lane's chunk (may be <= 0 or > CHUNK)
// returns the adjoint flowing out of the segment's first column (into the previous segment)
//   COOP       the segment is one of the passes of a ray, each walked by one warp of the CTA (ZMODE only): `vin` is
//               ignored -- the passes exchange their affine maps (and, for the last column's d loss / d Z, the weight of the
//               next pass's first column) through zt->xch.  Every warp of the CTA must run the SAME instantiation:
//               the function holds two __syncthreads().
template <class G_, int LOSS, bool ZMODE = false, bool POSE_GRAD = false, bool STORE_ZBAR = false, bool FULL = false,
          bool COOP = false>
__device__ __forceinline__ M2 backward_chunk(const float r[G_::CHUNK], const M2& carry, const M2& vin, float* gbuf,
                                             const float* att_lane, float* frame_lane, float grad_scale, int ncol_lane,
                                             float& loss_acc, int lane, ZTail* zt = nullptr,
                                             const M2* known_total = nullptr, const M2* known_prefix = nullptr,
                                             const float* att_scale = nullptr) {
    constexpr int CHUNK = G_::CHUNK;
    static_assert(!COOP || ZMODE, "COOP: render kernels only");
    const int base = G_::pad(lane * CHUNK);        // columns lane*CHUNK .. +CHUNK-1 share a 32-column block
    // chunk product and exclusive prefix: reuse them when the caller already ran this sweep (prefix pass)
    M2 T, P;
    if (known_total) {
        T = *known_total;
        P = *known_prefix;
    } else {
        T = m2_identity();
#pragma unroll
        for (int i = 0; i < CHUNK; ++i) T = m2_mul_interface(T, r[i]);
        P = warp_exclusive_prefix(T, carry, lane);
    }
    constexpr int CK = G_::CKPT;   // a checkpoint every CK columns, the prefixes in between are recomputed
    M2 Pck[CHUNK / CK];            // true prefix BEFORE column CK*j of the chunk
    M2 G = m2_identity();          // local inclusive prefix
    M2 B = m2_zero();
#pragma unroll
    for (int i = 0; i < CHUNK; ++i) {
        if (i % CK == 0) Pck[i / CK] = P;
        P = m2_mul_interface(P, r[i]);
        G = m2_mul_interface(G, r[i]);
        float inv = fast_rcp(P.d());
        float e = echo_of(P.b(), inv);
        bool finite = fabsf(e) <= FLT_MAX;             // nan_to_num passes no gradient at NaN/inf
        float ge;
        const float att = att_lane ? (att_scale ? __fmul_rn(att_lane[i], *att_scale) : att_lane[i]) : 1.f;     // (scale: see render_bwd_kernel)
        if (LOSS == LOSS_MSE) {
            float fr = __fmul_rn(nan_to_num(e), att);
            float diff = fr - gbuf[base + i];
            if (FULL || i < ncol_lane) {
                loss_acc += diff * diff;
                if (frame_lane) frame_lane[i] = fr;      // 8 consecutive floats per lane: whole 32-byte sectors
            }
            ge = grad_scale * diff * att;
        } else {
            ge = gbuf[base + i] * att;
        }
        if (!finite || (!FULL && i >= ncol_lane)) ge = 0.f;   // columns that do not exist: the table beyond Sout is not filled
        gbuf[base + i] = ge;
        const float2 dcol = make_float2(ge * inv, -ge * e * inv);   // D = [[0, da], [0, db]];  B += D G^T
        B.c0 = __ffma2_rn(dcol, bcast(G.b()), B.c0);
        B.c1 = __ffma2_rn(dcol, bcast(G.d()), B.c1);
    }
    // suffix scan of the affine maps X -> X * A + B, A = T^T
    M2 As = m2_transpose(T), Bs = B;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        M2 An = m2_shfl_down(As, d), Bn = m2_shfl_down(Bs, d);
        if (lane + d < 32) {
            Bs = m2_add(m2_mul(Bn, As), Bs);
            As = m2_mul(An, As);
        }
    }
    // adjoint entering this lane's last column: maps of lanes lane+1..31 applied to vin
    M2 An = m2_shfl_down(As, 1), Bn = m2_shfl_down(Bs, 1);
    M2 vin_ = vin;
    if (COOP) {                                        // lane 0 holds the whole pass's map: publish it, then fold the later passes' maps
        const int w = threadIdx.x >> 5;
        if (lane == 0) {
            xch_store(zt->xch + CoopXch::MAP_A + 4 * w, As);
            xch_store(zt->xch + CoopXch::MAP_B + 4 * w, Bs);
        }
        __syncthreads();
        vin_ = m2_zero();
        for (int u = (int)(blockDim.x >> 5) - 1; u > w; --u)
            vin_ = m2_add(m2_mul(vin_, xch_load(zt->xch + CoopXch::MAP_A + 4 * u)), xch_load(zt->xch + CoopXch::MAP_B + 4 * u));
    }
    M2 V = (lane == 31) ? vin_ : m2_add(m2_mul(vin_, An), Bn);
    M2 vout = m2_add(m2_mul(vin_, As), Bs);            // valid on lane 0
    // ZMODE state: impedances of the samples at columns c+1, c (slot s = sample of column s-1) and the last weight
    const float* zl = nullptr;
    const float* dzl = nullptr;
    float z_hh = 0.f, z_hi = 0.f, w_prev = 0.f, part_last = 0.f, z_after = 0.f;
    if (ZMODE) {
        zl = zt->zbuf + G_::pad(zt->lane_col);          // slots lane_col .. lane_col+CHUNK-1: one 32-column block
        if (POSE_GRAD) dzl = zt->dz + G_::pad(zt->lane_col);
        z_hi = zt->zbuf[G_::pad(zt->lane_col + CHUNK)];
        z_hh = zt->zbuf[G_::pad(zt->lane_col + CHUNK + 1)];
        z_after = z_hh;
    }
    // one column's d loss / d Z: stored for the volume scatter and / or folded into the pose accumulators
    auto emit = [&](int i, float zbar) {
        if (!(zbar == zbar) || (!FULL && i >= ncol_lane)) zbar = 0.f;
        if (STORE_ZBAR) gbuf[base + i] = zbar;
        if (POSE_GRAD) {                                  // (d/dsource, d/ddirection) += zbar dZ/dp (1, k), one packed FMA per axis
            const float2 one_k = make_float2(1.f, zt->kbase + (float)i);
#pragma unroll
            for (int a = 0; a < 3; ++a)                   // the gather zero-fills dz where the pass has no sample
                zt->acc[a] = __ffma2_rn(bcast(zbar * dzl[a * BWD_DZ_STRIDE + i]), one_k, zt->acc[a]);
        }
    };
#pragma unroll
    for (int i = CHUNK - 1; i >= 0; --i) {
        M2 Q = Pck[i / CK];                            // prefix before column i
#pragma unroll
        for (int m = 0; m < i % CK; ++m) Q = m2_mul_interface(Q, r[i - i % CK + m]);
        const float2 pc1 = __ffma2_rn(Q.c0, bcast(r[i]), Q.c1);      // (b, d) of the prefix through column i
        float inv = fast_rcp(pc1.y);
        float e = echo_of(pc1.x, inv);
        float ge = gbuf[base + i];
        M2 Pbar = V;
        Pbar.c1 = __fadd2_rn(Pbar.c1, make_float2(ge * inv, -ge * e * inv));
        const float2 t0 = __fmul2_rn(Q.c0, Pbar.c0), t1 = __fmul2_rn(Q.c0, Pbar.c1), t2 = __fmul2_rn(Q.c1, Pbar.c0);
        float ma = t0.x + t0.y;          // Mbar = Q^T Pbar
        float mb = t1.x + t1.y;
        float mc = t2.x + t2.y;
        float rbar = -4.f * r[i] * ma + mb - mc;
        rbar = (rbar == rbar) ? rbar : 0.f;
        if (ZMODE) {
            if (zt->rbar1 && i == 1 && lane == 0) *zt->rbar1 = rbar;
            float z_lo = zl[i];
            float sum = z_lo + z_hi;
            float w = 2.f * rbar * fast_rcp(sum * sum);
            if ((!FULL && i >= ncol_lane) || ((zt->skip_mask >> i) & 1u)) w = 0.f;
            if (i == CHUNK - 1) part_last = w * z_lo;                  // its w_{c+1} lives in the next lane
            else emit(i, w * z_lo - w_prev * z_hh);
            z_hh = z_hi;
            z_hi = z_lo;
            w_prev = w;
        } else {
            gbuf[base + i] = rbar;
        }
        V = m2_mul_interface_t(Pbar, r[i]);
    }
    if (ZMODE) {
        float w_next = __shfl_down_sync(FULL, w_prev, 1);
        zt->w_first = __shfl_sync(FULL, w_prev, 0);
        if (COOP) {                                    // the column after this pass's last one belongs to the next warp
            const int w = threadIdx.x >> 5;
            if (lane == 0) zt->xch[CoopXch::W_FIRST + w] = zt->w_first;
            __syncthreads();
            if (lane == 31) w_next = w + 1 < (int)(blockDim.x >> 5) ? zt->xch[CoopXch::W_FIRST + w + 1] : 0.f;
        } else if (lane == 31) {
            w_next = zt->w_after;
        }
        emit(CHUNK - 1, part_last - w_next * z_after);
    }
    return m2_shfl(vout, 0);
}

// The target / upstream-gradient rows are read exactly once: mark them evict-first in L2 so that the
// stream does not push the (re-used) impedance and gradient volumes out of the 126 MB L2.
__device__ __forceinline__ uint64_t l2_evict_first_policy() {
    uint64_t pol;
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
    return pol;
}
__device__ __forceinline__ void cp_async_stream4(float* smem_dst, const float* gmem_src, uint64_t policy) {
    asm volatile("cp.async.ca.shared.global.L2::cache_hint [%0], [%1], 4, %2;" ::"r"((uint32_t)__cvta_generic_to_shared(smem_dst)),
                 "l"(gmem_src), "l"(policy)
                 : "memory");
}

// ray -> pose: a 32-bit division whenever the batch allows it (the 64-bit one is ~25 instructions of set-up per ray)
__device__ __forceinline__ int64_t pose_of_ray(int64_t ray, const RenderParams& p) {
    if (p.total_rays <= 0xffffffffLL) return (int64_t)((uint32_t)ray / (uint32_t)p.n_rays);
    return ray / p.n_rays;
}

// coefficient of the interface owned by column c from the two impedances around it
__device__ __forceinline__ float reflection(float z_prev, float z_cur) {
    return __fmul_rn(__fsub_rn(z_cur, z_prev), fast_rcp(__fadd_rn(z_prev, z_cur)));
}

// attenuation table exp(-alpha c), c = 0..Sout-1, shared by the rays of a CTA
__device__ __forceinline__ void fill_attenuation(float* att, int Sout, float alpha) {
    for (int c = threadIdx.x; c < Sout; c += blockDim.x) att[c] = expf(-alpha * (float)c);
    __syncthreads();
}

template <class G>
__device__ __forceinline__ void fill_attenuation_padded(float* att, int Sout, float alpha) {
    for (int c = threadIdx.x; c < Sout; c += blockDim.x) att[G::pad(c)] = expf(-alpha * (float)c);
    __syncthreads();
}

// lane's CH reflection coefficients from the padded impedance buffer (slot s holds sample c0 + s - 1)
// FULL: every column of every lane's chunk exists (the segment is complete) -- the per-column existence tests drop
// out and only the lane that holds the ray's first two columns patches them afterwards.
template <class G, bool FULL = false>
__device__ __forceinline__ void chunk_reflections(const float* zbuf, int c0, int ncol, const float* median, float med,
                                                  int lane, float r[G::CHUNK], int col_off = 0) {
    const int cl = col_off + lane * G::CHUNK;
    const int zb = G::pad(cl);                   // slots cl .. cl+CHUNK-1 share a 32-column block
    float zp = zbuf[zb];
#pragma unroll
    for (int i = 0; i < G::CHUNK; ++i) {
        float zc = i + 1 < G::CHUNK ? zbuf[zb + i + 1] : zbuf[G::pad(cl + G::CHUNK)];
        float ri = reflection(zp, zc);
        if (!FULL) {
            int c = c0 + cl + i;
            if (c == 1 && median) ri = med;
            ri = (c >= 1 && cl + i < ncol) ? ri : 0.f;
        }
        r[i] = ri;
        zp = zc;
    }
    if (FULL && c0 + cl == 0) {                  // column 0 has no interface; column 1 may carry the pose's median instead
        r[0] = 0.f;
        if (median) r[1] = med;
    }
}

// ---------------------------------------------------------------------------------------
// forward render
// ---------------------------------------------------------------------------------------
constexpr int FWD_SMEM_PER_WARP = FwdGeo::ZBUF + FwdGeo::OBUF;

__device__ __forceinline__ void store_prefix(const RenderParams& p, int64_t ray, int col, const M2& m) {
    // prefix before column `col` (a positive multiple of PREFIX_STRIDE below Sout)
    float4* sp = (float4*)(p.seg_prefix + (ray * p.nprefix + (col / PREFIX_STRIDE - 1)) * 4);
    *sp = make_float4(m.a(), m.b(), m.c(), m.d());
}

template <int SAMPLER, int LAYOUT, bool POSE64>
__global__ void __launch_bounds__(128, 7) render_fwd_kernel(const RenderParams p) {
    using G = FwdGeo;
    extern __shared__ __align__(16) float smem[];
    float* att = smem;
    if (p.frame) fill_attenuation(att, p.Sout, p.alpha);     // (a prefix-only run forms no frame: no table, att_slots = 0)
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int64_t ray = (int64_t)blockIdx.x * (blockDim.x >> 5) + warp;
    if (ray >= p.total_rays) return;
    float* zbuf = smem + p.att_slots + warp * FWD_SMEM_PER_WARP;
    float* obuf = zbuf + G::ZBUF;
    const int64_t pose = pose_of_ray(ray, p);
    RaySetup<POSE64> rs;
    rs.load(p.sources, p.directions, pose, ray - pose * p.n_rays, p.src_pose_stride, p.src_ray_stride, p.dir_pose_stride, p.product_f32);
    const float med = p.median ? __ldg(p.median + pose) : 0.f;
    float* out = p.frame + ray * (int64_t)p.Sout;
    if (lane == 0) zbuf[0] = 0.f;
    // without a frame to write only the prefixes entering segments 1.. are wanted: the last segment is not walked at all
    const int nseg = (p.Sout + G::SEG - 1) / G::SEG - (p.frame ? 0 : 1);

    M2 carry = m2_identity();
    for (int s = 0; s < nseg; ++s) {
        const int c0 = s * G::SEG;
        const int ncol = min(G::SEG, p.Sout - c0);
        // gather phase: lane = consecutive sample
        const int ntile = (ncol + 31) >> 5;
        // batches of tiles: every load of a batch is issued before the first one is combined.  One tile per batch for
        // the trilinear sampler: measured, 28 resident warps (7 CTAs at 72 registers) hide the gather latency better than
        // deeper batches at fewer warps (0.460 vs 0.470 ms per 1024 poses)
        constexpr int GB = SAMPLER == DIFFUS_SAMPLER_NEAREST ? 8 : FWD_GB;
        const int nt_full = (ncol >> 5) / GB * GB;       // batches of complete tiles run without the per-lane bounds tests
        for (int t0 = 0; t0 < nt_full; t0 += GB) {
            Fetch<SAMPLER, LAYOUT> fe[GB];
#pragma unroll
            for (int u = 0; u < GB; ++u) {
                int k = p.start + c0 + (t0 + u) * 32 + lane;
                fe[u].issue(p.vol, rs.coord(0, k), rs.coord(1, k), rs.coord(2, k));
            }
#pragma unroll
            for (int u = 0; u < GB; ++u) {
                float g[3];
                zbuf[G::pad((t0 + u) * 32 + lane + 1)] = fe[u].template finish<false>(g);
            }
        }
        for (int t0 = nt_full; t0 < ntile; t0 += GB) {
            Fetch<SAMPLER, LAYOUT> fe[GB];
#pragma unroll
            for (int u = 0; u < GB; ++u) {
                int idx = (t0 + u) * 32 + lane;
                if (idx < ncol) {
                    int k = p.start + c0 + idx;
                    fe[u].issue(p.vol, rs.coord(0, k), rs.coord(1, k), rs.coord(2, k));
                }
            }
#pragma unroll
            for (int u = 0; u < GB; ++u) {
                int idx = (t0 + u) * 32 + lane;
                if (idx < ncol) {
                    float g[3];
                    zbuf[G::pad(idx + 1)] = fe[u].template finish<false>(g);
                }
            }
        }
        __syncwarp();
        // chunk phase: lane = 16 consecutive columns
        float r[G::CHUNK];
        chunk_reflections<G>(zbuf, c0, ncol, p.median, med, lane, r);
        if (p.frame) {
            carry = forward_chunk<G>(r, carry, obuf, lane);
        } else {                                 // prefix-only run (for the fused backward of rays longer than one pass)
            M2 T = m2_identity();
#pragma unroll
            for (int i = 0; i < G::CHUNK; ++i) T = m2_mul_interface(T, r[i]);
            carry = m2_shfl(m2_mul(warp_exclusive_prefix(T, carry, lane), T), 31);
        }
        if (p.seg_prefix && lane == 0 && c0 + G::SEG < p.Sout) store_prefix(p, ray, c0 + G::SEG, carry);
        __syncwarp();
        // tile phase: attenuate and write, lane = consecutive column
        if (p.frame) {
#pragma unroll 4
            for (int t = 0; t < (ncol >> 5); ++t) {
                int idx = t * 32 + lane;
                __stcs(out + c0 + idx, __fmul_rn(obuf[G::pad(idx)], att[c0 + idx]));   // streaming store: frames are write-once
            }
            if (ncol & 31) {
                int idx = (ncol & ~31) + lane;
                if (idx < ncol) __stcs(out + c0 + idx, __fmul_rn(obuf[G::pad(idx)], att[c0 + idx]));
            }
        }
        if (lane == 0) zbuf[G::pad(0)] = zbuf[G::pad(G::SEG)];   // sample c0+SEG-1 becomes the next segment's left neighbour
        __syncwarp();
    }
}

// ---------------------------------------------------------------------------------------
// backward render (optionally fused with the forward and an MSE loss)
// ---------------------------------------------------------------------------------------
// buffers for PREFIX_STRIDE columns in the backward's padding (rows of CHUNK+1 floats)
constexpr int BWD_ZBUF = FwdGeo::ZBUF;          // PREFIX_STRIDE + 2 slots, padded
constexpr int BWD_OBUF = FwdGeo::OBUF;
constexpr int BWD_DZ = BWD_DZ_STRIDE;           // one padded row per axis
constexpr int BWD_SMEM_PER_WARP = BWD_ZBUF + BWD_OBUF + 3 * BWD_DZ;

// d loss / d volume accumulates with red.global.add.f32 (index_put_(accumulate=True) semantics) into a
// gradient volume that has the SAME layout as the volume being gathered: in the brick layout the 32 lanes
// of a tile (consecutive samples of a ray) hit ~10 cache lines instead of ~32, and the lines are the
// neighbours of the ones just gathered.
template <int SAMPLER, int LAYOUT, bool POSE64>
__device__ __forceinline__ void scatter_volume_grad(const RenderParams& p, const RaySetup<POSE64>& rs, int k, float zbar) {
    float p0 = rs.coord(0, k), p1 = rs.coord(1, k), p2 = rs.coord(2, k);
    if (SAMPLER == DIFFUS_SAMPLER_NEAREST) {
        int i = nearest_index(p0, p.vol.D), j = nearest_index(p1, p.vol.H), kk = nearest_index(p2, p.vol.W);
        atomicAdd(p.grad_volume + grad_offset<LAYOUT>(p.vol, i, j, kk), zbar);
    } else {
        TriCell c;
        tri_axis(p0, p.vol.D, c.i0[0], c.i1[0], c.f[0]);
        tri_axis(p1, p.vol.H, c.i0[1], c.i1[1], c.f[1]);
        tri_axis(p2, p.vol.W, c.i0[2], c.i1[2], c.f[2]);
        uint32_t off[8];
        tri_offsets<GradLayout<LAYOUT>::value>(p.vol, c, off);
#pragma unroll
        for (int q = 0; q < 8; ++q) {
            float w = ((q & 4) ? c.f[0] : 1.f - c.f[0]) * ((q & 2) ? c.f[1] : 1.f - c.f[1]) * ((q & 1) ? c.f[2] : 1.f - c.f[2]);
            if (w != 0.f) atomicAdd(p.grad_volume + off[q], w * zbar);
        }
    }
}

// ---------------------------------------------------------------------------------------
// d loss / d volume into a BRICK-layout gradient buffer with VECTOR reductions (red.global.add.v4.f32, sm_90+).
//
// What the L2 charges for a scattered reduction is the (instruction, 32-byte sector) pair -- about 195 G of them per
// second on a B200 whether the lane carries one float or four (benchmarks/micro/red_probe.cu, profiles/r2_red_probe.md)
// -- and the scalar scatter above pays 4.2 of them per sample.  Here a lane owns 16 CONSECUTIVE samples of the ray and
// walks them in order, keeping in registers one 16-byte "quad" accumulator (1 x 2 x 2 voxels = 4 consecutive floats of a
// brick: (j & 1, k & 1) at fixed i) per PARITY SLOT (i & 1, (j >> 1) & 1, (k >> 1) & 1).  A trilinear cell spans two
// i-planes and at most two quads along j and along k, one of each parity, so its 8 corners fall into the 8 slots; along
// a straight ray the samples that touch a given quad are consecutive, and a quad can only ever live in its own slot.  A
// slot is therefore flushed -- ONE red.v4 -- exactly when the ray has left its quad: 1.4 vector reductions per sample
// instead of 4.2 scalar ones (5.6 atomics), with no shared-memory atomics, no tags in memory and no divergent control flow.
// Measured and rejected (benchmarks/gpu/r2_call45.sh): six per-axis key components instead of eight slot keys, every slot
// re-keyed at every sample and flushed inside a branch when one of its components changed -- fewer instructions on paper
// (no slot-key sums, no "touched" flags), but a slot misses in some lane of the warp at almost every sample, so the branch
// bodies run nearly always: config 4 step 5.78 vs 5.10 ms (5.65 with two samples per trip).
// ---------------------------------------------------------------------------------------
constexpr uint32_t QUAD_NONE = 0xffffffffu;
constexpr int SCATTER_RUN = PREFIX_STRIDE / 32;      // consecutive samples per lane in the scatter phase

__device__ __forceinline__ void red_add_v4(float* base, uint32_t quad, const float4& v) {
    asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(base + (size_t)quad * 4), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w)
                 : "memory");
}

// predicated form of red_add_v4: no branch around the (rare) flush, so the eight slot updates of a sample stay straight-line code
__device__ __forceinline__ void red_add_v4_if(float* base, uint32_t quad, const float4& v, bool go) {
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %5, 0;\n\t@p red.global.add.v4.f32 [%0], {%1, %2, %3, %4};\n\t}\n" ::"l"(base + (size_t)quad * 4),
        "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w), "r"((int)go)
        : "memory");
}

// one parity slot: accumulate a * (w0, w1) x (k-weights) under `key`; when the slot holds another quad, that quad is complete --
// it is flushed (predicated reduction) and the slot restarts from zero.  Branch-free: 4 selects + 4 FMAs for the accumulators.
__device__ __forceinline__ void quad_slot_fma(float* grad, uint32_t& K, float4& acc, uint32_t key, float a0, float a1, float k0, float k1,
                                              bool nz) {
    const bool miss = nz && key != K;
    red_add_v4_if(grad, K, acc, miss && K != QUAD_NONE);
    K = miss ? key : K;
    acc.x = __fmaf_rn(a0, k0, miss ? 0.f : acc.x);          // a0 = a1 = 0 when !nz: the slot is left as it is
    acc.y = __fmaf_rn(a0, k1, miss ? 0.f : acc.y);
    acc.z = __fmaf_rn(a1, k0, miss ? 0.f : acc.z);
    acc.w = __fmaf_rn(a1, k1, miss ? 0.f : acc.w);
}

// (nearest sampler) one parity slot: accumulate `v` under `key`
__device__ __forceinline__ void quad_slot_update(float* grad, uint32_t& K, float4& acc, uint32_t key, const float4& v, bool nz) {
    const bool miss = nz && key != K;
    if (miss && K != QUAD_NONE) red_add_v4(grad, K, acc);
    if (miss) { K = key; acc = make_float4(0.f, 0.f, 0.f, 0.f); }
    acc.x += v.x; acc.y += v.y; acc.z += v.z; acc.w += v.w;          // v is all zero when !nz
}

// the two voxels (v0, v0 + 1 clamped) of a cell along j or k, split over the quad of each parity:
// q[par] = quad index, w[par][local] = weight of the voxel at position `local` of that quad (0 if the cell does not reach it)
__device__ __forceinline__ void split_over_quads(int v0, float f, uint32_t q[2], float w[2][2]) {
    const float w0 = 1.f - f, w1 = f;
    const uint32_t q0 = (uint32_t)v0 >> 1;
    const bool odd = v0 & 1, same0 = (q0 & 1u) == 0u;
    const float s0 = odd ? 0.f : w0, s1 = odd ? w0 : w1, o0 = odd ? w1 : 0.f;       // the quad of v0 / the next quad
    q[0] = same0 ? q0 : q0 + 1u;
    q[1] = same0 ? q0 + 1u : q0;
    w[0][0] = same0 ? s0 : o0; w[0][1] = same0 ? s1 : 0.f;
    w[1][0] = same0 ? o0 : s0; w[1][1] = same0 ? 0.f : s1;
}

template <int SAMPLER, bool POSE64>
__device__ __forceinline__ void scatter_pass_quads(const RenderParams& p, const RaySetup<POSE64>& rs, const float* gbuf, int c0, int ncol,
                                                   int lane) {
    using G = BwdGeo;
    const uint32_t qsx = p.vol.gsx >> 2, qsy = p.vol.gsy >> 2;      // brick strides in quads
    float* grad = p.grad_volume;
    const int col0 = lane * SCATTER_RUN;
    if (SAMPLER == DIFFUS_SAMPLER_NEAREST) {
        uint32_t K = QUAD_NONE;
        float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll 2
        for (int i = 0; i < SCATTER_RUN; ++i) {
            const int c = col0 + i;
            const float zbar = c < ncol ? gbuf[G::pad(c)] : 0.f;
            const int k = p.start + c0 + c;
            const int vi = nearest_index(rs.coord(0, k), p.vol.D), vj = nearest_index(rs.coord(1, k), p.vol.H),
                      vk = nearest_index(rs.coord(2, k), p.vol.W);
            const uint32_t key = ((uint32_t)vi >> 2) * qsx + (((uint32_t)vi & 3u) << 1) + ((uint32_t)vj >> 2) * qsy + (((uint32_t)vj >> 1) & 1u) +
                                 (((uint32_t)vk >> 1) << 3);
            const int pos = ((vj & 1) << 1) | (vk & 1);
            const float4 v = make_float4(pos == 0 ? zbar : 0.f, pos == 1 ? zbar : 0.f, pos == 2 ? zbar : 0.f, pos == 3 ? zbar : 0.f);
            quad_slot_update(grad, K, acc, key, v, zbar != 0.f);
        }
        if (K != QUAD_NONE) red_add_v4(grad, K, acc);
        return;
    }
    uint32_t K[8];
    float4 acc[8];
#pragma unroll
    for (int s = 0; s < 8; ++s) { K[s] = QUAD_NONE; acc[s] = make_float4(0.f, 0.f, 0.f, 0.f); }
    // one sample per trip (two: config 4 step 5.26 vs 5.04 ms, benchmarks/gpu/r2_call56.sh)
#pragma unroll 1
    for (int i = 0; i < SCATTER_RUN; ++i) {
        const int c = col0 + i;
        const float zbar = c < ncol ? gbuf[G::pad(c)] : 0.f;
        const int k = p.start + c0 + c;
        int i0, i1, j0, j1, k0, k1;
        float f0, f1, f2;
        tri_axis(rs.coord(0, k), p.vol.D, i0, i1, f0);
        tri_axis(rs.coord(1, k), p.vol.H, j0, j1, f1);
        tri_axis(rs.coord(2, k), p.vol.W, k0, k1, f2);
        // i: one plane per parity (the clamped top plane repeats i0 with weight 0: a no-op)
        const bool iodd = i0 & 1;
        const int ip[2] = {iodd ? i1 : i0, iodd ? i0 : i1};
        const float wi[2] = {(iodd ? f0 : 1.f - f0) * zbar, (iodd ? 1.f - f0 : f0) * zbar};
        uint32_t jq[2], kq[2];
        float wj[2][2], wk[2][2];
        split_over_quads(j0, f1, jq, wj);
        split_over_quads(k0, f2, kq, wk);
        uint32_t X[2], Y[2], Z[2];
        bool nzi[2], nzj[2], nzk[2];
#pragma unroll
        for (int a = 0; a < 2; ++a) {
            X[a] = ((uint32_t)ip[a] >> 2) * qsx + (((uint32_t)ip[a] & 3u) << 1);
            Y[a] = (jq[a] >> 1) * qsy + (jq[a] & 1u);
            Z[a] = kq[a] << 3;
            nzi[a] = wi[a] != 0.f;
            nzj[a] = wj[a][0] != 0.f || wj[a][1] != 0.f;
            nzk[a] = wk[a][0] != 0.f || wk[a][1] != 0.f;
        }
#pragma unroll
        for (int pi = 0; pi < 2; ++pi)
#pragma unroll
            for (int pj = 0; pj < 2; ++pj) {
                const float a0 = wi[pi] * wj[pj][0], a1 = wi[pi] * wj[pj][1];
#pragma unroll
                for (int pk = 0; pk < 2; ++pk) {
                    const int s = (pi << 2) | (pj << 1) | pk;
                    quad_slot_fma(grad, K[s], acc[s], X[pi] + Y[pj] + Z[pk], a0, a1, wk[pk][0], wk[pk][1], nzi[pi] && nzj[pj] && nzk[pk]);
                }
            }
    }
#pragma unroll
    for (int s = 0; s < 8; ++s)
        if (K[s] != QUAD_NONE) red_add_v4(grad, K[s], acc[s]);
}

// ONE_PASS: the ray fits one 512-column pass (every BASELINE config but the 2048-sample stress case).  The pass
// loop disappears, so the accumulators and the adjoint carried between passes are not live during the gather; the
// pose-only kernels then fit 96 registers and run 5 CTAs (20 warps) per SM: 0.817 -> 0.753 ms per 1024 poses.
// WIDE (one-pass rays longer than 256 columns): the reverse sweep walks the pass as ONE 512-column segment, 16 columns per
// lane with a prefix checkpoint every 4 (Geo<16, 4>), instead of two 256-column sub-segments of 8 columns per lane: one
// prefix scan and one suffix scan per ray instead of two of each, no prefix pre-pass over the first sub-segment, for 1.5
// instead of 0.5 recomputed transfer products per column.  (Rays longer than one pass as WIDE segments: 612 bytes of spills.)
using WideGeo = Geo<16, 4>;
// COOP (rays of 513..2048 columns = two to four passes; config 5 has four): ONE ray per CTA of as many warps as the ray has
// passes, warp w walks pass w.  The passes of a ray
// depend on each other only through (i) the forward prefix entering the pass = the product of the earlier passes' transfer
// products, (ii) the adjoint entering its last column = the later passes' reverse sweeps, each an affine map V -> V A + B that
// the pass knows once its own prefix is known, and (iii) the weight of the next pass's first column.  All three go through
// shared memory (CoopXch; five __syncthreads per ray in all), so the ray is gathered ONCE: no forward pre-pass for the 512-column
// prefixes (it re-gathered 3 of 4 passes, ~30 % of the config-5 step), no state carried from pass to pass through the gather
// loop (the single 512-column WIDE sweep fits 128 registers like the one-pass kernel's).
template <int SAMPLER, int LAYOUT, bool POSE64, bool POSE_GRAD, bool VOL_GRAD, int LOSS, bool ONE_PASS, bool WIDE = false,
          bool COOP = false>
__global__ void __launch_bounds__(128, COOP ? 4 : WIDE ? WIDE_CTAS : ((ONE_PASS && !VOL_GRAD) ? 5 : 4))
render_bwd_kernel(const RenderParams p) {
    static_assert(!COOP || (WIDE && !ONE_PASS && !VOL_GRAD && !POSE64), "COOP: long rays, WIDE sweep, no volume gradient");
    using G = typename std::conditional<WIDE, WideGeo, BwdGeo>::type;
    constexpr int BWD_SUB = PREFIX_STRIDE / G::SEG;
    constexpr int SS = PREFIX_STRIDE;        // columns gathered per pass (BWD_SUB sub-segments of G::SEG)
    extern __shared__ __align__(16) float smem[];
    float* att = smem;                       // padded like the column buffers: conflict free in the chunk phase
    // Rays longer than one pass keep only the first 512 entries, exp(-alpha i), and multiply by exp(-alpha c0) per pass
    // (one more rounding, one more multiply per column): the table then costs 2 KB instead of 8 KB at 2048 samples, and four
    // CTAs fit the 196 KB carveout -- 60 instead of 28 KB of L1 / texture cache for the gathers of config 5.
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int64_t ray = COOP ? (int64_t)blockIdx.x : (int64_t)blockIdx.x * (blockDim.x >> 5) + warp;
    const bool live = ray < p.total_rays;
    // the ray's pose is loaded BEFORE the attenuation table is filled: the loads fly while the table is computed (a CTA's
    // serial start -- table, barrier, pose loads, first gathers -- is time during which its slot on the SM does no work)
    const int64_t pose = live ? pose_of_ray(ray, p) : 0;
    RaySetup<POSE64> rs;
    float med = 0.f;
    if (live) {
        rs.load(p.sources, p.directions, pose, ray - pose * p.n_rays, p.src_pose_stride, p.src_ray_stride, p.dir_pose_stride, p.product_f32);
        if (p.median) med = __ldg(p.median + pose);
    }
    fill_attenuation_padded<G>(att, ONE_PASS ? p.Sout : min(p.Sout, SS), p.alpha);
    if (!live) return;                       // (COOP: the grid is exactly the rays -- no warp leaves before the barriers)
    float* zbuf = smem + p.att_slots_padded + warp * BWD_SMEM_PER_WARP;
    float* gbuf = zbuf + BWD_ZBUF;           // target / upstream gradient in, d loss / d r out
    float* dz = gbuf + BWD_OBUF;             // [3][BWD_DZ] spatial gradient of Z at each sample (padded rows)
    const float* gin = (LOSS == LOSS_MSE ? p.target : p.grad_frame) + ray * (int64_t)p.Sout;
    float* fout = (LOSS == LOSS_MSE && p.frame) ? p.frame + ray * (int64_t)p.Sout : nullptr;
    if (lane == 0) zbuf[0] = 0.f;
    const int nss = ONE_PASS ? 1 : (p.Sout + SS - 1) / SS;
    const uint64_t stream_policy = l2_evict_first_policy();

    M2 vin = m2_zero();
    float carry_w = 0.f, carry_z = 0.f;      // first column of the later pass: its weight w and its impedance
    ZTail zt;
    zt.zbuf = zbuf;
    zt.dz = dz;
    zt.rbar1 = nullptr;
    zt.xch = smem + p.att_slots_padded + (blockDim.x >> 5) * BWD_SMEM_PER_WARP;     // (COOP only; the launcher adds the room)
#pragma unroll
    for (int a = 0; a < 3; ++a) zt.acc[a] = make_float2(0.f, 0.f);
    float loss_acc = 0.f;

    for (int s = COOP ? warp : nss - 1; s >= (COOP ? warp : 0); --s) {
        const int c0 = s * SS;
        const int ncol = min(SS, p.Sout - c0);
        const int ntile = (ncol + 31) >> 5;
        const int nsub = (ncol + G::SEG - 1) / G::SEG;
        // The target (or upstream-gradient) row streams from HBM: copy it straight into shared
        // memory with cp.async at the top of the pass so its latency hides behind the gathers.  (Staged lane-major and moved
        // as float4 in the sweeps: 132 fewer instructions per ray, bit-identical, but 0.560 vs 0.536 ms.)
        {
            const int nt = nsub * (G::SEG / 32);
            // complete tiles: no bounds test.  pad(32 t + lane) = 33 t + lane: both addresses advance by a constant per
            // tile, so the copies are one instruction each with immediate offsets
            {
                float* dst = gbuf + lane;
                const float* src = gin + c0 + lane;
                const int nfull = ncol >> 5;
                if ((ONE_PASS || COOP) && nfull == SS / 32) {
#pragma unroll
                    for (int t = 0; t < SS / 32; ++t) cp_async_stream4(dst + 33 * t, src + 32 * t, stream_policy);
                } else {
                    for (int t = 0; t < nfull; ++t) cp_async_stream4(dst + 33 * t, src + 32 * t, stream_policy);
                }
            }
            for (int t = ncol >> 5; t < nt; ++t) {
                int idx = t * 32 + lane;
                if (idx < ncol) cp_async_stream4(gbuf + G::pad(idx), gin + c0 + idx, stream_policy);
                else gbuf[G::pad(idx)] = 0.f;            // columns that do not exist carry no gradient
            }
            __pipeline_commit();
            // gather phase: one pass over the volume for these columns.  (A cp.async ring for the
            // gathers themselves was measured slower than plain loads: LDGSTS issues at a quarter of
            // the LDG rate and adds eight shared-memory reads per sample, DESIGN.md section 4.)
            // Tiles go in batches: all loads of a batch are issued before the first is combined, so a warp
            // keeps GB tiles of gathers in flight.
            // Measured on the one-pass pose kernel (96 registers, 5 CTAs = 20 warps per SM), batches of 1 / 2 / 4 tiles:
            // 0.701 / 0.687 / 0.705 ms per 1024 poses (before the bounds tests left the loop below, two tiles still
            // spilled and one tile per batch was the fastest: 0.753 / 0.779 / 0.785).
            // TEXTURE (round 2): with the shared-memory carveout sized to the resident CTAs (60 KB of L1 / texture cache instead of 28)
            // deeper batches pay again on the WIDE kernel (128 registers): 1 pipelined / 2 / 2 pipelined / 4 / 4 pipelined / 8 tiles:
            // 0.564 / 0.573 / 0.555 / 0.542 / 0.562 / 0.586 ms (profiles/r2_carveout.md; pipelined: the next batch is issued
            // before the current one is combined).
            constexpr int GB = SAMPLER == DIFFUS_SAMPLER_NEAREST ? 8 : (LAYOUT == DIFFUS_LAYOUT_TEXTURE ? (WIDE ? TEX_GB_WIDE : TEX_GB) : ((LAYOUT == DIFFUS_LAYOUT_QUAD && ONE_PASS) ? 4 : 2));
            // batches whose tiles are all complete run without the per-lane bounds tests; the tail keeps them
            const int nt_full = (ncol >> 5) / GB * GB;
            auto issue_batch = [&](Fetch<SAMPLER, LAYOUT>(&fe)[GB], int t0) {
#pragma unroll
                for (int u = 0; u < GB; ++u) {
                    int k = p.start + c0 + (t0 + u) * 32 + lane;
                    fe[u].template issue<POSE_GRAD>(p.vol, rs.coord(0, k), rs.coord(1, k), rs.coord(2, k));
                }
            };
            // pad(32 t + lane) = 33 t + lane and pad(32 t + lane + 1) = 33 t + lane + 1 (+ 1 more for lane 31): one base per
            // batch, immediate offsets per tile
            const int lane_z = lane + 1 + (lane == 31 ? 1 : 0);
            auto finish_batch = [&](const Fetch<SAMPLER, LAYOUT>(&fe)[GB], int t0) {
                float* zt0 = zbuf + 33 * t0 + lane_z;
                float* dt0 = dz + 33 * t0 + lane;
#pragma unroll
                for (int u = 0; u < GB; ++u) {
                    float g[3];
                    float z = fe[u].template finish<POSE_GRAD>(g);
                    zt0[33 * u] = z;
                    if (POSE_GRAD) {
                        dt0[33 * u] = g[0]; dt0[BWD_DZ + 33 * u] = g[1]; dt0[2 * BWD_DZ + 33 * u] = g[2];
                    }
                }
            };
            for (int t0 = 0; t0 < nt_full; t0 += GB) {
                Fetch<SAMPLER, LAYOUT> fe[GB];
                issue_batch(fe, t0);
                finish_batch(fe, t0);
            }
            for (int t0 = nt_full; t0 < nt; t0 += GB) {
                Fetch<SAMPLER, LAYOUT> fe[GB];
#pragma unroll
                for (int u = 0; u < GB; ++u) {
                    int idx = (t0 + u) * 32 + lane;
                    if (idx < ncol) {
                        int k = p.start + c0 + idx;
                        fe[u].template issue<POSE_GRAD>(p.vol, rs.coord(0, k), rs.coord(1, k), rs.coord(2, k));
                    }
                }
#pragma unroll
                for (int u = 0; u < GB; ++u) {
                    int idx = (t0 + u) * 32 + lane;
                    if (idx < ncol) {
                        float g[3];
                        float z = fe[u].template finish<POSE_GRAD>(g);
                        zbuf[G::pad(idx + 1)] = z;
                        if (POSE_GRAD) {
                            const int di = G::pad(idx);
                            dz[di] = g[0]; dz[BWD_DZ + di] = g[1]; dz[2 * BWD_DZ + di] = g[2];
                        }
                    } else if (POSE_GRAD) {               // no sample: the reverse sweep multiplies these by zbar = 0
                        const int di = G::pad(idx);
                        dz[di] = 0.f; dz[BWD_DZ + di] = 0.f; dz[2 * BWD_DZ + di] = 0.f;
                    }
                }
            }
            __pipeline_wait_prior(0);
        }
        if (COOP) {
            // the sample before the pass's first column is the previous warp's last one: one more barrier instead of one more
            // (dependent, single-lane) gather per pass: config 5 9.64 -> 9.42 ms (benchmarks/gpu/r2_call57.sh)
            __syncthreads();
            if (lane == 0 && warp > 0) zbuf[G::pad(0)] = zbuf[G::pad(SS) - BWD_SMEM_PER_WARP];
        }
        if (lane == 0) {
            if (s > 0 && !COOP) {                     // left neighbour of the pass's first column
                int k = p.start + c0 - 1;
                float g[3];
                zbuf[G::pad(0)] = sample_volume<SAMPLER, LAYOUT, false>(p.vol, rs.coord(0, k), rs.coord(1, k), rs.coord(2, k), g);
            }
            if (!COOP) zbuf[G::pad(ncol + 1)] = carry_z;    // the sample after the pass's last column lives in the later pass
        }
        __syncwarp();

        // forward prefixes entering each sub-segment (the first one comes from the forward kernel)
        M2 carry[BWD_SUB];
        carry[0] = m2_identity();
        if (!COOP && s > 0) {
            float4 c4 = __ldg((const float4*)(p.seg_prefix + (ray * p.nprefix + (s - 1)) * 4));
            carry[0] = m2_make(c4.x, c4.y, c4.z, c4.w);
        }
        float r[G::CHUNK];
        M2 T0 = m2_identity(), E0 = m2_identity();       // sub-segment 0's chunk products and prefixes, kept for its reverse scan
        static_assert(BWD_SUB <= 2, "the prefix pass keeps one sub-segment's products in registers");
        static_assert(!COOP || BWD_SUB == 1, "COOP: one sub-segment per pass");
        const bool have0 = BWD_SUB == 2 && nsub > 1;
        // COOP: every pass but the last is complete; the instantiation of the reverse sweep must be the same for all the warps
        const bool coop_full = COOP && p.Sout == (int)(blockDim.x >> 5) * SS;
        if (COOP) {
            if (ncol == SS) chunk_reflections<G, true>(zbuf, c0, ncol, p.median, med, lane, r, 0);
            else chunk_reflections<G, false>(zbuf, c0, ncol, p.median, med, lane, r, 0);
#pragma unroll
            for (int i = 0; i < G::CHUNK; ++i) T0 = m2_mul_interface(T0, r[i]);
            const M2 el = warp_exclusive_prefix(T0, m2_identity(), lane);          // within the pass
            const M2 tot = m2_shfl(m2_mul(el, T0), 31);
            if (lane == 0) xch_store(zt.xch + CoopXch::TOTAL + 4 * warp, tot);
            __syncthreads();
            for (int u = 0; u < warp; ++u) carry[0] = m2_mul(carry[0], xch_load(zt.xch + CoopXch::TOTAL + 4 * u));
            E0 = m2_mul(carry[0], el);
            // the sample after the pass's last column is the next warp's first one (its gathers are done: same barrier)
            if (lane == 0) zbuf[G::pad(ncol + 1)] = warp + 1 < (int)(blockDim.x >> 5) ? zbuf[BWD_SMEM_PER_WARP + G::pad(1)] : 0.f;
            __syncwarp();
        } else if (BWD_SUB == 1) {
        } else if (have0) {                      // sub-segment 0 is complete whenever there is a second one
            chunk_reflections<G, true>(zbuf, c0, ncol, p.median, med, lane, r, 0);
#pragma unroll
            for (int i = 0; i < G::CHUNK; ++i) T0 = m2_mul_interface(T0, r[i]);
            E0 = warp_exclusive_prefix(T0, carry[0], lane);
            carry[BWD_SUB - 1] = m2_shfl(m2_mul(E0, T0), 31);
        } else {
            carry[BWD_SUB - 1] = carry[0];
        }
        // reverse scan, last sub-segment first; it ends in d loss / d Z per column and the pose accumulators
        zt.w_after = (c0 + ncol < p.Sout) ? carry_w : 0.f;
#pragma unroll
        for (int h = BWD_SUB - 1; h >= 0; --h) {
            if (h < nsub) {
                const int off = h * G::SEG;
                const bool full = COOP ? coop_full : ncol - off >= G::SEG;   // warp-uniform (COOP: CTA-uniform): every column of this sub-segment exists
                if (COOP) {                              // r is already there
                } else if (full) chunk_reflections<G, true>(zbuf, c0, ncol, p.median, med, lane, r, off);
                else chunk_reflections<G, false>(zbuf, c0, ncol, p.median, med, lane, r, off);
                const int lane_col = off + lane * G::CHUNK;
                // columns without a direct impedance dependence: column 0 and the median-replaced column 1
                zt.skip_mask = 0u;
                if (c0 + lane_col == 0) zt.skip_mask = p.median ? 3u : 1u;
                zt.lane_col = lane_col;
                zt.kbase = (float)(p.start + c0 + lane_col);
                zt.rbar1 = (p.first_rbar && s == 0 && h == 0) ? p.first_rbar + ray : nullptr;
                const M2* kt = (COOP || (h == 0 && have0)) ? &T0 : nullptr;
                M2 ch = carry[0];                        // (a select, not an indexed read: carry[h] changes the code and its registers)
                if (BWD_SUB == 2 && h == 1) ch = carry[BWD_SUB - 1];
                float* fl = fout ? fout + c0 + lane_col : nullptr;
                float* gl = gbuf + G::pad(off);
                const float pass_scale = ONE_PASS ? 1.f : expf(-p.alpha * (float)c0);
                const float* asc = ONE_PASS ? nullptr : &pass_scale;
                if (full)
                    vin = backward_chunk<G, LOSS, true, POSE_GRAD, VOL_GRAD, true, COOP>(
                        r, ch, vin, gl, att + G::pad(ONE_PASS ? c0 + lane_col : lane_col), fl, p.grad_scale, ncol - lane_col,
                        loss_acc, lane, &zt, kt, &E0, asc);
                else
                    vin = backward_chunk<G, LOSS, true, POSE_GRAD, VOL_GRAD, false, COOP>(
                        r, ch, vin, gl, att + G::pad(ONE_PASS ? c0 + lane_col : lane_col), fl, p.grad_scale, ncol - lane_col,
                        loss_acc, lane, &zt, kt, &E0, asc);
                zt.w_after = zt.w_first;
            }
        }
        carry_w = zt.w_first;
        carry_z = zbuf[G::pad(1)];
        __syncwarp();

        // tile phase, only for the volume gradient: scatter d loss / d Z_c with lane = consecutive sample
        if (VOL_GRAD) {
            if (GradLayout<LAYOUT>::value == DIFFUS_LAYOUT_BRICK) {
                scatter_pass_quads<SAMPLER, POSE64>(p, rs, gbuf, c0, ncol, lane);       // lane = 16 consecutive samples
            } else {
                for (int t = 0; t < ntile; ++t) {                                        // lane = consecutive sample
                    int idx = t * 32 + lane;
                    if (idx < ncol) {
                        float zbar = gbuf[G::pad(idx)];
                        if (zbar != 0.f) scatter_volume_grad<SAMPLER, LAYOUT, POSE64>(p, rs, p.start + c0 + idx, zbar);
                    }
                }
            }
            __syncwarp();
        }
    }
    if (COOP) {                                  // the ray's passes add up in a fixed order: warp 0 writes the ray's partials
        float* out = zt.xch + CoopXch::OUT + 8 * warp;
        {                                        // (COOP kernels are pose-gradient kernels) the pass's seven sums, transposed
            float v[8] = {zt.acc[0].x, zt.acc[1].x, zt.acc[2].x, zt.acc[0].y, zt.acc[1].y, zt.acc[2].y, loss_acc, 0.f};
            const float t = warp_sum8(v, lane);
            if (lane < 8) out[warp_sum8_index(lane)] = t;
        }
        __syncthreads();
        if (warp == 0 && lane < 7) {
            const float* o = zt.xch + CoopXch::OUT + lane;
            float v = o[0];
            for (int u = 1; u < (int)(blockDim.x >> 5); ++u) v += o[8 * u];
            if (POSE_GRAD && lane < 3) p.grad_src_partial[ray * 3 + lane] = v;
            if (POSE_GRAD && lane >= 3 && lane < 6) p.grad_dir[ray * 3 + lane - 3] = v;
            if (LOSS == LOSS_MSE && lane == 6 && p.loss_partial) p.loss_partial[ray] = v;
        }
        return;
    }
    if (POSE_GRAD) {             // the ray's seven sums (3 + 3 + loss) in one transposing reduction: 9 shuffles instead of 35
        float v[8] = {zt.acc[0].x, zt.acc[1].x, zt.acc[2].x, zt.acc[0].y, zt.acc[1].y, zt.acc[2].y, loss_acc, 0.f};
        const float t = warp_sum8(v, lane);
        const int j = warp_sum8_index(lane);
        if (lane < 8) {
            if (j < 3) p.grad_src_partial[ray * 3 + j] = t;
            else if (j < 6) p.grad_dir[ray * 3 + j - 3] = t;
            else if (j == 6 && LOSS == LOSS_MSE && p.loss_partial) p.loss_partial[ray] = t;
        }
        return;
    }
    if (LOSS == LOSS_MSE && p.loss_partial) {
        float l = warp_sum(loss_acc);
        if (lane == 0) p.loss_partial[ray] = l;
    }
}

#ifndef DIFFUS_LAYOUT_SLICE
// ---------------------------------------------------------------------------------------
// echo-only kernels: compute_echo_traces on explicit coefficients (src/renderer.py:439-457)
// refl (B, N) -> echo (B, N+1); column c >= 1 uses refl[c-1]
// ---------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128) echo_fwd_kernel(const float* __restrict__ refl, int64_t n_rays, int N,
                                                       float* __restrict__ echo) {
    using G = FwdGeo;
    extern __shared__ __align__(16) float smem[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int64_t ray = (int64_t)blockIdx.x * (blockDim.x >> 5) + warp;
    if (ray >= n_rays) return;
    float* rbuf = smem + warp * (2 * G::OBUF);
    float* obuf = rbuf + G::OBUF;
    const int Sout = N + 1, nseg = (Sout + G::SEG - 1) / G::SEG;
    const float* rin = refl + ray * (int64_t)N;
    float* out = echo + ray * (int64_t)Sout;
    M2 carry = m2_identity();
    for (int s = 0; s < nseg; ++s) {
        const int c0 = s * G::SEG, ncol = min(G::SEG, Sout - c0);
        for (int idx = lane; idx < G::SEG; idx += 32) {
            int c = c0 + idx;
            rbuf[G::pad(idx)] = (c >= 1 && idx < ncol) ? __ldg(rin + c - 1) : 0.f;
        }
        __syncwarp();
        float r[G::CHUNK];
#pragma unroll
        for (int i = 0; i < G::CHUNK; ++i) r[i] = rbuf[G::pad(lane * G::CHUNK + i)];
        carry = forward_chunk<G>(r, carry, obuf, lane);
        __syncwarp();
        for (int idx = lane; idx < ncol; idx += 32) out[c0 + idx] = obuf[G::pad(idx)];
        __syncwarp();
    }
}

// two passes over the segments: forward to collect the prefixes, then the reverse scan
__global__ void __launch_bounds__(128) echo_bwd_kernel(const float* __restrict__ refl, const float* __restrict__ grad_echo,
                                                       int64_t n_rays, int N, float* __restrict__ grad_refl) {
    using G = BwdGeo;
    extern __shared__ __align__(16) float smem[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int64_t ray = (int64_t)blockIdx.x * (blockDim.x >> 5) + warp;
    if (ray >= n_rays) return;
    const int Sout = N + 1, nseg = (Sout + G::SEG - 1) / G::SEG;
    float* rbuf = smem + warp * (2 * G::OBUF + 4 * nseg);
    float* gbuf = rbuf + G::OBUF;
    float* prefix = gbuf + G::OBUF;          // carry entering segment s, 4 floats each
    const float* rin = refl + ray * (int64_t)N;
    const float* gin = grad_echo + ray * (int64_t)Sout;
    float* gout = grad_refl + ray * (int64_t)N;
    M2 carry = m2_identity();
    for (int s = 0; s < nseg; ++s) {
        const int c0 = s * G::SEG, ncol = min(G::SEG, Sout - c0);
        if (lane == 0) { prefix[4 * s] = carry.a(); prefix[4 * s + 1] = carry.b(); prefix[4 * s + 2] = carry.c(); prefix[4 * s + 3] = carry.d(); }
        if (s + 1 == nseg) break;
        for (int idx = lane; idx < G::SEG; idx += 32) {
            int c = c0 + idx;
            rbuf[G::pad(idx)] = (c >= 1 && idx < ncol) ? __ldg(rin + c - 1) : 0.f;
        }
        __syncwarp();
        M2 T = m2_identity();
#pragma unroll
        for (int i = 0; i < G::CHUNK; ++i) T = m2_mul_interface(T, rbuf[G::pad(lane * G::CHUNK + i)]);
        M2 P = warp_exclusive_prefix(T, carry, lane);
        carry = m2_shfl(m2_mul(P, T), 31);
        __syncwarp();
    }
    __syncwarp();
    M2 vin = m2_zero();
    float unused = 0.f;
    for (int s = nseg - 1; s >= 0; --s) {
        const int c0 = s * G::SEG, ncol = min(G::SEG, Sout - c0);
        for (int idx = lane; idx < G::SEG; idx += 32) {
            int c = c0 + idx;
            bool ok = idx < ncol;
            rbuf[G::pad(idx)] = (c >= 1 && ok) ? __ldg(rin + c - 1) : 0.f;
            gbuf[G::pad(idx)] = ok ? __ldg(gin + c) : 0.f;
        }
        __syncwarp();
        float r[G::CHUNK];
#pragma unroll
        for (int i = 0; i < G::CHUNK; ++i) r[i] = rbuf[G::pad(lane * G::CHUNK + i)];
        M2 cs = m2_make(prefix[4 * s], prefix[4 * s + 1], prefix[4 * s + 2], prefix[4 * s + 3]);
        vin = backward_chunk<G, LOSS_GRAD>(r, cs, vin, gbuf, nullptr, nullptr, 0.f, ncol - lane * G::CHUNK, unused, lane);
        __syncwarp();
        for (int idx = lane; idx < ncol; idx += 32) {
            int c = c0 + idx;
            if (c >= 1) gout[c - 1] = gbuf[G::pad(idx)];
        }
        __syncwarp();
    }
}

// sum of per-ray partials -> one float in a FIXED order (run-to-run identical), without atomics, tickets or memsets:
// up to 2^18 partials one 1024-thread block does it all (a few us for the 131 072 rays of a 1024-pose sweep); above that a
// first launch leaves REDUCE_BLOCKS double partials in the workspace and a second one adds them up in index order.
__device__ __forceinline__ double block_sum_fixed_order(double acc, double* warp_part) {
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) acc += __shfl_xor_sync(FULL, acc, d);
    if ((threadIdx.x & 31) == 0) warp_part[threadIdx.x >> 5] = acc;
    __syncthreads();
    double t = 0.0;
    if (threadIdx.x == 0)
        for (int w = 0; w < (int)(blockDim.x >> 5); ++w) t += warp_part[w];
    return t;                                 // valid on thread 0
}

// this thread's share of the sum of n floats, in double: four independent chains of 16-byte loads when the array is 16-byte
// aligned (a single chain of scalar loads made the sum of 2^17 loss partials a 10 us latency chain in one CTA)
__device__ __forceinline__ double sum_partials(const float* __restrict__ x, int64_t n) {
    double a0 = 0.0, a1 = 0.0, a2 = 0.0, a3 = 0.0;
    const int64_t n4 = ((((uintptr_t)x) & 15u) == 0) ? n >> 2 : 0;
    const float4* x4 = (const float4*)x;
#pragma unroll 4
    for (int64_t i = threadIdx.x; i < n4; i += blockDim.x) {
        const float4 v = __ldg(x4 + i);
        a0 += (double)v.x; a1 += (double)v.y; a2 += (double)v.z; a3 += (double)v.w;
    }
    for (int64_t i = (n4 << 2) + threadIdx.x; i < n; i += blockDim.x) a0 += (double)__ldg(x + i);
    return (a0 + a1) + (a2 + a3);
}

__global__ void __launch_bounds__(1024) reduce_sum_kernel(const float* __restrict__ partial, int64_t n, float scale,
                                                          float* __restrict__ out, double* __restrict__ block_sums) {
    __shared__ double warp_part[32];
    const int64_t per = ((n + gridDim.x - 1) / gridDim.x + 3) & ~(int64_t)3;      // a multiple of 4: every block starts 16-byte aligned
    const int64_t lo = min(n, (int64_t)blockIdx.x * per), hi = min(n, lo + per);
    const double acc = sum_partials(partial + lo, hi - lo);
    const double t = block_sum_fixed_order(acc, warp_part);
    if (threadIdx.x == 0) {
        if (block_sums) block_sums[blockIdx.x] = t;
        else out[0] = (float)(t * (double)scale);
    }
}

__global__ void reduce_final_kernel(const double* __restrict__ block_sums, int n, float scale, float* __restrict__ out) {
    if (threadIdx.x == 0) {
        double t = 0.0;
        for (int b = 0; b < n; ++b) t += block_sums[b];
        out[0] = (float)(t * (double)scale);
    }
}

// The two reductions behind the fused pose step in ONE launch (one launch gap less per step: what a 128-pose shard of a strong-
// scaled sweep, or a single pose-recovery step, notices): the last CTA sums the per-ray loss partials (the job of
// reduce_sum_kernel<<<1, 1024>>>), every other CTA sums the per-ray d loss / d source partials of 32 poses exactly like
// reduce_rays_kernel (one warp per pose: same operations in the same order, bit-identical).  The loss is summed in double in the
// fixed order of sum_partials, like reduce_sum_kernel<<<1, 1024>>>: run-to-run identical.
__global__ void __launch_bounds__(1024) reduce_rays_and_sum_kernel(const float* __restrict__ src_partial, int64_t n_poses, int64_t n_rays,
                                                                   float* __restrict__ grad_src, const float* __restrict__ loss_partial,
                                                                   int64_t n, float scale, float* __restrict__ loss_out) {
    __shared__ double warp_part[32];
    if (blockIdx.x == gridDim.x - 1) {
        const double t = block_sum_fixed_order(sum_partials(loss_partial, n), warp_part);
        if (threadIdx.x == 0) loss_out[0] = (float)(t * (double)scale);
        return;
    }
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int64_t pose = (int64_t)blockIdx.x * 32 + warp;
    if (pose >= n_poses) return;
    float a0 = 0.f, a1 = 0.f, a2 = 0.f;
    const float* src = src_partial + pose * n_rays * 3;
    for (int64_t r = lane; r < n_rays; r += 32) { a0 += src[r * 3]; a1 += src[r * 3 + 1]; a2 += src[r * 3 + 2]; }
    a0 = warp_sum(a0); a1 = warp_sum(a1); a2 = warp_sum(a2);
    if (lane == 0) { grad_src[pose * 3] = a0; grad_src[pose * 3 + 1] = a1; grad_src[pose * 3 + 2] = a2; }
}

bool reduce_rays_and_sum_fits(int64_t n) { return n <= ((int64_t)1 << 18); }      // (the single-CTA form of the loss sum)

cudaError_t launch_reduce_rays_and_sum(const float* src_partial, int64_t n_poses, int64_t n_rays, float* grad_src,
                                       const float* loss_partial, int64_t n, float scale, float* loss_out, cudaStream_t st) {
    const unsigned grid = (unsigned)((n_poses + 31) / 32) + 1u;
    return launch_kernel(reduce_rays_and_sum_kernel, grid, 1024, 0, st, src_partial, n_poses, n_rays, grad_src, loss_partial, n, scale, loss_out);
}

constexpr int REDUCE_BLOCKS = 64;
int64_t reduce_sum_workspace_bytes() { return REDUCE_BLOCKS * sizeof(double); }

cudaError_t launch_reduce_sum(const float* partial, int64_t n, float scale, float* out, void* workspace, cudaStream_t st) {
    if (n <= ((int64_t)1 << 18)) {        // (one SM sums 1 MB in ~10 us; the 2 MB of a 4096-pose batch took 79 us under ncu)
        return launch_kernel(reduce_sum_kernel, 1, 1024, 0, st, partial, n, scale, out, nullptr);
    }
    double* sums = (double*)workspace;
    cudaError_t e = launch_kernel(reduce_sum_kernel, REDUCE_BLOCKS, 1024, 0, st, partial, n, scale, out, sums);
    if (e != cudaSuccess) return e;
    return launch_kernel(reduce_final_kernel, 1, 32, 0, st, sums, REDUCE_BLOCKS, scale, out);
}

#endif  // !DIFFUS_LAYOUT_SLICE

// ---------------------------------------------------------------------------------------
// launchers
// ---------------------------------------------------------------------------------------
static int warps_per_block(int64_t total_rays) {
    // small problems: one ray per CTA so a single frame still spreads over the SMs
    if (total_rays >= 4 * 148 * 4) return 4;
    if (total_rays >= 2 * 148 * 2) return 2;
    return 1;
}

#ifdef DIFFUS_LAYOUT_SLICE
#define DIFFUS_CAT2(a, b) a##b
#define DIFFUS_CAT(a, b) DIFFUS_CAT2(a, b)
#define DIFFUS_FWD_NAME DIFFUS_CAT(launch_render_fwd_layout, DIFFUS_LAYOUT_SLICE)
#define DIFFUS_BWD_NAME DIFFUS_CAT(launch_render_bwd_layout, DIFFUS_LAYOUT_SLICE)

cudaError_t DIFFUS_FWD_NAME(const RenderParams& p_in, int sampler, int layout, int pose64, cudaStream_t st) {
    RenderParams p = p_in;
    if (!p.frame) p.att_slots = 0;               // prefix-only run (the fused backward of long rays): no attenuation table
    int wpb = warps_per_block(p.total_rays);
    size_t smem = ((size_t)p.att_slots + (size_t)wpb * FWD_SMEM_PER_WARP) * sizeof(float);
    unsigned grid = (unsigned)((p.total_rays + wpb - 1) / wpb);
    DIFFUS_DISPATCH(auto k = render_fwd_kernel<S_, L_, P64_>; cudaError_t e = ensure_smem(k, smem, 28 / wpb);
                    if (e != cudaSuccess) return e; return launch_kernel(k, grid, wpb * 32, smem, st, p))
    return cudaErrorInvalidValue;
}

template <int S_, int L_, bool P64_, int LOSS>
static cudaError_t launch_bwd_g(const RenderParams& p, bool pg, bool vg, unsigned grid, int threads, size_t smem,
                                cudaStream_t st) {
    constexpr bool TRI = S_ == DIFFUS_SAMPLER_TRILINEAR;
#define DIFFUS_BWD_GO(PG, VG)                                                                                         \
    {                                                                                                                 \
        /* the one-pass specialisations exist for float32 poses only (build time); the WIDE sweep serves the pose */   \
        /* gradient alone and, under MSE, the volume gradient alone */                                                \
        constexpr bool WIDE_ = !P64_ && ((TRI && PG && !VG) || (VG && !PG && LOSS == LOSS_MSE));                      \
        constexpr bool COOP_ = !P64_ && TRI && PG && !VG;                                                             \
        if (WIDE_ && p.Sout <= PREFIX_STRIDE && p.Sout > BwdGeo::SEG) {                                               \
            auto k = render_bwd_kernel<S_, L_, false, PG, VG, LOSS, true, WIDE_>;                                     \
            cudaError_t e = ensure_smem(k, smem, WIDE_CTAS * 4 / (threads / 32));                                     \
            if (e != cudaSuccess) return e;                                                                           \
            return launch_kernel(k, grid, threads, smem, st, p);                                                      \
        }                                                                                                             \
        if (!P64_ && p.Sout <= PREFIX_STRIDE) {                                                                       \
            auto k = render_bwd_kernel<S_, L_, false, PG, VG, LOSS, true>;                                            \
            cudaError_t e = ensure_smem(k, smem, ((VG) ? 16 : 20) / (threads / 32));                                  \
            if (e != cudaSuccess) return e;                                                                           \
            return launch_kernel(k, grid, threads, smem, st, p);                                                      \
        }                                                                                                             \
        if (render_bwd_is_coop(p.Sout, p.total_rays, S_, P64_, PG, VG)) { /* rays of 2..4 passes (config 5: 4): one ray per CTA, no pre-pass */ \
            auto k = render_bwd_kernel<S_, L_, false, PG, VG, LOSS, false, COOP_, COOP_>;                             \
            const int nw_ = (p.Sout + PREFIX_STRIDE - 1) / PREFIX_STRIDE;       /* 2, 3 or 4 warps: 8, 5 or 4 CTAs per SM */ \
            const size_t smem_ = ((size_t)p.att_slots_padded + (size_t)nw_ * BWD_SMEM_PER_WARP + CoopXch::FLOATS) * sizeof(float); \
            cudaError_t e = ensure_smem(k, smem_, 16 / nw_);                                                          \
            if (e != cudaSuccess) return e;                                                                           \
            return launch_kernel(k, (unsigned)p.total_rays, nw_ * 32, smem_, st, p);                                  \
        }                                                                                                             \
        auto k = render_bwd_kernel<S_, L_, P64_, PG, VG, LOSS, false>;                                                \
        cudaError_t e = ensure_smem(k, smem, 16 / (threads / 32));                                                    \
        if (e != cudaSuccess) return e;                                                                               \
        return launch_kernel(k, grid, threads, smem, st, p);                                                          \
    }
    if (!TRI) pg = false;                      // no pose gradient exists (round+long cuts the graph)
    if (pg && vg) DIFFUS_BWD_GO(TRI, true)
    if (pg) DIFFUS_BWD_GO(TRI, false)
    if (vg) DIFFUS_BWD_GO(false, true)
    DIFFUS_BWD_GO(false, false)                // loss / frame only
#undef DIFFUS_BWD_GO
}

// One CTA per four rays, NOT a persistent grid: a grid sized to the resident CTAs with every warp striding over the
// rays was measured 16 % slower (0.871 vs 0.753 ms).  CTAs that start together stay in step -- all gathering (L1-bound)
// or all sweeping (issue-bound) at once -- while the hardware's staggered CTA launches keep the two phases overlapped.
cudaError_t DIFFUS_BWD_NAME(const RenderParams& p, int sampler, int layout, int pose64, bool pose_grad, bool vol_grad,
                            cudaStream_t st) {
    int wpb = warps_per_block(p.total_rays);
    size_t smem = ((size_t)p.att_slots_padded + (size_t)wpb * BWD_SMEM_PER_WARP) * sizeof(float);
    unsigned grid = (unsigned)((p.total_rays + wpb - 1) / wpb);
    const bool mse = p.target != nullptr;
    DIFFUS_DISPATCH(if (mse) return launch_bwd_g<S_, L_, P64_, LOSS_MSE>(p, pose_grad, vol_grad, grid, wpb * 32, smem, st);
                    return launch_bwd_g<S_, L_, P64_, LOSS_GRAD>(p, pose_grad, vol_grad, grid, wpb * 32, smem, st))
    return cudaErrorInvalidValue;
}

#else  // !DIFFUS_LAYOUT_SLICE: the dispatching entry points and the echo-only launchers

cudaError_t launch_render_fwd(const RenderParams& p, int sampler, int layout, int pose64, cudaStream_t st) {
    switch (layout) {
        case DIFFUS_LAYOUT_LINEAR: return launch_render_fwd_layout0(p, sampler, layout, pose64, st);
        case DIFFUS_LAYOUT_BRICK: return launch_render_fwd_layout1(p, sampler, layout, pose64, st);
        case DIFFUS_LAYOUT_QUAD: return launch_render_fwd_layout2(p, sampler, layout, pose64, st);
        case DIFFUS_LAYOUT_TEXTURE: return launch_render_fwd_layout3(p, sampler, layout, pose64, st);
    }
    return cudaErrorInvalidValue;
}

cudaError_t launch_render_bwd(const RenderParams& p, int sampler, int layout, int pose64, bool pose_grad, bool vol_grad,
                              cudaStream_t st) {
    switch (layout) {
        case DIFFUS_LAYOUT_LINEAR: return launch_render_bwd_layout0(p, sampler, layout, pose64, pose_grad, vol_grad, st);
        case DIFFUS_LAYOUT_BRICK: return launch_render_bwd_layout1(p, sampler, layout, pose64, pose_grad, vol_grad, st);
        case DIFFUS_LAYOUT_QUAD: return launch_render_bwd_layout2(p, sampler, layout, pose64, pose_grad, vol_grad, st);
        case DIFFUS_LAYOUT_TEXTURE: return launch_render_bwd_layout3(p, sampler, layout, pose64, pose_grad, vol_grad, st);
    }
    return cudaErrorInvalidValue;
}

cudaError_t launch_echo_fwd(const float* refl, int64_t n_rays, int N, float* echo, cudaStream_t st) {
    int wpb = warps_per_block(n_rays);
    size_t smem = (size_t)wpb * 2 * FwdGeo::OBUF * sizeof(float);
    return launch_kernel(echo_fwd_kernel, (unsigned)((n_rays + wpb - 1) / wpb), wpb * 32, smem, st, refl, n_rays, N, echo);
}

cudaError_t launch_echo_bwd(const float* refl, const float* grad_echo, int64_t n_rays, int N, float* grad_refl,
                            cudaStream_t st) {
    int wpb = warps_per_block(n_rays);
    int nseg = (N + 1 + BwdGeo::SEG - 1) / BwdGeo::SEG;
    size_t smem = (size_t)wpb * (2 * BwdGeo::OBUF + 4 * nseg) * sizeof(float);
    cudaError_t e = ensure_smem(echo_bwd_kernel, smem);
    if (e != cudaSuccess) return e;
    return launch_kernel(echo_bwd_kernel, (unsigned)((n_rays + wpb - 1) / wpb), wpb * 32, smem, st, refl, grad_echo, n_rays, N, grad_refl);
}
#endif  // DIFFUS_LAYOUT_SLICE

}  // namespace diffus
