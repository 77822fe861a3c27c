// Shared device helpers for the DiffUS B-mode renderer kernels (sm_100a).
//
// Column convention used by every kernel in this directory
// --------------------------------------------------------
// A ray has S samples; after the `start` crop there are Sout = S - start output columns
// c = 0..Sout-1, column c belonging to sample k = start + c.  Column c >= 1 owns the
// interface between samples c-1 and c with reflection coefficient
//     r_c = (Z_c - Z_{c-1}) / (Z_{c-1} + Z_c)                (reference src/renderer.py:33,65-68)
// and transfer matrix M_c = [[1 - 2 r_c^2, r_c], [-r_c, 1]]; M_0 = I.  With
//     P_c = M_0 M_1 ... M_c,     echo[c] = P_c[0][1] / P_c[1][1]
// the echo line equals what the reference obtains from one dense linear solve per
// truncation depth (src/renderer.py:367-457); see oracle/port.py::echo_closed_form.
//
// A warp owns a ray and walks it in passes of 512 columns: a gather phase with
// lane = consecutive sample (coalesced stores, few cache lines per load instruction)
// parks impedances in shared memory, a chunk phase with lane = CH consecutive columns does
// the sequential 2x2 products plus one warp-shuffle scan per 32*CH columns, and a tile phase
// writes the result back with lane = consecutive column.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <float.h>

#include "../../include/diffus_b200.h"

namespace diffus {

constexpr unsigned FULL = 0xffffffffu;

// Geometry of one warp pass: 32 lanes x CH consecutive columns per lane.  The forward uses
// CH = 16 (one warp scan per 512 columns); the backward keeps per-column prefixes in
// registers for its reverse sweep and uses CH = 8 to fit 128 registers (4 CTAs per SM) without spills.
template <int CH, int CK = 2>
struct Geo {
    static constexpr int CHUNK = CH;
    static constexpr int CKPT = CK;      // backward: columns between saved prefixes
    static constexpr int SEG = 32 * CH;
    // Padded shared-memory slot: one spare word per 32 columns.  Both access patterns are then conflict free:
    // lane = consecutive column (offset constant over the 32 lanes) and lane = CH consecutive columns
    // (slot CH*l + i sits in bank CH*(l mod 32/CH) + i + l/(32/CH): all 32 distinct).
    __device__ __forceinline__ static int pad(int i) { return i + (i >> 5); }
    static constexpr int ZBUF = (SEG + 2) + (SEG + 2) / 32 + 3;   // slots 0..SEG+1 (slot s = sample c0+s-1)
    static constexpr int OBUF = (SEG + 1) + (SEG + 1) / 32 + 3;   // slots 0..SEG
};
using FwdGeo = Geo<16>;
using BwdGeo = Geo<8, 2>;
// The forward saves its transfer-matrix carry at every PREFIX_STRIDE columns; the backward
// gathers PREFIX_STRIDE columns at a time and walks them as BWD_SUB sub-segments of BwdGeo::SEG.
constexpr int PREFIX_STRIDE = FwdGeo::SEG;

// 2x2 transfer matrix [[a, b], [c, d]] held as its two COLUMNS, (a, c) and (b, d), each in one 64-bit
// register pair: every product below is then a handful of packed FP32 operations (sm_100 `fma.rn.f32x2`
// -> SASS FFMA2 / FMUL2 / FADD2, which take a scalar broadcast operand and negation for free).  A packed
// op rounds each half exactly like its scalar counterpart, so the roundings spelled out here (one multiply
// + one fused multiply-add per entry) are what every kernel walking the same ray reproduces bit for bit.
struct M2 {
    float2 c0, c1;       // c0 = (a, c), c1 = (b, d)
    __device__ __forceinline__ float a() const { return c0.x; }
    __device__ __forceinline__ float b() const { return c1.x; }
    __device__ __forceinline__ float c() const { return c0.y; }
    __device__ __forceinline__ float d() const { return c1.y; }
};
__device__ __forceinline__ float2 bcast(float s) { return make_float2(s, s); }
__device__ __forceinline__ M2 m2_make(float a, float b, float c, float d) { return M2{make_float2(a, c), make_float2(b, d)}; }
__device__ __forceinline__ M2 m2_identity() { return m2_make(1.f, 0.f, 0.f, 1.f); }
__device__ __forceinline__ M2 m2_zero() { return m2_make(0.f, 0.f, 0.f, 0.f); }
// x * y: entry = fma(x_row[0], y_col[0], x_row[1] * y_col[1])
__device__ __forceinline__ M2 m2_mul(const M2& x, const M2& y) {
    return M2{__ffma2_rn(x.c0, bcast(y.c0.x), __fmul2_rn(x.c1, bcast(y.c0.y))),
              __ffma2_rn(x.c0, bcast(y.c1.x), __fmul2_rn(x.c1, bcast(y.c1.y)))};
}
// P * M(r),  M(r) = [[1 - 2 r^2, r], [-r, 1]]
__device__ __forceinline__ M2 m2_mul_interface(const M2& p, float r) {
    float q = __fmaf_rn(-2.f * r, r, 1.f);
    return M2{__ffma2_rn(p.c0, bcast(q), __fmul2_rn(p.c1, bcast(-r))), __ffma2_rn(p.c0, bcast(r), p.c1)};
}
// X * M(r)^T
__device__ __forceinline__ M2 m2_mul_interface_t(const M2& x, float r) {
    float q = __fmaf_rn(-2.f * r, r, 1.f);
    return M2{__ffma2_rn(x.c0, bcast(q), __fmul2_rn(x.c1, bcast(r))), __ffma2_rn(x.c0, bcast(-r), x.c1)};
}
__device__ __forceinline__ M2 m2_transpose(const M2& x) { return m2_make(x.a(), x.c(), x.b(), x.d()); }
__device__ __forceinline__ M2 m2_add(const M2& x, const M2& y) { return M2{__fadd2_rn(x.c0, y.c0), __fadd2_rn(x.c1, y.c1)}; }
__device__ __forceinline__ float2 shfl_up2(float2 v, int d) { return make_float2(__shfl_up_sync(FULL, v.x, d), __shfl_up_sync(FULL, v.y, d)); }
__device__ __forceinline__ float2 shfl_down2(float2 v, int d) { return make_float2(__shfl_down_sync(FULL, v.x, d), __shfl_down_sync(FULL, v.y, d)); }
__device__ __forceinline__ float2 shfl2(float2 v, int src) { return make_float2(__shfl_sync(FULL, v.x, src), __shfl_sync(FULL, v.y, src)); }
__device__ __forceinline__ M2 m2_shfl_up(const M2& x, int d) { return M2{shfl_up2(x.c0, d), shfl_up2(x.c1, d)}; }
__device__ __forceinline__ M2 m2_shfl_down(const M2& x, int d) { return M2{shfl_down2(x.c0, d), shfl_down2(x.c1, d)}; }
__device__ __forceinline__ M2 m2_shfl(const M2& x, int src) { return M2{shfl2(x.c0, src), shfl2(x.c1, src)}; }

// nan_to_num(nan=0) of src/renderer.py:408 (+-inf -> +-FLT_MAX like torch's default)
__device__ __forceinline__ float nan_to_num(float e) {
    if (e != e) return 0.f;
    return fminf(fmaxf(e, -FLT_MAX), FLT_MAX);
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) v += __shfl_xor_sync(FULL, v, d);
    return v;
}

// Sums EIGHT values over the warp with 9 shuffles instead of 40: the first three butterfly steps halve the number of values a
// lane carries (a lane keeps the half its bit selects and sends the other half to its partner), the last two finish the one
// value left.  On return lane l holds the total of value 4 (l & 1) + 2 ((l >> 1) & 1) + ((l >> 2) & 1); warp_sum8_index(l).
__device__ __forceinline__ int warp_sum8_index(int lane) { return ((lane & 1) << 2) | (lane & 2) | ((lane >> 2) & 1); }
__device__ __forceinline__ float warp_sum8(float v[8], int lane) {
    const bool b0 = lane & 1, b1 = lane & 2, b2 = lane & 4;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        const float send = b0 ? v[j] : v[j + 4], keep = b0 ? v[j + 4] : v[j];
        v[j] = keep + __shfl_xor_sync(FULL, send, 1);
    }
#pragma unroll
    for (int j = 0; j < 2; ++j) {
        const float send = b1 ? v[j] : v[j + 2], keep = b1 ? v[j + 2] : v[j];
        v[j] = keep + __shfl_xor_sync(FULL, send, 2);
    }
    const float send = b2 ? v[0] : v[1], keep = b2 ? v[1] : v[0];
    float t = keep + __shfl_xor_sync(FULL, send, 4);
    t += __shfl_xor_sync(FULL, t, 8);
    t += __shfl_xor_sync(FULL, t, 16);
    return t;
}

// ---------------------------------------------------------------------------------------
// volume addressing: offset(i, j, k) = ox(i) + oy(j) + oz(k) in 32-bit element units, so the
// eight corners of a trilinear cell cost six per-axis terms and a handful of adds instead
// of eight full index computations (integer address math was 47 % of the forward's
// instructions in the first profile, profiles/r1_first_ncu.md).
//
// Layouts (include/diffus_b200.h):
//   LINEAR  the torch tensor as is
//   BRICK   4x4x2 voxels per 128-byte line, one float per voxel
//   QUAD    one float4 per voxel holding the voxel and its +j, +k, +j+k neighbours (clamped at the faces),
//           2x2x2 voxels per 128-byte line with the i-pair sharing a 32-byte sector.  A trilinear cell is
//           two 16-byte loads (i0 and i1) instead of eight 4-byte ones: a quarter of the load instructions
//           and L1 tag look-ups for four times the footprint.  Read-only: gradients w.r.t. a QUAD volume
//           are scattered into a BRICK buffer (gsx / gsy below).
//   TEXTURE a layered 2-D CUDA array (layer = p0, y = p1, x = p2) behind a texture object with clamp addressing and
//           point sampling.  A trilinear cell is two `tld4` gathers (the 2x2 (p1, p2) footprint of layer i0 and of
//           layer i1, unfiltered fp32 texels): the texture unit does the address arithmetic and the border clamp,
//           the footprint stays 1x (L2-resident at 256^3, unlike QUAD), and the gathers leave the LSU pipe.
//           `data` carries the cudaTextureObject_t.  Read-only: gradients go to a BRICK buffer like QUAD's.
// ---------------------------------------------------------------------------------------
struct VolumeView {
    const float* data;
    int D, H, W;          // extents along point components 0, 1, 2
    uint32_t sx, sy;      // LINEAR: H*W, W     BRICK: bricks-per-slab*32, bricks-per-row*32    QUAD: same in float4 units (*8)
    uint32_t gsx, gsy;    // strides of the gradient volume: = sx, sy for LINEAR / BRICK, the BRICK strides for QUAD
};

constexpr int BRICK_I = 4, BRICK_J = 4, BRICK_K = 2;   // 32 floats = one 128-byte line
constexpr int QUAD_B = 2;                              // 2x2x2 float4 = one 128-byte line

// layout of the gradient volume that belongs to a gathered layout
template <int LAYOUT>
struct GradLayout {
    static constexpr int value = (LAYOUT == DIFFUS_LAYOUT_QUAD || LAYOUT == DIFFUS_LAYOUT_TEXTURE) ? DIFFUS_LAYOUT_BRICK : LAYOUT;
};

// texel fetches of the TEXTURE layout (x = p2, y = p1, layer = p0; unnormalised coordinates, texel centres at +0.5)
__device__ __forceinline__ cudaTextureObject_t volume_texture(const void* data) { return (cudaTextureObject_t)(uintptr_t)data; }
// The 2x2 (p1, p2) footprint of `layer` that bilinear filtering at texture coordinate (x, y) would blend, unfiltered, in
// tld4's own order: .x = (x0, y1), .y = (x1, y1), .z = (x1, y0), .w = (x0, y0) with x0 = floor(x - 0.5) -- i.e. with
// j = p1 = y and k = p2 = x:  (j1k0, j1k1, j0k1, j0k0), the "cell face" order of tri_combine (no register shuffling between
// the gather and the packed arithmetic).  Clamp addressing supplies the border rule: x = x0 + 1 gives (x0, min(x0 + 1, n - 1)),
// x = 0 gives (0, 0).
__device__ __forceinline__ float4 tex_gather_face(cudaTextureObject_t tex, int layer, float x, float y) {
    float4 r;
    asm volatile("tld4.r.a2d.v4.f32.f32 {%0, %1, %2, %3}, [%4, {%5, %6, %7, %7}];"
                 : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w)
                 : "l"(tex), "r"(layer), "f"(x), "f"(y)
                 : "memory");      // keeps the gathers where the software pipeline puts them (before the previous batch's combine + stores)
    return r;
}
__device__ __forceinline__ float tex_fetch_voxel(cudaTextureObject_t tex, int i, int j, int k) {
    return tex2DLayered<float>(tex, (float)k + 0.5f, (float)j + 0.5f, i);
}

template <int LAYOUT>
__device__ __forceinline__ uint32_t axis_x(uint32_t sx, int i) {
    if (LAYOUT == DIFFUS_LAYOUT_LINEAR) return (uint32_t)i * sx;
    if (LAYOUT == DIFFUS_LAYOUT_BRICK) return (uint32_t)(i >> 2) * sx + ((uint32_t)(i & 3) << 3);
    return (uint32_t)(i >> 1) * sx + (uint32_t)(i & 1);
}
template <int LAYOUT>
__device__ __forceinline__ uint32_t axis_y(uint32_t sy, int j) {
    if (LAYOUT == DIFFUS_LAYOUT_LINEAR) return (uint32_t)j * sy;
    if (LAYOUT == DIFFUS_LAYOUT_BRICK) return (uint32_t)(j >> 2) * sy + ((uint32_t)(j & 3) << 1);
    return (uint32_t)(j >> 1) * sy + ((uint32_t)(j & 1) << 2);
}
template <int LAYOUT>
__device__ __forceinline__ uint32_t axis_z(int k) {
    if (LAYOUT == DIFFUS_LAYOUT_LINEAR) return (uint32_t)k;
    if (LAYOUT == DIFFUS_LAYOUT_BRICK) return ((uint32_t)(k >> 1) << 5) + (uint32_t)(k & 1);
    return ((uint32_t)(k >> 1) << 3) + ((uint32_t)(k & 1) << 1);
}
// element offset in the gathered layout (float units for LINEAR / BRICK, float4 units for QUAD)
template <int LAYOUT>
__device__ __forceinline__ uint32_t voxel_offset(const VolumeView& v, int i, int j, int k) {
    return axis_x<LAYOUT>(v.sx, i) + axis_y<LAYOUT>(v.sy, j) + axis_z<LAYOUT>(k);
}

// element offset in the gradient volume that belongs to a LAYOUT volume
template <int LAYOUT>
__device__ __forceinline__ uint32_t grad_offset(const VolumeView& v, int i, int j, int k) {
    constexpr int GL = GradLayout<LAYOUT>::value;
    return axis_x<GL>(v.gsx, i) + axis_y<GL>(v.gsy, j) + axis_z<GL>(k);
}

// a / b without the IEEE slow path (<= 2 ulp): the reference's own float32 run is ~1e-5 of
// peak away from its float64 run, so correctly-rounded division buys nothing here
// One MUFU.RCP, no range fix-ups (__fdividef adds a scaling branch for |b| > 2^126, never met here).
__device__ __forceinline__ float fast_rcp(float b) {
    float r;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(b));
    return r;
}
__device__ __forceinline__ float fast_div(float a, float b) { return a * fast_rcp(b); }
// echo of a prefix: P[0][1] / P[1][1] (same rounding in the forward and in the fused backward)
__device__ __forceinline__ float echo_of(float pb, float inv_pd) { return __fmul_rn(pb, inv_pd); }

// ---------------------------------------------------------------------------------------
// ray points:  p = source + k * direction   (src/renderer.py:119-124), cast to float32 (:751)
// The reference multiplies and adds in separate roundings; no FMA contraction here so the
// nearest-voxel indices are bit-identical.
// ---------------------------------------------------------------------------------------
template <bool POSE64>
struct RaySetup;

// Float32 poses: the ray's origin is at src + pose * src_pose_stride + ray * src_ray_stride -- (3, 0) for one source per pose,
// (3R, 3) for one origin per ray (DIFFUS_POSE_F32_PER_RAY: linear and convex array probes).
template <>
struct RaySetup<false> {
    float s[3], d[3];
    __device__ __forceinline__ void load(const void* src, const void* dir, int64_t pose, int64_t ray,
                                         int64_t src_pose_stride, int64_t src_ray_stride, int64_t dir_pose_stride, int) {
        const float* sp = (const float*)src + pose * src_pose_stride + ray * src_ray_stride;
        const float* dp = (const float*)dir + pose * dir_pose_stride + ray * 3;
#pragma unroll
        for (int a = 0; a < 3; ++a) { s[a] = __ldg(sp + a); d[a] = __ldg(dp + a); }
    }
    __device__ __forceinline__ float coord(int a, int k) const {
        return __fadd_rn(s[a], __fmul_rn((float)k, d[a]));
    }
};

template <>
struct RaySetup<true> {
    double s[3], d[3];
    int product_f32;
    __device__ __forceinline__ void load(const void* src, const void* dir, int64_t pose, int64_t ray,
                                         int64_t, int64_t, int64_t dir_pose_stride, int prod_f32) {
        const double* sp = (const double*)src + pose * 3;
        const double* dp = (const double*)dir + pose * dir_pose_stride + ray * 3;
#pragma unroll
        for (int a = 0; a < 3; ++a) { s[a] = __ldg(sp + a); d[a] = __ldg(dp + a); }
        product_f32 = prod_f32;
    }
    __device__ __forceinline__ float coord(int a, int k) const {
        double prod = product_f32 ? (double)__fmul_rn((float)k, (float)d[a]) : __dmul_rn((double)k, d[a]);
        return (float)__dadd_rn(s[a], prod);
    }
};

// ---------------------------------------------------------------------------------------
// samplers
// ---------------------------------------------------------------------------------------
__device__ __forceinline__ int nearest_index(float p, int n) {
    int i = __float2int_rn(p);                 // round half to even == torch.round; saturating
    return min(max(i, 0), n - 1);
}

struct TriCell {       // clamp-then-floor cell of a trilinear sample, grid_sample border semantics
    int i0[3], i1[3];
    float f[3];        // fraction in [0, 1)
};

// grid_sample(padding_mode='border', align_corners=True) along one axis: the coordinate clamps to [0, n - 1], the cell is
// [floor, floor + 1] and the derivative w.r.t. the coordinate is ZERO at or beyond a face (p <= 0 or p >= n - 1).
// A clamped coordinate has fraction exactly 0, so the value never needs to know; the derivative is the difference of the
// cell's two faces across the axis, and it vanishes by itself when both faces are the SAME voxels:
//   * at the top face floor = n - 1 and i1 = min(i0 + 1, n - 1) = i0 already;
//   * at the bottom face (p <= 0) the cell is collapsed explicitly, i1 = i0 = 0 -- one compare and one select per axis, and
//     only in kernels that form the spatial gradient (COLLAPSE).  No per-sample "inside" flags travel anywhere.
// (A volume holding inf / NaN voxels would turn 0 into NaN there; such a volume has no meaningful frame either.)
template <bool COLLAPSE = false>
__device__ __forceinline__ void tri_axis(float p, int n, int& i0, int& i1, float& f) {
    float hi = (float)(n - 1);
    float pc = fminf(fmaxf(p, 0.f), hi);
    float fl = floorf(pc);
    f = pc - fl;
    i0 = (int)fl;
    i1 = min(i0 + 1, n - 1);
    if (COLLAPSE) i1 = (p > 0.f) ? i1 : i0;
}

// The same for an axis addressed through the texture unit.  The tld4 coordinate whose footprint is (fl, fl + 1) is fl + 1, and
// CLAMP ADDRESSING does the rest: no explicit clamp of the coordinate is needed.  Beyond the top face both texels clamp to
// n - 1, below the bottom face both clamp to 0 -- the two corners are then the same texel, so whatever fraction p - floor(p)
// says, the value is that texel and the derivative 0.  Only p <= 0 with floor(p) = 0 (p = 0 exactly, where grid_sample's
// derivative is 0 but the cell (0, 1) has one) needs the collapse: coordinate 0 selects the footprint (-1, 0) = (0, 0).
template <bool COLLAPSE>
__device__ __forceinline__ void tri_axis_tex(float p, int n, float& coord, float& f) {
    (void)n;
    const float fl = floorf(p);
    f = p - fl;
    coord = fl + 1.0f;
    if (COLLAPSE) coord = (p > 0.f) ? coord : 0.f;
}

// QUAD elements carry their +j / +k neighbours inside the element, so the bottom-face cell cannot be collapsed by an index:
// there "at or below the bottom face" travels in the sign bit of f (-0.0f interpolates exactly like +0.0f)
__device__ __forceinline__ bool tri_inside(float f) { return (__float_as_uint(f) >> 31) == 0u; }
__device__ __forceinline__ void tri_axis_flag(float p, int n, int& i0, float& f) {
    float hi = (float)(n - 1);
    float pc = fminf(fmaxf(p, 0.f), hi);
    float fl = floorf(pc);
    f = (p > 0.f) ? pc - fl : -0.f;
    i0 = (int)fl;
}

// offsets of the eight corners in the layout of the GRADIENT volume (also the gathered one for LINEAR / BRICK)
template <int GLAYOUT>
__device__ __forceinline__ void tri_offsets(const VolumeView& v, const TriCell& c, uint32_t off[8]) {
    uint32_t x0 = axis_x<GLAYOUT>(v.gsx, c.i0[0]), x1 = axis_x<GLAYOUT>(v.gsx, c.i1[0]);
    uint32_t y0 = axis_y<GLAYOUT>(v.gsy, c.i0[1]), y1 = axis_y<GLAYOUT>(v.gsy, c.i1[1]);
    uint32_t z0 = axis_z<GLAYOUT>(c.i0[2]), z1 = axis_z<GLAYOUT>(c.i1[2]);
    uint32_t a00 = x0 + y0, a01 = x0 + y1, a10 = x1 + y0, a11 = x1 + y1;
    off[0] = a00 + z0; off[1] = a00 + z1; off[2] = a01 + z0; off[3] = a01 + z1;
    off[4] = a10 + z0; off[5] = a10 + z1; off[6] = a11 + z0; off[7] = a11 + z1;
}

// Value (and optionally the spatial gradient) of the border-clamped trilinear interpolant from the two faces of the
// cell: q0 = face i0, q1 = face i1, each in tld4 order (j1k0, j1k1, j0k1, j0k0) -- the pairs (x, y) and (z, w) are what the
// packed FP32 instructions take as they come out of the gather.  Interpolation is a + f (b - a) along i (4 wide), then j
// (2 wide: the j0 pair enters with its halves swapped, a free operand modifier), then k; the derivative along an axis is the
// difference of the two faces across it, interpolated along the other two.  FLAGS: bottom-face flags in the sign of f[1], f[2].
template <bool GRAD, bool FLAGS = false>
__device__ __forceinline__ float tri_combine(const float4& q0, const float4& q1, const float f[3], float g[3]) {
    const float2 a0 = make_float2(q0.x, q0.y), b0 = make_float2(q0.z, q0.w);      // face i0: j1 (k0, k1), j0 (k1, k0)
    const float2 da = __fadd2_rn(make_float2(q1.x, q1.y), make_float2(-a0.x, -a0.y));     // d / d i at j1 (k0, k1)
    const float2 db = __fadd2_rn(make_float2(q1.z, q1.w), make_float2(-b0.x, -b0.y));     // d / d i at j0 (k1, k0)
    const float2 fx = bcast(f[0]), fy = bcast(f[1]);
    const float2 la = __ffma2_rn(da, fx, a0), lb = __ffma2_rn(db, fx, b0);        // along i
    const float2 lbs = make_float2(lb.y, lb.x);                                   // j0 (k0, k1)
    const float2 ej = __fadd2_rn(la, make_float2(-lbs.x, -lbs.y));                // d / d j at k0, k1
    const float2 m = __ffma2_rn(ej, fy, lbs);                                     // along j: value at k0, k1
    const float dk = m.y - m.x;
    if (GRAD) {
        const float2 dbs = make_float2(db.y, db.x);
        const float2 di = __ffma2_rn(__fadd2_rn(da, make_float2(-dbs.x, -dbs.y)), fy, dbs);   // d / d i at k0, k1
        g[0] = __fmaf_rn(di.y - di.x, f[2], di.x);
        g[1] = __fmaf_rn(ej.y - ej.x, f[2], ej.x);
        g[2] = dk;
        if (FLAGS) {
            g[1] = tri_inside(f[1]) ? g[1] : 0.f;
            g[2] = tri_inside(f[2]) ? g[2] : 0.f;
        }
    }
    return __fmaf_rn(dk, f[2], m.x);
}

// A sample split into "issue the loads" and "combine", so a gather loop can keep the next
// tile's loads in flight while it combines the current one (software pipelining).
template <int SAMPLER, int LAYOUT>
struct Fetch {
    float4 q0, q1;     // nearest: q0.x only; trilinear: the cell's faces i0 and i1 in tld4 order (see tri_combine)
    float f[3];

    // GRAD: the caller will ask finish<true> for the spatial gradient (the cell is collapsed at the bottom faces)
    template <bool GRAD = false>
    __device__ __forceinline__ void issue(const VolumeView& v, float p0, float p1, float p2) {
        if (SAMPLER == DIFFUS_SAMPLER_NEAREST) {
            int i = nearest_index(p0, v.D), j = nearest_index(p1, v.H), k = nearest_index(p2, v.W);
            if (LAYOUT == DIFFUS_LAYOUT_TEXTURE) {
                q0.x = tex_fetch_voxel(volume_texture(v.data), i, j, k);
            } else {
                const uint32_t off = voxel_offset<LAYOUT>(v, i, j, k);
                q0.x = __ldg(v.data + (LAYOUT == DIFFUS_LAYOUT_QUAD ? (size_t)off * 4 : (size_t)off));
            }
        } else if (LAYOUT == DIFFUS_LAYOUT_TEXTURE) {
            int i0, i1;
            float y, x;
            tri_axis<GRAD>(p0, v.D, i0, i1, f[0]);
            tri_axis_tex<GRAD>(p1, v.H, y, f[1]);
            tri_axis_tex<GRAD>(p2, v.W, x, f[2]);
            const cudaTextureObject_t tex = volume_texture(v.data);
            q0 = tex_gather_face(tex, i0, x, y);
            q1 = tex_gather_face(tex, i1, x, y);
        } else if (LAYOUT == DIFFUS_LAYOUT_QUAD) {
            int i0, i1, j0, k0;
            tri_axis<GRAD>(p0, v.D, i0, i1, f[0]);
            tri_axis_flag(p1, v.H, j0, f[1]);
            tri_axis_flag(p2, v.W, k0, f[2]);
            const uint32_t base = axis_y<LAYOUT>(v.sy, j0) + axis_z<LAYOUT>(k0);
            const float4* q = (const float4*)v.data;
            const float4 e0 = __ldg(q + (base + axis_x<LAYOUT>(v.sx, i0)));      // (j0k0, j1k0, j0k1, j1k1)
            const float4 e1 = __ldg(q + (base + axis_x<LAYOUT>(v.sx, i1)));
            q0 = make_float4(e0.y, e0.w, e0.z, e0.x);
            q1 = make_float4(e1.y, e1.w, e1.z, e1.x);
        } else {
            TriCell c;
            tri_axis<GRAD>(p0, v.D, c.i0[0], c.i1[0], f[0]);
            tri_axis<GRAD>(p1, v.H, c.i0[1], c.i1[1], f[1]);
            tri_axis<GRAD>(p2, v.W, c.i0[2], c.i1[2], f[2]);
            uint32_t x0 = axis_x<LAYOUT>(v.sx, c.i0[0]), x1 = axis_x<LAYOUT>(v.sx, c.i1[0]);
            uint32_t y0 = axis_y<LAYOUT>(v.sy, c.i0[1]), y1 = axis_y<LAYOUT>(v.sy, c.i1[1]);
            uint32_t z0 = axis_z<LAYOUT>(c.i0[2]), z1 = axis_z<LAYOUT>(c.i1[2]);
            uint32_t a00 = x0 + y0, a01 = x0 + y1, a10 = x1 + y0, a11 = x1 + y1;
            q0 = make_float4(__ldg(v.data + (a01 + z0)), __ldg(v.data + (a01 + z1)), __ldg(v.data + (a00 + z1)), __ldg(v.data + (a00 + z0)));
            q1 = make_float4(__ldg(v.data + (a11 + z0)), __ldg(v.data + (a11 + z1)), __ldg(v.data + (a10 + z1)), __ldg(v.data + (a10 + z0)));
        }
    }
    template <bool GRAD>
    __device__ __forceinline__ float finish(float g[3]) const {
        if (SAMPLER == DIFFUS_SAMPLER_NEAREST) {
            if (GRAD) { g[0] = g[1] = g[2] = 0.f; }
            return q0.x;
        } else {
            return tri_combine<GRAD, LAYOUT == DIFFUS_LAYOUT_QUAD>(q0, q1, f, g);
        }
    }
};

template <int SAMPLER, int LAYOUT, bool GRAD>
__device__ __forceinline__ float sample_volume(const VolumeView& v, float p0, float p1, float p2, float g[3]) {
    Fetch<SAMPLER, LAYOUT> fe;
    fe.template issue<GRAD>(v, p0, p1, p2);
    return fe.template finish<GRAD>(g);
}

// kernel parameter block (host fills it from the C-ABI structs)
struct RenderParams {
    VolumeView vol;
    const void* sources;
    const void* directions;
    int64_t dir_pose_stride;
    int64_t src_pose_stride;    // float32 origins: (3, 0) per pose, (3R, 3) per ray; float64 poses are always per pose
    int64_t src_ray_stride;
    int product_f32;
    int64_t n_poses, n_rays, total_rays;
    int S, start, Sout;
    int nprefix;                // saved prefixes per ray: ceil(Sout / PREFIX_STRIDE) - 1
    int att_slots;              // floats reserved at the start of dynamic smem for the attenuation table
    int att_slots_padded;       // same, for the backward's padded table
    float alpha;
    float* frame;
    float* seg_prefix;          // (total_rays, nprefix, 4) or null
    const float* median;        // (P) replacement for r_1 when start > 0, else null
    // backward
    const float* grad_frame;
    float* grad_volume;
    float* grad_src_partial;    // (total_rays, 3); per-ray origins: the caller's grad_sources itself
    float* grad_dir;            // (total_rays, 3)
    float* first_rbar;          // (total_rays) d loss / d (median-replaced r_1), start > 0
    // fused MSE loss (target != null): d loss / d frame = grad_scale * (frame - target)
    const float* target;        // (total_rays, Sout)
    float grad_scale;
    float* loss_partial;        // (total_rays) sum over the ray of (frame - target)^2, or null
};

}  // namespace diffus
