// MRI -> impedance MLP (reference src/impedance.py:6-17): Linear(1,32)-ReLU-Linear(32,32)-ReLU-Linear(32,1)
// evaluated over a whole volume, and its weight gradient from a d loss / d Z volume.
//
// fp32 on the CUDA cores.  Layers 1 and 3 are an outer and an inner product; only layer 2
// (M x 32 x 32) is a dense contraction, and the 1e-5 frame tolerance rules out TF32/BF16
// single-pass tensor-core math for it (impedances enter the reflection coefficient as a
// difference of nearly equal numbers), see DESIGN.md.
#include "common.cuh"
#include "launch.h"

namespace diffus {

constexpr int H = 32;
// packed parameter offsets (nn.Linear layout, out x in)
constexpr int OFF_W1 = 0, OFF_B1 = 32, OFF_W2 = 64, OFF_B2 = 64 + 1024, OFF_W3 = OFF_B2 + 32, OFF_B3 = OFF_W3 + 32;
static_assert(OFF_B3 + 1 == DIFFUS_MLP_NPARAMS, "parameter packing");

// ---------------------------------------------------------------------------------------
// forward: one thread evaluates VPT voxels; weights broadcast from shared memory as float4
// ---------------------------------------------------------------------------------------
constexpr int FWD_VPT = 2;

__global__ void __launch_bounds__(256) mlp_fwd_kernel(const float* __restrict__ params, const float* __restrict__ x,
                                                      const uint8_t* __restrict__ mask, int64_t n, float out_scale,
                                                      float fill, float* __restrict__ out) {
    __shared__ __align__(16) float w[DIFFUS_MLP_NPARAMS + 3];
    for (int i = threadIdx.x; i < DIFFUS_MLP_NPARAMS; i += blockDim.x) w[i] = params[i];
    __syncthreads();
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t base = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; base < n; base += stride * FWD_VPT) {
        float xv[FWD_VPT];
        bool live[FWD_VPT];
        float h1[FWD_VPT][H];
#pragma unroll
        for (int v = 0; v < FWD_VPT; ++v) {
            int64_t idx = base + v * stride;
            live[v] = idx < n;
            xv[v] = live[v] ? __ldg(x + idx) : 0.f;
        }
#pragma unroll
        for (int i = 0; i < H; ++i) {
            float w1 = w[OFF_W1 + i], b1 = w[OFF_B1 + i];
#pragma unroll
            for (int v = 0; v < FWD_VPT; ++v) h1[v][i] = fmaxf(fmaf(w1, xv[v], b1), 0.f);
        }
        float acc[FWD_VPT];
#pragma unroll
        for (int v = 0; v < FWD_VPT; ++v) acc[v] = w[OFF_B3];
#pragma unroll 4
        for (int j = 0; j < H; ++j) {
            float s[FWD_VPT];
#pragma unroll
            for (int v = 0; v < FWD_VPT; ++v) s[v] = w[OFF_B2 + j];
            const float4* row = (const float4*)(w + OFF_W2 + j * H);
#pragma unroll
            for (int i4 = 0; i4 < H / 4; ++i4) {
                float4 q = row[i4];
#pragma unroll
                for (int v = 0; v < FWD_VPT; ++v) {
                    s[v] = fmaf(q.x, h1[v][4 * i4], s[v]);
                    s[v] = fmaf(q.y, h1[v][4 * i4 + 1], s[v]);
                    s[v] = fmaf(q.z, h1[v][4 * i4 + 2], s[v]);
                    s[v] = fmaf(q.w, h1[v][4 * i4 + 3], s[v]);
                }
            }
            float w3 = w[OFF_W3 + j];
#pragma unroll
            for (int v = 0; v < FWD_VPT; ++v) acc[v] = fmaf(w3, fmaxf(s[v], 0.f), acc[v]);
        }
#pragma unroll
        for (int v = 0; v < FWD_VPT; ++v) {
            int64_t idx = base + v * stride;
            if (live[v]) out[idx] = (mask && !mask[idx]) ? fill : out_scale * acc[v];
        }
    }
}

cudaError_t launch_mlp_fwd(const float* params, const float* x, const uint8_t* mask, int64_t n, float out_scale,
                           float fill, float* out, cudaStream_t st) {
    int64_t want = (n + 256 * FWD_VPT - 1) / (256 * FWD_VPT);
    unsigned grid = (unsigned)max((int64_t)1, min(want, (int64_t)148 * 8));
    return launch_kernel(mlp_fwd_kernel, grid, 256, 0, st, params, x, mask, n, out_scale, fill, out);
}

// ---------------------------------------------------------------------------------------
// backward: a warp owns a tile of 32 voxels.
//   phase A (lane = voxel)      : h1 = relu(W1 x + b1)                     -> smem tile
//   phase B (lane = unit j)     : h2_j, dh2_j = g W3_j [h2_j > 0]          -> smem tile; dW3, db2
//   phase C (lane = unit i)     : dW2[:, i] += dh2 h1_i ; dh1_i ; db1, dW1
// Every lane keeps its slice of the gradient in registers for the whole kernel; blocks
// write their partial 1153-vector once and a second kernel sums the blocks in fixed
// order (atomic-free, deterministic).  Tiles whose upstream gradient is all zero (voxels no
// ray touched, or masked) are skipped.
// ---------------------------------------------------------------------------------------
constexpr int BWD_WARPS = 4;     // 2 x 18 KB of tiles: stays under the 48 KB static limit
constexpr int TILE_LD = H + 4;     // padded row: float4 reads stay aligned, rows land on distinct banks

__global__ void __launch_bounds__(BWD_WARPS * 32) mlp_bwd_kernel(const float* __restrict__ params, const float* __restrict__ x,
                                                                 const uint8_t* __restrict__ mask,
                                                                 const float* __restrict__ grad_out, int64_t n,
                                                                 float out_scale, float* __restrict__ block_partials,
                                                                 const int* __restrict__ gate) {
    if (gate && *gate == 0) return;          // fallback launch behind the piecewise-linear path: not needed
    __shared__ __align__(16) float h1_tile[BWD_WARPS][32 * TILE_LD];
    __shared__ __align__(16) float dh2_tile[BWD_WARPS][32 * TILE_LD];
    __shared__ float xs[BWD_WARPS][32], gs[BWD_WARPS][32];
    __shared__ float red[DIFFUS_MLP_NPARAMS];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    float* h1t = h1_tile[warp];
    float* d2t = dh2_tile[warp];

    float w2_row[H], w2_col[H];                       // W2[lane][:] and W2[:][lane]
#pragma unroll
    for (int i = 0; i < H; ++i) {
        w2_row[i] = __ldg(params + OFF_W2 + lane * H + i);
        w2_col[i] = __ldg(params + OFF_W2 + i * H + lane);
    }
    const float w1 = __ldg(params + OFF_W1 + lane), b1 = __ldg(params + OFF_B1 + lane);
    const float b2 = __ldg(params + OFF_B2 + lane), w3 = __ldg(params + OFF_W3 + lane);

    float g_w2[H];                                    // d W2[j][lane], j = 0..31
#pragma unroll
    for (int j = 0; j < H; ++j) g_w2[j] = 0.f;
    float g_w1 = 0.f, g_b1 = 0.f, g_b2 = 0.f, g_w3 = 0.f, g_b3 = 0.f;

    const int64_t n_tiles = (n + 31) / 32;
    const int64_t warp_global = (int64_t)blockIdx.x * BWD_WARPS + warp, n_warps = (int64_t)gridDim.x * BWD_WARPS;
    for (int64_t tile = warp_global; tile < n_tiles; tile += n_warps) {
        int64_t idx = tile * 32 + lane;
        float g = 0.f, xv = 0.f;
        if (idx < n) {
            g = __ldg(grad_out + idx) * out_scale;
            if (mask && !mask[idx]) g = 0.f;
            xv = __ldg(x + idx);
        }
        if (__ballot_sync(FULL, g != 0.f) == 0u) continue;
        // phase A: this lane's voxel, all 32 hidden units -> row `lane` of the tile
        xs[warp][lane] = xv;
        gs[warp][lane] = g;
        g_b3 += g;
#pragma unroll
        for (int i = 0; i < H; ++i) {
            float w1i = __shfl_sync(FULL, w1, i), b1i = __shfl_sync(FULL, b1, i);
            h1t[lane * TILE_LD + i] = fmaxf(fmaf(w1i, xv, b1i), 0.f);
        }
        __syncwarp();
        // phase B: lane = unit j of layer 2.  Four voxels per iteration with split accumulators: the dot
        // products are 32 dependent FMAs each, so without this the FMA pipe idles on its own latency.
        for (int v = 0; v < 32; v += 4) {
            float sa[4], sb[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) { sa[u] = b2; sb[u] = 0.f; }
#pragma unroll
            for (int i4 = 0; i4 < H / 4; ++i4) {
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    float4 q = ((const float4*)(h1t + (v + u) * TILE_LD))[i4];
                    sa[u] = fmaf(w2_row[4 * i4], q.x, sa[u]);
                    sb[u] = fmaf(w2_row[4 * i4 + 1], q.y, sb[u]);
                    sa[u] = fmaf(w2_row[4 * i4 + 2], q.z, sa[u]);
                    sb[u] = fmaf(w2_row[4 * i4 + 3], q.w, sb[u]);
                }
            }
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                float s = sa[u] + sb[u];
                float gv = gs[warp][v + u];
                float h2 = fmaxf(s, 0.f);
                float dh2 = (s > 0.f) ? gv * w3 : 0.f;
                g_w3 = fmaf(gv, h2, g_w3);
                g_b2 += dh2;
                d2t[(v + u) * TILE_LD + lane] = dh2;
            }
        }
        __syncwarp();
        // phase C: lane = unit i of layer 1 (two voxels per iteration for the same reason)
        for (int v = 0; v < 32; v += 2) {
            float h1a = h1t[v * TILE_LD + lane], h1b = h1t[(v + 1) * TILE_LD + lane];
            const float4* rowa = (const float4*)(d2t + v * TILE_LD);
            const float4* rowb = (const float4*)(d2t + (v + 1) * TILE_LD);
            float da0 = 0.f, da1 = 0.f, db0 = 0.f, db1 = 0.f;
#pragma unroll
            for (int j4 = 0; j4 < H / 4; ++j4) {
                float4 qa = rowa[j4], qb = rowb[j4];
                g_w2[4 * j4] = fmaf(qb.x, h1b, fmaf(qa.x, h1a, g_w2[4 * j4]));
                g_w2[4 * j4 + 1] = fmaf(qb.y, h1b, fmaf(qa.y, h1a, g_w2[4 * j4 + 1]));
                g_w2[4 * j4 + 2] = fmaf(qb.z, h1b, fmaf(qa.z, h1a, g_w2[4 * j4 + 2]));
                g_w2[4 * j4 + 3] = fmaf(qb.w, h1b, fmaf(qa.w, h1a, g_w2[4 * j4 + 3]));
                da0 = fmaf(qa.x, w2_col[4 * j4], da0);
                da1 = fmaf(qa.y, w2_col[4 * j4 + 1], da1);
                da0 = fmaf(qa.z, w2_col[4 * j4 + 2], da0);
                da1 = fmaf(qa.w, w2_col[4 * j4 + 3], da1);
                db0 = fmaf(qb.x, w2_col[4 * j4], db0);
                db1 = fmaf(qb.y, w2_col[4 * j4 + 1], db1);
                db0 = fmaf(qb.z, w2_col[4 * j4 + 2], db0);
                db1 = fmaf(qb.w, w2_col[4 * j4 + 3], db1);
            }
            float dh1a = (h1a > 0.f) ? da0 + da1 : 0.f, dh1b = (h1b > 0.f) ? db0 + db1 : 0.f;
            g_b1 += dh1a + dh1b;
            g_w1 = fmaf(dh1b, xs[warp][v + 1], fmaf(dh1a, xs[warp][v], g_w1));
        }
        __syncwarp();
    }
    // block reduction in a fixed order (warp 0 first), then one partial vector per block
    g_b3 = warp_sum(g_b3);
    for (int i = threadIdx.x; i < DIFFUS_MLP_NPARAMS; i += blockDim.x) red[i] = 0.f;
    __syncthreads();
    for (int wv = 0; wv < BWD_WARPS; ++wv) {
        if (warp == wv) {
            red[OFF_W1 + lane] += g_w1;
            red[OFF_B1 + lane] += g_b1;
            red[OFF_B2 + lane] += g_b2;
            red[OFF_W3 + lane] += g_w3;
#pragma unroll
            for (int j = 0; j < H; ++j) red[OFF_W2 + j * H + lane] += g_w2[j];
            if (lane == 0) red[OFF_B3] += g_b3;
        }
        __syncthreads();
    }
    float* dst = block_partials + (int64_t)blockIdx.x * DIFFUS_MLP_NPARAMS;
    for (int i = threadIdx.x; i < DIFFUS_MLP_NPARAMS; i += blockDim.x) dst[i] = red[i];
}

__global__ void mlp_bwd_reduce_kernel(const float* __restrict__ block_partials, int n_blocks, float* __restrict__ grad_params,
                                      const int* __restrict__ gate) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= DIFFUS_MLP_NPARAMS || (gate && *gate == 0)) return;
    double s = 0.0;                          // a few hundred partials of mixed sign: summed in double, fixed order
    for (int b = 0; b < n_blocks; ++b) s += (double)block_partials[(int64_t)b * DIFFUS_MLP_NPARAMS + i];
    grad_params[i] += (float)s;
}

static int mlp_bwd_blocks(int64_t n) {
    int64_t tiles = (n + 31) / 32;
    int64_t want = (tiles + BWD_WARPS - 1) / BWD_WARPS;
    return (int)max((int64_t)1, min(want, (int64_t)148 * 4));
}

// enough for every path: the piecewise-linear path's tables and partial moments, then the dense block partials (its fallback)
int64_t mlp_bwd_workspace_bytes(int64_t n) {
    return mlp_pwl_bwd_workspace_bytes(n) + (int64_t)mlp_bwd_blocks(n) * DIFFUS_MLP_NPARAMS * sizeof(float);
}

cudaError_t launch_mlp_bwd(const float* params, const float* x, const uint8_t* mask, const float* grad_out, int64_t n,
                           float out_scale, float* grad_params, void* workspace, const int* gate, cudaStream_t st) {
    const int blocks = mlp_bwd_blocks(n);
    cudaError_t e = launch_kernel(mlp_bwd_kernel, blocks, BWD_WARPS * 32, 0, st, params, x, mask, grad_out, n, out_scale,
                                  (float*)workspace, gate);
    if (e != cudaSuccess) return e;
    return launch_kernel(mlp_bwd_reduce_kernel, (DIFFUS_MLP_NPARAMS + 127) / 128, 128, 0, st, (const float*)workspace, blocks, grad_params, gate);
}

}  // namespace diffus
