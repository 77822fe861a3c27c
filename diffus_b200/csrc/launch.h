// Host-side launcher declarations (internal to the shared library).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <atomic>

#include "common.cuh"

namespace diffus {

// Every kernel the library enqueues goes through launch_kernel, so that diffus_launch_count() (api.cu) states how many
// kernels the library launched: memsets and copies are not counted.
extern std::atomic<int64_t> launch_counter;
template <typename K, typename... Args>
static inline cudaError_t launch_kernel(K kernel, dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args... args) {
    kernel<<<grid, block, smem, st>>>(args...);
    launch_counter.fetch_add(1, std::memory_order_relaxed);
    return cudaGetLastError();
}

// 8-way template dispatch on (sampler, layout, pose dtype); the body sees S_, L_, P64_.
#define DIFFUS_DISPATCH_CASE(Sv, Lv, Pv, ...)                              \
    if (sampler == (Sv) && layout == (Lv) && pose64 == ((Pv) ? 1 : 0)) {   \
        constexpr int S_ = (Sv);                                           \
        constexpr int L_ = (Lv);                                           \
        constexpr bool P64_ = (Pv);                                        \
        __VA_ARGS__;                                                       \
    }
// The cases of one layout.  -DDIFFUS_LAYOUT_SLICE=n keeps one layout only: render_kernels.cu is compiled once per layout,
// in parallel (build.py).
#define DIFFUS_LAYOUT_CASES(Lv, ...)                                        \
    DIFFUS_DISPATCH_CASE(DIFFUS_SAMPLER_NEAREST, Lv, false, __VA_ARGS__)    \
    DIFFUS_DISPATCH_CASE(DIFFUS_SAMPLER_NEAREST, Lv, true, __VA_ARGS__)     \
    DIFFUS_DISPATCH_CASE(DIFFUS_SAMPLER_TRILINEAR, Lv, false, __VA_ARGS__)  \
    DIFFUS_DISPATCH_CASE(DIFFUS_SAMPLER_TRILINEAR, Lv, true, __VA_ARGS__)
#if !defined(DIFFUS_LAYOUT_SLICE) || DIFFUS_LAYOUT_SLICE == 0
#define DIFFUS_DISPATCH_L0(...) DIFFUS_LAYOUT_CASES(DIFFUS_LAYOUT_LINEAR, __VA_ARGS__)
#else
#define DIFFUS_DISPATCH_L0(...)
#endif
#if !defined(DIFFUS_LAYOUT_SLICE) || DIFFUS_LAYOUT_SLICE == 1
#define DIFFUS_DISPATCH_L1(...) DIFFUS_LAYOUT_CASES(DIFFUS_LAYOUT_BRICK, __VA_ARGS__)
#else
#define DIFFUS_DISPATCH_L1(...)
#endif
#if !defined(DIFFUS_LAYOUT_SLICE) || DIFFUS_LAYOUT_SLICE == 2
#define DIFFUS_DISPATCH_L2(...) DIFFUS_LAYOUT_CASES(DIFFUS_LAYOUT_QUAD, __VA_ARGS__)
#else
#define DIFFUS_DISPATCH_L2(...)
#endif
#if !defined(DIFFUS_LAYOUT_SLICE) || DIFFUS_LAYOUT_SLICE == 3
#define DIFFUS_DISPATCH_L3(...) DIFFUS_LAYOUT_CASES(DIFFUS_LAYOUT_TEXTURE, __VA_ARGS__)
#else
#define DIFFUS_DISPATCH_L3(...)
#endif
#define DIFFUS_DISPATCH(...) \
    DIFFUS_DISPATCH_L0(__VA_ARGS__) DIFFUS_DISPATCH_L1(__VA_ARGS__) DIFFUS_DISPATCH_L2(__VA_ARGS__) DIFFUS_DISPATCH_L3(__VA_ARGS__)

// api.cu: kernel attributes are set ONCE per (kernel, device), not on every launch: the largest shared-memory carveout
// and the full 227 KB of opt-in dynamic shared memory.  Two host threads launching the same kernel with different
// sizes can then never lower each other's limit, and the ~2 x 3 us of cudaFuncSetAttribute leave the launch path.
constexpr size_t MAX_DYNAMIC_SMEM = 227 * 1024;
cudaError_t prepare_kernel(const void* kernel, int carveout_pct = 100);
// ctas_per_sm > 0: the kernel's launch bounds fix how many CTAs are resident, so only ctas_per_sm x (smem + 1 KB reserved) of
// shared memory is ever needed; the preferred carveout is set to that (first launch decides) and the remainder of the 256 KB
// stays L1 / texture cache for the gathers.
template <typename K>
static inline cudaError_t ensure_smem(K kernel, size_t smem, int ctas_per_sm = 0) {
    if (smem > MAX_DYNAMIC_SMEM) return cudaErrorInvalidValue;
    int pct = 100;
    if (ctas_per_sm > 0) {
        const size_t need = (size_t)ctas_per_sm * (smem + 1024);
        // ask for the smallest shared-memory configuration of sm_100 that holds `need`.  Measured on B200 (carveout sweep,
        // profiles/r2_carveout.md): the driver rounds percent x 228 KB UP to the next configuration -- 72..82 % give the
        // 196 KB one (ncu: launch__shared_mem_config_size 200.7 KB), 86 % already the full 228 KB -- so the request is the
        // configuration's own size rounded DOWN to a whole percent.
        const size_t sizes_kb[] = {8, 16, 32, 64, 100, 132, 164, 196, 228};
        size_t pick = 228;
        for (size_t kb : sizes_kb)
            if (kb * 1024 >= need) { pick = kb; break; }
        pct = (int)(pick * 100 / 228);
        if (pct > 100) pct = 100;
    }
    return prepare_kernel((const void*)kernel, pct);
}

// Rays of two to four 512-column passes (513..2048 columns) with a pose gradient and no volume gradient go through the COOP form
// of render_bwd_kernel (one ray per CTA, one pass per warp): it needs no forward pre-pass for the 512-column prefixes, so
// DiffusRenderArgs.seg_prefix may be NULL for them.
inline bool render_bwd_is_coop(int Sout, int64_t total_rays, int sampler, bool pose64, bool pose_grad, bool vol_grad) {
    return sampler == DIFFUS_SAMPLER_TRILINEAR && !pose64 && pose_grad && !vol_grad && Sout > PREFIX_STRIDE &&
           Sout <= 4 * PREFIX_STRIDE && total_rays <= 0x7fffffffLL;      // (one CTA per ray)
}

// render_kernels.cu
cudaError_t launch_render_fwd(const RenderParams& p, int sampler, int layout, int pose64, cudaStream_t st);
cudaError_t launch_render_bwd(const RenderParams& p, int sampler, int layout, int pose64, bool pose_grad,
                              bool vol_grad, cudaStream_t st);
// the same for one layout each: four translation units built from render_kernels.cu with -DDIFFUS_LAYOUT_SLICE=n
#define DIFFUS_DECLARE_SLICE(n)                                                                                        \
    cudaError_t launch_render_fwd_layout##n(const RenderParams& p, int sampler, int layout, int pose64, cudaStream_t st); \
    cudaError_t launch_render_bwd_layout##n(const RenderParams& p, int sampler, int layout, int pose64, bool pose_grad, \
                                            bool vol_grad, cudaStream_t st);
DIFFUS_DECLARE_SLICE(0)
DIFFUS_DECLARE_SLICE(1)
DIFFUS_DECLARE_SLICE(2)
DIFFUS_DECLARE_SLICE(3)
int64_t reduce_sum_workspace_bytes();
cudaError_t launch_reduce_sum(const float* partial, int64_t n, float scale, float* out, void* workspace, cudaStream_t st);
bool reduce_rays_and_sum_fits(int64_t n);
cudaError_t launch_reduce_rays_and_sum(const float* src_partial, int64_t n_poses, int64_t n_rays, float* grad_src,
                                       const float* loss_partial, int64_t n, float scale, float* loss_out, cudaStream_t st);
cudaError_t launch_echo_fwd(const float* refl, int64_t n_rays, int N, float* echo, cudaStream_t st);
cudaError_t launch_echo_bwd(const float* refl, const float* grad_echo, int64_t n_rays, int N, float* grad_refl,
                            cudaStream_t st);

// aux_kernels.cu
cudaError_t launch_first_refl_median(const RenderParams& p, int sampler, int layout, int pose64, float* median,
                                     int32_t* tie_count, cudaStream_t st);
cudaError_t launch_median_backward(const RenderParams& p, int sampler, int layout, int pose64,
                                   const int32_t* tie_count, bool pose_grad, bool vol_grad, cudaStream_t st);
cudaError_t launch_ray_indices(const RenderParams& p, int pose64, int64_t* x, int64_t* y, int64_t* z, cudaStream_t st);
cudaError_t launch_trace_values(const RenderParams& p, int sampler, int layout, int pose64, float* out, cudaStream_t st);
cudaError_t launch_sample_points(const RenderParams& p, int sampler, int layout, const float* pts, int64_t n, float* val,
                                 int64_t* x, int64_t* y, int64_t* z, cudaStream_t st);
cudaError_t launch_trace_values_bwd(const RenderParams& p, int sampler, int layout, int pose64, const float* gval,
                                    bool pose_grad, bool vol_grad, cudaStream_t st);
cudaError_t launch_reduce_rays(const float* partial, int64_t n_poses, int64_t n_rays, float* out, cudaStream_t st);
cudaError_t launch_cone_directions(const double* median, int64_t n_poses, int64_t n_rays, double opening_angle,
                                   float* out, cudaStream_t st);
cudaError_t launch_fan_directions(const float* median, const float* hint, int64_t n_poses, int64_t n_rays, double angle,
                                  float* out, cudaStream_t st);
cudaError_t launch_fan_directions_bwd(const float* median, const float* hint, const float* grad_dirs, int64_t n_poses,
                                      int64_t n_rays, double angle, float* grad_median, float* grad_hint, cudaStream_t st);
cudaError_t launch_probe_rays(int kind, const float* centre, const float* median, const float* hint, int64_t n_poses, int64_t n_rays,
                              double angle, double radius, double width, float* origins, float* dirs, cudaStream_t st);
cudaError_t launch_probe_rays_bwd(int kind, const float* centre, const float* median, const float* hint, const float* grad_origins,
                                  const float* grad_dirs, int64_t n_poses, int64_t n_rays, double angle, double radius, double width,
                                  float* grad_centre, float* grad_median, float* grad_hint, cudaStream_t st);
cudaError_t launch_to_bricks(const float* linear, const int32_t dim[3], float* bricks, cudaStream_t st);
cudaError_t launch_from_bricks(const float* bricks, const int32_t dim[3], float* linear, cudaStream_t st);
cudaError_t launch_to_quads(const float* linear, const int32_t dim[3], float* quads, cudaStream_t st);
cudaError_t launch_gather_probe(const float* buf, int64_t n_floats, int reads, int64_t n_threads, uint32_t seed, float* sink,
                                cudaStream_t st);

// gn_kernels.cu: the Gauss-Newton system of each pose (trilinear sampler, float32 poses); partial holds 32 floats per ray,
// med_tan 6 floats per pose (start > 0 only).  pivot (3 doubles per pose, from launch_gn_pivot) is given for per-ray origins
// only, and selects the instantiations that rotate about it; NULL = one source per pose.
// The lever of the twist: about each pose's source, about each pose's pivot (per-ray origins), about one pivot for the sweep.
enum GnLever { GN_LEVER_SOURCE = 0, GN_LEVER_POSE = 1, GN_LEVER_SWEEP = 2 };
cudaError_t launch_gn_pivot(const float* sources, int64_t n_poses, int64_t n_rays, double* pivot, cudaStream_t st);
cudaError_t launch_gn_median_tangent(const RenderParams& p, int layout, int lever, const int32_t* tie_count, const double* pivot,
                                     float* med_tan, cudaStream_t st);
cudaError_t launch_render_gn(const RenderParams& p, int layout, const float* med_tan, const double* pivot, float* partial, float* loss,
                             float* jtr, float* jtj, cudaStream_t st);
// Tracked sweeps: ONE system (double loss, jtr (6), jtj (6x6)) of a twist about the one pivot (3 doubles) shared by all poses.
// range_ws holds gn_sweep_ranges(P*R) * 32 doubles; launch_gn_sweep_pivot writes the mean of n_rows origins (3 floats each) to
// pivot, using the same workspace.
int64_t gn_sweep_ranges(int64_t rows);
cudaError_t launch_gn_sweep_pivot(const float* origins, int64_t n_rows, double* range_ws, double* pivot, cudaStream_t st);
cudaError_t launch_render_gn_sweep(const RenderParams& p, int layout, const float* med_tan, const double* pivot, float* partial,
                                   double* range_ws, double* loss, double* jtr, double* jtj, cudaStream_t st);

// smooth_kernels.cu: scipy.ndimage.gaussian_filter(mode='nearest') of a (D,H,W) float32 volume in three separable passes,
// radius r = int(truncate sigma + 0.5) <= BLUR_MAX_RADIUS (r = 0: a copy); dst and scratch hold D*H*W floats each
constexpr int BLUR_MAX_RADIUS = 64;
cudaError_t launch_gaussian_blur(const float* src, const int32_t dim[3], float sigma, int r, float* dst, float* scratch,
                                 cudaStream_t st);

// splat_kernels.cu
int64_t splat_workspace_bytes(int H, int W);
cudaError_t launch_splat_fwd(const float* c0, const float* c1, const float* c2, const float* val, int64_t n, int H, int W,
                             float sigma, float* out, void* ws, cudaStream_t st);
cudaError_t launch_splat_bwd(const float* c0, const float* c1, const float* c2, const float* val, int64_t n, int H, int W,
                             float sigma, const float* grad_out, float* grad_val, void* ws, cudaStream_t st);

// preprocess_kernels.cu
cudaError_t launch_brain_mask(const float* volume, const int32_t dim[3], float threshold, int iterations, uint8_t* mask,
                              uint8_t* scratch, cudaStream_t st);
cudaError_t launch_masked_zscore(const float* volume, const uint8_t* mask, int64_t n, float* out, void* ws, cudaStream_t st);

// train_kernels.cu
cudaError_t launch_adam_step(float* params, const float* grads, float* state, int64_t n, float lr, float beta1, float beta2,
                             float eps, float weight_decay, float grad_scale, cudaStream_t st);
cudaError_t launch_volume_slice(float* vol, const int32_t dim[3], int layout, int axis, int index, float* slice, bool scatter,
                                cudaStream_t st);
cudaError_t launch_conv1d_rows(const float* in, int64_t rows, int n_in, const float* w, int taps, int pad, int flip, float* out,
                               int n_out, cudaStream_t st);
cudaError_t launch_rotate_apex(const float* x, const float* z, int64_t n, float cos_a, float sin_a, float shift, float apex0,
                               float apex1, float* xr, float* zr, cudaStream_t st);
cudaError_t launch_log_compress_fwd(const float* x, int64_t n, float* out, float* max_out, cudaStream_t st);
cudaError_t launch_log_compress_bwd(const float* x, const float* gout, int64_t n, float* gx, cudaStream_t st);
cudaError_t launch_rf_to_bmode(const float* rf, int64_t n_rays, int S, const float* g, float* out, void* workspace, cudaStream_t st);

// loss_kernels.cu
cudaError_t launch_masked_mse_edge_fwd(const float* a, const float* b, const uint8_t* mask, int H, int W, float edge_weight,
                                       float* stats, cudaStream_t st);
cudaError_t launch_masked_mse_edge_bwd(const float* a, const float* b, const uint8_t* mask, int H, int W, float edge_weight,
                                       const float* stats, const float* grad_loss, float* ga, cudaStream_t st);
int64_t ssim_workspace_bytes(int H, int W, int K);
cudaError_t launch_ssim_fwd(const float* s, const float* y, int H, int W, int K, float sigma, float k1, float k2, int normalize,
                            float* loss, void* workspace, cudaStream_t st);
cudaError_t launch_ssim_bwd(const float* s, const float* y, int H, int W, int K, float sigma, int normalize, const float* grad_loss,
                            float* grad_s, void* workspace, cudaStream_t st);

// mlp_kernels.cu
cudaError_t launch_mlp_fwd(const float* params, const float* x, const uint8_t* mask, int64_t n, float out_scale,
                           float fill, float* out, cudaStream_t st);
int64_t mlp_bwd_workspace_bytes(int64_t n);
// gate: NULL, or a device int; the kernels return at once when it reads 0 (the fallback behind the piecewise-linear path)
cudaError_t launch_mlp_bwd(const float* params, const float* x, const uint8_t* mask, const float* grad_out, int64_t n,
                           float out_scale, float* grad_params, void* workspace, const int* gate, cudaStream_t st);
// mlp_pwl_kernels.cu: the scalar-input MLP as a piecewise-linear table
int64_t mlp_pwl_bwd_workspace_bytes(int64_t n);
cudaError_t launch_mlp_pwl_fwd(const float* params, const float* x, const uint8_t* mask, int64_t n, float out_scale, float fill,
                               float* out, cudaStream_t st);
cudaError_t launch_mlp_pwl_dx(const float* params, const float* x, const uint8_t* mask, const float* grad_out, int64_t n,
                              float out_scale, float* grad_x, cudaStream_t st);
cudaError_t launch_mlp_pwl_bwd(const float* params, const float* x, const uint8_t* mask, const float* grad_out, int64_t n,
                               float out_scale, float* grad_params, void* workspace, cudaStream_t st);

}  // namespace diffus
