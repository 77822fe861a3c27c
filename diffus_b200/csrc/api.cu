// extern "C" entry points of libdiffus_b200.so (see include/diffus_b200.h).
// Argument validation and parameter packing only; kernels live in the other translation units.
#include <cmath>
#include <mutex>
#include <unordered_map>
#include <unordered_set>

#include "common.cuh"
#include "launch.h"

using namespace diffus;

namespace diffus {
cudaError_t prepare_kernel(const void* kernel, int carveout_pct) {
    static std::mutex mu;
    static std::unordered_map<uint64_t, int> done;   // (kernel, device) -> carveout last set
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    const uint64_t key = (uint64_t)(uintptr_t)kernel * 64u + (uint64_t)dev;
    std::lock_guard<std::mutex> lock(mu);
    auto it = done.find(key);
    if (it != done.end() && it->second == carveout_pct) return cudaSuccess;
    // carveout_pct < 100: the kernel's resident CTAs need less than the whole 228 KB -- the rest stays L1 / texture cache.
    // (Only a different launch geometry of the same kernel changes the value: the common case above is one map look-up.)
    e = cudaFuncSetAttribute(kernel, cudaFuncAttributePreferredSharedMemoryCarveout,
                             carveout_pct >= 100 ? (int)cudaSharedmemCarveoutMaxShared : carveout_pct);
    if (e != cudaSuccess) return e;
    if (it == done.end()) {
        // the opt-in limit covers static + dynamic shared memory: a kernel with static arrays (the median select's
        // histogram) is refused the whole 227 KB as dynamic memory
        cudaFuncAttributes fa;
        e = cudaFuncGetAttributes(&fa, kernel);
        if (e != cudaSuccess) return e;
        e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(MAX_DYNAMIC_SMEM - fa.sharedSizeBytes));
        if (e != cudaSuccess) return e;
    }
    done[key] = carveout_pct;
    return cudaSuccess;
}
}  // namespace diffus

namespace {

inline int64_t align_up(int64_t v, int64_t a) { return (v + a - 1) / a * a; }

int32_t check_volume(const DiffusVolume& v) {
    if (!v.data) return DIFFUS_E_NULL;
    if (v.dim[0] < 1 || v.dim[1] < 1 || v.dim[2] < 1) return DIFFUS_E_SHAPE;
    // 32-bit element offsets (also in the padded brick layout)
    if (((int64_t)v.dim[0] + 3) * ((int64_t)v.dim[1] + 3) * ((int64_t)v.dim[2] + 1) >= ((int64_t)1 << 31)) return DIFFUS_E_UNSUPPORTED;
    if (v.layout != DIFFUS_LAYOUT_LINEAR && v.layout != DIFFUS_LAYOUT_BRICK && v.layout != DIFFUS_LAYOUT_QUAD &&
        v.layout != DIFFUS_LAYOUT_TEXTURE)
        return DIFFUS_E_ENUM;
    if (v.layout == DIFFUS_LAYOUT_TEXTURE && (v.dim[0] > 2048 || v.dim[1] > 32768 || v.dim[2] > 32768)) return DIFFUS_E_UNSUPPORTED;
    if (v.layout == DIFFUS_LAYOUT_QUAD && ((uintptr_t)v.data & 15)) return DIFFUS_E_UNSUPPORTED;   // float4 loads
    return DIFFUS_OK;
}

bool pose_dtype_ok(int32_t t) { return t == DIFFUS_POSE_F32 || t == DIFFUS_POSE_F64 || t == DIFFUS_POSE_F32_PER_RAY; }
bool per_ray(const DiffusRenderArgs* a) { return a->pose_dtype == DIFFUS_POSE_F32_PER_RAY; }

int32_t check_render(const DiffusRenderArgs* a, bool need_frame) {
    if (!a) return DIFFUS_E_NULL;
    int32_t e = check_volume(a->volume);
    if (e) return e;
    if (!a->sources || !a->directions) return DIFFUS_E_NULL;
    if (need_frame && !a->frame) return DIFFUS_E_NULL;
    if (!pose_dtype_ok(a->pose_dtype)) return DIFFUS_E_ENUM;
    if (a->sampler != DIFFUS_SAMPLER_NEAREST && a->sampler != DIFFUS_SAMPLER_TRILINEAR) return DIFFUS_E_ENUM;
    if (a->n_poses < 1 || a->n_rays < 1 || a->n_samples < 2) return DIFFUS_E_SHAPE;
    if (a->n_samples > 32768) return DIFFUS_E_UNSUPPORTED;           // attenuation table lives in shared memory
    if (a->start < 0 || a->start > a->n_samples - 2) return DIFFUS_E_SHAPE;
    if (a->dir_pose_stride != 0 && a->dir_pose_stride != a->n_rays * 3) return DIFFUS_E_SHAPE;
    if (a->n_poses * a->n_rays >= ((int64_t)1 << 31)) return DIFFUS_E_SHAPE;
    if (a->start > 0 && a->n_rays > 49152) return DIFFUS_E_UNSUPPORTED; // median kernel keeps a pose's rays in shared memory
    return DIFFUS_OK;
}

RenderParams pack(const DiffusRenderArgs* a) {
    RenderParams p{};
    p.vol.data = a->volume.data;
    p.vol.D = a->volume.dim[0];
    p.vol.H = a->volume.dim[1];
    p.vol.W = a->volume.dim[2];
    const uint32_t nbj = (p.vol.H + BRICK_J - 1) / BRICK_J, nbk = (p.vol.W + BRICK_K - 1) / BRICK_K;
    if (a->volume.layout == DIFFUS_LAYOUT_BRICK) {
        p.vol.gsy = p.vol.sy = nbk * 32;
        p.vol.gsx = p.vol.sx = nbj * nbk * 32;
    } else if (a->volume.layout == DIFFUS_LAYOUT_QUAD) {
        const uint32_t nqj = (p.vol.H + QUAD_B - 1) / QUAD_B, nqk = (p.vol.W + QUAD_B - 1) / QUAD_B;
        p.vol.sy = nqk * 8;                 // float4 units
        p.vol.sx = nqj * nqk * 8;
        p.vol.gsy = nbk * 32;               // gradients of a QUAD volume go to a BRICK buffer
        p.vol.gsx = nbj * nbk * 32;
    } else if (a->volume.layout == DIFFUS_LAYOUT_TEXTURE) {
        p.vol.sx = p.vol.sy = 0;            // addressed by the texture unit
        p.vol.gsy = nbk * 32;               // gradients go to a BRICK buffer
        p.vol.gsx = nbj * nbk * 32;
    } else {
        p.vol.gsy = p.vol.sy = (uint32_t)p.vol.W;
        p.vol.gsx = p.vol.sx = (uint32_t)p.vol.H * (uint32_t)p.vol.W;
    }
    p.sources = a->sources;
    p.directions = a->directions;
    p.dir_pose_stride = a->dir_pose_stride;
    p.src_pose_stride = per_ray(a) ? a->n_rays * 3 : 3;
    p.src_ray_stride = per_ray(a) ? 3 : 0;
    p.product_f32 = a->product_f32;
    p.n_poses = a->n_poses;
    p.n_rays = a->n_rays;
    p.total_rays = a->n_poses * a->n_rays;
    p.S = a->n_samples;
    p.start = a->start;
    p.Sout = a->n_samples - a->start;
    p.nprefix = (p.Sout + PREFIX_STRIDE - 1) / PREFIX_STRIDE - 1;
    p.att_slots = (p.Sout + 3) / 4 * 4;
    {   // the backward's padded table: rays longer than one pass keep one pass's worth (render_bwd_kernel)
        const int n = p.Sout <= PREFIX_STRIDE ? p.Sout : PREFIX_STRIDE;
        p.att_slots_padded = (n + n / 32 + 8) / 4 * 4;
    }
    p.alpha = a->attenuation;
    p.frame = a->frame;
    p.seg_prefix = a->seg_prefix;
    return p;
}

// forward workspace (start > 0): [median float P | number of rays tied with the median, int32 P]
struct FwdWorkspace {
    float* median;
    int32_t* tie_count;
    int64_t bytes;
};
FwdWorkspace fwd_workspace(const DiffusRenderArgs* a, void* base) {
    FwdWorkspace w{};
    int64_t off = 0;
    if (a->start > 0) {
        w.median = (float*)((char*)base + off);
        off += align_up(a->n_poses * 4, 256);
        w.tie_count = (int32_t*)((char*)base + off);
        off += align_up(a->n_poses * 4, 256);
    }
    w.bytes = off;
    return w;
}

// backward workspace: [fwd workspace | source partials (P*R*3) | direction scratch (P*R*3) | first_rbar (P*R)]; with per-ray
// origins the kernels write grad_sources itself, so there are no source partials when it is given
struct BwdWorkspace {
    FwdWorkspace fwd;
    float* src_partial;
    float* dir_scratch;
    float* first_rbar;
    float* loss_partial;
    void* reduce_ws;
    int64_t bytes;
};
BwdWorkspace bwd_workspace(const DiffusRenderBwdArgs* b, void* base) {
    BwdWorkspace w{};
    const DiffusRenderArgs* a = &b->fwd;
    w.fwd = fwd_workspace(a, base);
    int64_t off = w.fwd.bytes;
    int64_t rays = a->n_poses * a->n_rays;
    bool pose_grad = a->sampler == DIFFUS_SAMPLER_TRILINEAR && (b->grad_sources || b->grad_directions);
    if (pose_grad) {
        if (per_ray(a) && b->grad_sources) {
            w.src_partial = b->grad_sources;
        } else {
            w.src_partial = (float*)((char*)base + off);
            off += align_up(rays * 12, 256);
        }
        if (!b->grad_directions) {
            w.dir_scratch = (float*)((char*)base + off);
            off += align_up(rays * 12, 256);
        }
    }
    if (a->start > 0) {
        w.first_rbar = (float*)((char*)base + off);
        off += align_up(rays * 4, 256);
    }
    if (b->target && b->loss) {
        w.loss_partial = (float*)((char*)base + off);
        off += align_up(rays * 4, 256);
        w.reduce_ws = (char*)base + off;
        off += align_up(reduce_sum_workspace_bytes(), 256);
    }
    w.bytes = off;
    return w;
}

int32_t cuda_rc(cudaError_t e) { return e == cudaSuccess ? DIFFUS_OK : (int32_t)e; }

// Gauss-Newton workspace: [fwd workspace | median tangent (P*6) | per-ray partials (P*R*32) | pivots (P*3 doubles, per-ray origins)]
struct GnWorkspace {
    FwdWorkspace fwd;
    float* med_tan;
    double* pivot;
    float* partial;
    int64_t bytes;
};
GnWorkspace gn_workspace(const DiffusGaussNewtonArgs* g, void* base) {
    GnWorkspace w{};
    const DiffusRenderArgs* a = &g->fwd;
    w.fwd = fwd_workspace(a, base);
    int64_t off = w.fwd.bytes;
    if (a->start > 0) {
        w.med_tan = (float*)((char*)base + off);
        off += align_up(a->n_poses * 24, 256);
    }
    w.partial = (float*)((char*)base + off);
    off += align_up(a->n_poses * a->n_rays * 128, 256);
    if (per_ray(a)) {
        w.pivot = (double*)((char*)base + off);
        off += align_up(a->n_poses * 24, 256);
    }
    w.bytes = off;
    return w;
}

// sweep workspace: [fwd workspace | median tangent (P*6) | per-ray partials (P*R*32) | range sums (32 doubles per range) |
// pivot (3 doubles, when the caller passes none)]
struct GnSweepWorkspace {
    FwdWorkspace fwd;
    float* med_tan;
    float* partial;
    double* range_sum;
    double* pivot;
    int64_t bytes;
};
GnSweepWorkspace gn_sweep_workspace(const DiffusGaussNewtonSweepArgs* g, void* base) {
    GnSweepWorkspace w{};
    const DiffusRenderArgs* a = &g->fwd;
    const int64_t rays = a->n_poses * a->n_rays;
    w.fwd = fwd_workspace(a, base);
    int64_t off = w.fwd.bytes;
    if (a->start > 0) {
        w.med_tan = (float*)((char*)base + off);
        off += align_up(a->n_poses * 24, 256);
    }
    w.partial = (float*)((char*)base + off);
    off += align_up(rays * 128, 256);
    w.range_sum = (double*)((char*)base + off);
    off += align_up(gn_sweep_ranges(rays) * 256, 256);
    if (!g->pivot) {
        w.pivot = (double*)((char*)base + off);
        off += 256;
    }
    w.bytes = off;
    return w;
}

}  // namespace

std::atomic<int64_t> diffus::launch_counter{0};

extern "C" {

int32_t diffus_abi_version(void) { return DIFFUS_ABI_VERSION; }

int64_t diffus_launch_count(void) { return diffus::launch_counter.load(std::memory_order_relaxed); }

const char* diffus_error_string(int32_t code) {
    switch (code) {
        case DIFFUS_OK: return "ok";
        case DIFFUS_E_NULL: return "a required pointer is NULL";
        case DIFFUS_E_SHAPE: return "non-positive or inconsistent sizes";
        case DIFFUS_E_ENUM: return "unknown sampler / layout / dtype tag";
        case DIFFUS_E_WORKSPACE: return "workspace missing or too small";
        case DIFFUS_E_UNSUPPORTED: return "unsupported configuration";
        default: return code > 0 ? cudaGetErrorString((cudaError_t)code) : "unknown error";
    }
}

int64_t diffus_render_workspace_bytes(const DiffusRenderArgs* a) {
    if (!a) return 0;
    return fwd_workspace(a, nullptr).bytes;
}

int32_t diffus_render_forward(const DiffusRenderArgs* a, void* stream) {
    int32_t e = check_render(a, a && !a->seg_prefix);      // frame may be NULL in a prefix-only run
    if (e) return e;
    if (!a->frame && a->n_samples - a->start <= PREFIX_STRIDE) return DIFFUS_OK;   // nothing to produce
    cudaStream_t st = (cudaStream_t)stream;
    RenderParams p = pack(a);
    const int pose64 = a->pose_dtype == DIFFUS_POSE_F64;
    if (a->start > 0) {
        FwdWorkspace w = fwd_workspace(a, a->workspace);
        if (!a->workspace || a->workspace_bytes < w.bytes) return DIFFUS_E_WORKSPACE;
        cudaError_t ce = launch_first_refl_median(p, a->sampler, a->volume.layout, pose64, w.median, w.tie_count, st);
        if (ce != cudaSuccess) return (int32_t)ce;
        p.median = w.median;
    }
    return cuda_rc(launch_render_fwd(p, a->sampler, a->volume.layout, pose64, st));
}

int64_t diffus_render_bwd_workspace_bytes(const DiffusRenderBwdArgs* b) {
    if (!b) return 0;
    return bwd_workspace(b, nullptr).bytes;
}

int32_t diffus_render_bwd_needs_prefix(const DiffusRenderBwdArgs* b) {
    if (!b) return DIFFUS_E_NULL;
    const DiffusRenderArgs* a = &b->fwd;
    if (!pose_dtype_ok(a->pose_dtype)) return DIFFUS_E_ENUM;
    if (a->sampler != DIFFUS_SAMPLER_NEAREST && a->sampler != DIFFUS_SAMPLER_TRILINEAR) return DIFFUS_E_ENUM;
    if (a->n_poses < 1 || a->n_rays < 1 || a->n_samples < 2 || a->start < 0 || a->start > a->n_samples - 2) return DIFFUS_E_SHAPE;
    const int sout = (int)(a->n_samples - a->start);
    if (sout <= PREFIX_STRIDE) return 0;
    const bool pose_grad = a->sampler == DIFFUS_SAMPLER_TRILINEAR && (b->grad_sources || b->grad_directions);
    return render_bwd_is_coop(sout, a->n_poses * a->n_rays, a->sampler, a->pose_dtype == DIFFUS_POSE_F64, pose_grad,
                              b->grad_volume != nullptr) ? 0 : 1;
}

int32_t diffus_render_backward(const DiffusRenderBwdArgs* b, void* stream) {
    if (!b) return DIFFUS_E_NULL;
    const DiffusRenderArgs* a = &b->fwd;
    int32_t e = check_render(a, false);
    if (e) return e;
    const bool mse = b->target != nullptr;
    if (!mse && !b->grad_frame) return DIFFUS_E_NULL;
    const bool trilinear = a->sampler == DIFFUS_SAMPLER_TRILINEAR;
    const bool pose_grad = trilinear && (b->grad_sources || b->grad_directions);
    const bool vol_grad = b->grad_volume != nullptr;
    if (!pose_grad && !vol_grad && !(mse && (b->loss || a->frame))) return DIFFUS_OK;
    cudaStream_t st = (cudaStream_t)stream;
    RenderParams p = pack(a);
    const int pose64 = a->pose_dtype == DIFFUS_POSE_F64;
    const bool coop = render_bwd_is_coop(p.Sout, p.total_rays, a->sampler, pose64, pose_grad, vol_grad);
    if (p.nprefix > 0 && !coop && !a->seg_prefix) return DIFFUS_E_NULL;
    BwdWorkspace w = bwd_workspace(b, b->workspace);
    if (w.bytes > 0 && (!b->workspace || b->workspace_bytes < w.bytes)) return DIFFUS_E_WORKSPACE;
    cudaError_t ce;
    if (a->start > 0) {
        ce = launch_first_refl_median(p, a->sampler, a->volume.layout, pose64, w.fwd.median, w.fwd.tie_count, st);
        if (ce != cudaSuccess) return (int32_t)ce;
        p.median = w.fwd.median;
        p.first_rbar = w.first_rbar;
    }
    p.grad_frame = b->grad_frame;
    p.target = b->target;
    p.grad_scale = b->grad_scale;
    p.loss_partial = w.loss_partial;
    if (!mse) p.frame = nullptr;
    p.grad_volume = b->grad_volume;
    p.grad_src_partial = w.src_partial;
    p.grad_dir = b->grad_directions ? b->grad_directions : w.dir_scratch;
    ce = launch_render_bwd(p, a->sampler, a->volume.layout, pose64, pose_grad, vol_grad, st);
    if (ce != cudaSuccess) return (int32_t)ce;
    if (a->start > 0) {
        ce = launch_median_backward(p, a->sampler, a->volume.layout, pose64, w.fwd.tie_count, pose_grad, vol_grad, st);
        if (ce != cudaSuccess) return (int32_t)ce;
    }
    // per-ray origins: the kernels wrote grad_sources themselves, there is nothing to fold over the rays
    const bool fold_sources = pose_grad && b->grad_sources && !per_ray(a);
    if (fold_sources && w.loss_partial && reduce_rays_and_sum_fits(a->n_poses * a->n_rays)) {
        // the fused pose step: both reductions in one launch
        return cuda_rc(launch_reduce_rays_and_sum(w.src_partial, a->n_poses, a->n_rays, b->grad_sources, w.loss_partial,
                                                  a->n_poses * a->n_rays, b->loss_scale, b->loss, st));
    }
    if (fold_sources) {
        ce = launch_reduce_rays(w.src_partial, a->n_poses, a->n_rays, b->grad_sources, st);
        if (ce != cudaSuccess) return (int32_t)ce;
    }
    if (w.loss_partial) {
        ce = launch_reduce_sum(w.loss_partial, a->n_poses * a->n_rays, b->loss_scale, b->loss, w.reduce_ws, st);
        if (ce != cudaSuccess) return (int32_t)ce;
    }
    return DIFFUS_OK;
}

int64_t diffus_render_gauss_newton_workspace_bytes(const DiffusGaussNewtonArgs* g) {
    if (!g) return 0;
    return gn_workspace(g, nullptr).bytes;
}

int32_t diffus_render_gauss_newton(const DiffusGaussNewtonArgs* g, void* stream) {
    if (!g) return DIFFUS_E_NULL;
    const DiffusRenderArgs* a = &g->fwd;
    int32_t e = check_render(a, false);
    if (e) return e;
    if (!g->target || !g->loss || !g->jtr || !g->jtj) return DIFFUS_E_NULL;
    if (a->sampler != DIFFUS_SAMPLER_TRILINEAR || a->pose_dtype == DIFFUS_POSE_F64) return DIFFUS_E_UNSUPPORTED;
    GnWorkspace w = gn_workspace(g, g->workspace);
    if (!g->workspace || g->workspace_bytes < w.bytes) return DIFFUS_E_WORKSPACE;
    cudaStream_t st = (cudaStream_t)stream;
    RenderParams p = pack(a);
    p.frame = nullptr;
    p.seg_prefix = nullptr;
    p.target = g->target;
    cudaError_t ce;
    if (w.pivot) {
        ce = launch_gn_pivot((const float*)a->sources, a->n_poses, a->n_rays, w.pivot, st);
        if (ce != cudaSuccess) return (int32_t)ce;
    }
    if (a->start > 0) {
        ce = launch_first_refl_median(p, a->sampler, a->volume.layout, 0, w.fwd.median, w.fwd.tie_count, st);
        if (ce != cudaSuccess) return (int32_t)ce;
        p.median = w.fwd.median;
        ce = launch_gn_median_tangent(p, a->volume.layout, w.pivot ? GN_LEVER_POSE : GN_LEVER_SOURCE, w.fwd.tie_count, w.pivot,
                                      w.med_tan, st);
        if (ce != cudaSuccess) return (int32_t)ce;
    }
    return cuda_rc(launch_render_gn(p, a->volume.layout, w.med_tan, w.pivot, w.partial, g->loss, g->jtr, g->jtj, st));
}

int64_t diffus_render_gauss_newton_sweep_workspace_bytes(const DiffusGaussNewtonSweepArgs* g) {
    if (!g) return 0;
    return gn_sweep_workspace(g, nullptr).bytes;
}

int32_t diffus_render_gauss_newton_sweep(const DiffusGaussNewtonSweepArgs* g, void* stream) {
    if (!g) return DIFFUS_E_NULL;
    const DiffusRenderArgs* a = &g->fwd;
    int32_t e = check_render(a, false);
    if (e) return e;
    if (!g->target || !g->loss || !g->jtr || !g->jtj) return DIFFUS_E_NULL;
    if (a->sampler != DIFFUS_SAMPLER_TRILINEAR || a->pose_dtype == DIFFUS_POSE_F64) return DIFFUS_E_UNSUPPORTED;
    GnSweepWorkspace w = gn_sweep_workspace(g, g->workspace);
    if (!g->workspace || g->workspace_bytes < w.bytes) return DIFFUS_E_WORKSPACE;
    cudaStream_t st = (cudaStream_t)stream;
    RenderParams p = pack(a);
    p.frame = nullptr;
    p.seg_prefix = nullptr;
    p.target = g->target;
    const double* pivot = g->pivot;
    cudaError_t ce;
    if (!pivot) {   // one source per pose stands for its R rays: the mean of the P sources is the mean of all P*R origins
        const int64_t rows = per_ray(a) ? a->n_poses * a->n_rays : a->n_poses;
        ce = launch_gn_sweep_pivot((const float*)a->sources, rows, w.range_sum, w.pivot, st);
        if (ce != cudaSuccess) return (int32_t)ce;
        pivot = w.pivot;
    }
    if (a->start > 0) {
        ce = launch_first_refl_median(p, a->sampler, a->volume.layout, 0, w.fwd.median, w.fwd.tie_count, st);
        if (ce != cudaSuccess) return (int32_t)ce;
        p.median = w.fwd.median;
        ce = launch_gn_median_tangent(p, a->volume.layout, GN_LEVER_SWEEP, w.fwd.tie_count, pivot, w.med_tan, st);
        if (ce != cudaSuccess) return (int32_t)ce;
    }
    return cuda_rc(launch_render_gn_sweep(p, a->volume.layout, w.med_tan, pivot, w.partial, w.range_sum, g->loss, g->jtr, g->jtj,
                                          st));
}

int32_t diffus_ray_indices(const DiffusRenderArgs* a, int64_t* x, int64_t* y, int64_t* z, void* stream) {
    int32_t e = check_render(a, false);
    if (e) return e;
    if (!x || !y || !z) return DIFFUS_E_NULL;
    RenderParams p = pack(a);
    return cuda_rc(launch_ray_indices(p, a->pose_dtype == DIFFUS_POSE_F64, x, y, z, (cudaStream_t)stream));
}

int32_t diffus_trace_values(const DiffusRenderArgs* a, float* out, void* stream) {
    int32_t e = check_render(a, false);
    if (e) return e;
    if (!out) return DIFFUS_E_NULL;
    RenderParams p = pack(a);
    return cuda_rc(launch_trace_values(p, a->sampler, a->volume.layout, a->pose_dtype == DIFFUS_POSE_F64, out,
                                       (cudaStream_t)stream));
}

int32_t diffus_sample_points(const DiffusVolume* volume, const float* points, int64_t n, int32_t sampler, float* values,
                             int64_t* x, int64_t* y, int64_t* z, void* stream) {
    if (!volume || !points || !values) return DIFFUS_E_NULL;
    int32_t e = check_volume(*volume);
    if (e) return e;
    if (n < 1) return DIFFUS_E_SHAPE;
    if (sampler != DIFFUS_SAMPLER_NEAREST && sampler != DIFFUS_SAMPLER_TRILINEAR) return DIFFUS_E_ENUM;
    if ((x || y || z) && !(x && y && z)) return DIFFUS_E_NULL;
    DiffusRenderArgs a{};
    a.volume = *volume;
    RenderParams p = pack(&a);
    return cuda_rc(launch_sample_points(p, sampler, volume->layout, points, n, values, x, y, z, (cudaStream_t)stream));
}

int32_t diffus_trace_values_backward(const DiffusRenderArgs* a, const float* grad_values, float* grad_volume,
                                     float* grad_sources, float* grad_directions, void* workspace,
                                     int64_t workspace_bytes, void* stream) {
    int32_t e = check_render(a, false);
    if (e) return e;
    if (!grad_values) return DIFFUS_E_NULL;
    const bool pose_grad = a->sampler == DIFFUS_SAMPLER_TRILINEAR && (grad_sources || grad_directions);
    if (!pose_grad && !grad_volume) return DIFFUS_OK;
    if (pose_grad && (!grad_sources || !grad_directions)) return DIFFUS_E_NULL;
    // per-ray origins: the kernel writes grad_sources itself
    const int64_t need = pose_grad && !per_ray(a) ? align_up(a->n_poses * a->n_rays * 12, 256) : 0;
    if (need > 0 && (!workspace || workspace_bytes < need)) return DIFFUS_E_WORKSPACE;
    RenderParams p = pack(a);
    p.start = 0;
    p.Sout = p.S;
    p.grad_volume = grad_volume;
    p.grad_src_partial = per_ray(a) ? grad_sources : (float*)workspace;
    p.grad_dir = grad_directions;
    cudaStream_t st = (cudaStream_t)stream;
    cudaError_t ce = launch_trace_values_bwd(p, a->sampler, a->volume.layout, a->pose_dtype == DIFFUS_POSE_F64, grad_values,
                                             pose_grad, grad_volume != nullptr, st);
    if (ce != cudaSuccess) return (int32_t)ce;
    if (pose_grad && !per_ray(a)) return cuda_rc(launch_reduce_rays(p.grad_src_partial, a->n_poses, a->n_rays, grad_sources, st));
    return DIFFUS_OK;
}

int32_t diffus_echo_forward(const float* refl, int64_t n_rays, int32_t n_interfaces, float* echo, void* stream) {
    if (!refl || !echo) return DIFFUS_E_NULL;
    if (n_rays < 1 || n_interfaces < 1 || n_rays >= ((int64_t)1 << 31)) return DIFFUS_E_SHAPE;
    return cuda_rc(launch_echo_fwd(refl, n_rays, n_interfaces, echo, (cudaStream_t)stream));
}

int32_t diffus_echo_backward(const float* refl, const float* grad_echo, int64_t n_rays, int32_t n_interfaces,
                             float* grad_refl, void* stream) {
    if (!refl || !grad_echo || !grad_refl) return DIFFUS_E_NULL;
    if (n_rays < 1 || n_interfaces < 1 || n_rays >= ((int64_t)1 << 31)) return DIFFUS_E_SHAPE;
    return cuda_rc(launch_echo_bwd(refl, grad_echo, n_rays, n_interfaces, grad_refl, (cudaStream_t)stream));
}

int32_t diffus_cone_directions(const double* median, int64_t n_poses, int64_t n_rays, double opening_angle, float* out,
                               void* stream) {
    if (!median || !out) return DIFFUS_E_NULL;
    if (n_poses < 1 || n_rays < 1) return DIFFUS_E_SHAPE;
    return cuda_rc(launch_cone_directions(median, n_poses, n_rays, opening_angle, out, (cudaStream_t)stream));
}

// value 2 selected a removed tensor-core path: rejected like any unknown value
static bool mlp_path_valid(int32_t path) {
    return path == DIFFUS_MLP_PATH_AUTO || path == DIFFUS_MLP_PATH_CUDA_CORES || path == DIFFUS_MLP_PATH_PIECEWISE;
}

int32_t diffus_mlp_forward_ex(const float* params, const float* x, const uint8_t* mask, int64_t n, float out_scale,
                              float fill, float* out, int32_t path, void* stream) {
    if (!params || !x || !out) return DIFFUS_E_NULL;
    if (n < 1) return DIFFUS_E_SHAPE;
    if (!mlp_path_valid(path)) return DIFFUS_E_ENUM;
    // volumes go through the piecewise-linear table; a handful of samples is not worth building it
    if (path == DIFFUS_MLP_PATH_PIECEWISE || (path == DIFFUS_MLP_PATH_AUTO && n >= 1024))
        return cuda_rc(launch_mlp_pwl_fwd(params, x, mask, n, out_scale, fill, out, (cudaStream_t)stream));
    return cuda_rc(launch_mlp_fwd(params, x, mask, n, out_scale, fill, out, (cudaStream_t)stream));
}

int32_t diffus_mlp_forward(const float* params, const float* x, const uint8_t* mask, int64_t n, float out_scale,
                           float fill, float* out, void* stream) {
    return diffus_mlp_forward_ex(params, x, mask, n, out_scale, fill, out, DIFFUS_MLP_PATH_AUTO, stream);
}

int64_t diffus_mlp_bwd_workspace_bytes(int64_t n) { return n < 1 ? 0 : mlp_bwd_workspace_bytes(n); }

int32_t diffus_mlp_backward_ex(const float* params, const float* x, const uint8_t* mask, const float* grad_out, int64_t n,
                               float out_scale, float* grad_params, void* workspace, int64_t workspace_bytes, int32_t path,
                               void* stream) {
    if (!params || !x || !grad_out || !grad_params) return DIFFUS_E_NULL;
    if (n < 1) return DIFFUS_E_SHAPE;
    if (!mlp_path_valid(path)) return DIFFUS_E_ENUM;
    if (!workspace || workspace_bytes < mlp_bwd_workspace_bytes(n)) return DIFFUS_E_WORKSPACE;
    if (((uintptr_t)workspace & 7u) != 0) return DIFFUS_E_WORKSPACE;
    if (path == DIFFUS_MLP_PATH_PIECEWISE || (path == DIFFUS_MLP_PATH_AUTO && n >= 1024))
        return cuda_rc(launch_mlp_pwl_bwd(params, x, mask, grad_out, n, out_scale, grad_params, workspace, (cudaStream_t)stream));
    return cuda_rc(launch_mlp_bwd(params, x, mask, grad_out, n, out_scale, grad_params, workspace, nullptr, (cudaStream_t)stream));
}

int32_t diffus_mlp_backward(const float* params, const float* x, const uint8_t* mask, const float* grad_out, int64_t n,
                            float out_scale, float* grad_params, void* workspace, int64_t workspace_bytes,
                            void* stream) {
    return diffus_mlp_backward_ex(params, x, mask, grad_out, n, out_scale, grad_params, workspace, workspace_bytes,
                                  DIFFUS_MLP_PATH_AUTO, stream);
}

int32_t diffus_mlp_input_grad(const float* params, const float* x, const uint8_t* mask, const float* grad_out, int64_t n,
                              float out_scale, float* grad_x, void* stream) {
    if (!params || !x || !grad_out || !grad_x) return DIFFUS_E_NULL;
    if (n < 1) return DIFFUS_E_SHAPE;
    return cuda_rc(launch_mlp_pwl_dx(params, x, mask, grad_out, n, out_scale, grad_x, (cudaStream_t)stream));
}

int64_t diffus_splat_workspace_bytes(int32_t H, int32_t W) { return (H < 1 || W < 1) ? 0 : splat_workspace_bytes(H, W); }

int32_t diffus_splat_forward(const float* c0, const float* c1, const float* c2, const float* intensities, int64_t n,
                             int32_t H, int32_t W, float sigma, float* out, void* workspace, int64_t workspace_bytes,
                             void* stream) {
    if (!c0 || !c1 || !c2 || !intensities || !out) return DIFFUS_E_NULL;
    if (n < 1 || n >= ((int64_t)1 << 32) - 1 || H < 1 || W < 1 || !(sigma > 0.f)) return DIFFUS_E_SHAPE;
    if (((int)(6.f * sigma) | 1) > 63) return DIFFUS_E_UNSUPPORTED;
    if (!workspace || workspace_bytes < splat_workspace_bytes(H, W)) return DIFFUS_E_WORKSPACE;
    return cuda_rc(launch_splat_fwd(c0, c1, c2, intensities, n, H, W, sigma, out, workspace, (cudaStream_t)stream));
}

int32_t diffus_splat_backward(const float* c0, const float* c1, const float* c2, const float* intensities, int64_t n,
                              int32_t H, int32_t W, float sigma, const float* grad_out, float* grad_intensities,
                              void* workspace, int64_t workspace_bytes, void* stream) {
    if (!c0 || !c1 || !c2 || !intensities || !grad_out || !grad_intensities) return DIFFUS_E_NULL;
    if (n < 1 || n >= ((int64_t)1 << 32) - 1 || H < 1 || W < 1 || !(sigma > 0.f)) return DIFFUS_E_SHAPE;
    if (((int)(6.f * sigma) | 1) > 63) return DIFFUS_E_UNSUPPORTED;
    if (!workspace || workspace_bytes < splat_workspace_bytes(H, W)) return DIFFUS_E_WORKSPACE;
    return cuda_rc(launch_splat_bwd(c0, c1, c2, intensities, n, H, W, sigma, grad_out, grad_intensities, workspace,
                                    (cudaStream_t)stream));
}

int32_t diffus_adam_step(float* params, const float* grads, float* state, int64_t n, float lr, float beta1, float beta2, float eps,
                         float weight_decay, float grad_scale, void* stream) {
    if (!params || !grads || !state) return DIFFUS_E_NULL;
    if (n < 1) return DIFFUS_E_SHAPE;
    if (n > 65536) return DIFFUS_E_UNSUPPORTED;       // one CTA: every thread reads the step counter before it is advanced
    return cuda_rc(launch_adam_step(params, grads, state, n, lr, beta1, beta2, eps, weight_decay, grad_scale, (cudaStream_t)stream));
}

int32_t diffus_volume_slice(float* volume, const int32_t dim[3], int32_t layout, int32_t axis, int32_t index, float* slice,
                            int32_t scatter, void* stream) {
    if (!volume || !dim || !slice) return DIFFUS_E_NULL;
    if (dim[0] < 1 || dim[1] < 1 || dim[2] < 1 || axis < 0 || axis > 2 || index < 0 || index >= dim[axis]) return DIFFUS_E_SHAPE;
    if (layout != DIFFUS_LAYOUT_LINEAR && layout != DIFFUS_LAYOUT_BRICK) return DIFFUS_E_ENUM;
    return cuda_rc(launch_volume_slice(volume, dim, layout, axis, index, slice, scatter != 0, (cudaStream_t)stream));
}

int32_t diffus_conv1d_rows_forward(const float* in, int64_t rows, int32_t n_in, const float* w, int32_t taps, int32_t pad, float* out,
                                   void* stream) {
    if (!in || !w || !out) return DIFFUS_E_NULL;
    const int64_t n_out = (int64_t)n_in + 2 * (int64_t)pad - taps + 1;
    if (rows < 1 || n_in < 1 || taps < 1 || pad < 0 || n_out < 1) return DIFFUS_E_SHAPE;
    if (taps > 128) return DIFFUS_E_UNSUPPORTED;
    return cuda_rc(launch_conv1d_rows(in, rows, n_in, w, taps, pad, 0, out, (int)n_out, (cudaStream_t)stream));
}

int32_t diffus_conv1d_rows_backward(const float* grad_out, int64_t rows, int32_t n_in, const float* w, int32_t taps, int32_t pad,
                                    float* grad_in, void* stream) {
    if (!grad_out || !w || !grad_in) return DIFFUS_E_NULL;
    const int64_t n_out = (int64_t)n_in + 2 * (int64_t)pad - taps + 1;
    if (rows < 1 || n_in < 1 || taps < 1 || pad < 0 || n_out < 1) return DIFFUS_E_SHAPE;
    if (taps > 128) return DIFFUS_E_UNSUPPORTED;
    // grad_in[i] = sum_t w[t] grad_out[i - t + pad]: the same correlation over the (rows, n_out) gradient with w flipped
    return cuda_rc(launch_conv1d_rows(grad_out, rows, (int)n_out, w, taps, taps - 1 - pad, 1, grad_in, n_in, (cudaStream_t)stream));
}

int32_t diffus_rotate_around_apex(const float* x, const float* z, int64_t n, float cos_a, float sin_a, float shift, float apex0,
                                  float apex1, float* x_rot, float* z_rot, void* stream) {
    if (!x || !z || !x_rot || !z_rot) return DIFFUS_E_NULL;
    if (n < 1) return DIFFUS_E_SHAPE;
    return cuda_rc(launch_rotate_apex(x, z, n, cos_a, sin_a, shift, apex0, apex1, x_rot, z_rot, (cudaStream_t)stream));
}

int32_t diffus_log_compress_forward(const float* img, int64_t n, float* out, float* max_out, void* stream) {
    if (!img || !out) return DIFFUS_E_NULL;
    if (n < 1) return DIFFUS_E_SHAPE;
    return cuda_rc(launch_log_compress_fwd(img, n, out, max_out, (cudaStream_t)stream));
}

int32_t diffus_log_compress_backward(const float* img, const float* grad_out, int64_t n, float* grad_img, void* stream) {
    if (!img || !grad_out || !grad_img) return DIFFUS_E_NULL;
    if (n < 1) return DIFFUS_E_SHAPE;
    return cuda_rc(launch_log_compress_bwd(img, grad_out, n, grad_img, (cudaStream_t)stream));
}

int32_t diffus_rf_to_bmode(const float* profiles, int64_t n_rays, int32_t n_samples, const float* hilbert_kernel, float* out,
                           void* workspace, int64_t workspace_bytes, void* stream) {
    if (!profiles || !hilbert_kernel || !out) return DIFFUS_E_NULL;
    if (n_rays < 1 || n_samples < 1 || n_rays >= ((int64_t)1 << 31)) return DIFFUS_E_SHAPE;
    if (n_samples > 28000) return DIFFUS_E_UNSUPPORTED;          // a line and its kernel live in shared memory
    if (!workspace || workspace_bytes < 4) return DIFFUS_E_WORKSPACE;
    return cuda_rc(launch_rf_to_bmode(profiles, n_rays, n_samples, hilbert_kernel, out, workspace, (cudaStream_t)stream));
}

int32_t diffus_masked_mse_edge_forward(const float* synth, const float* real, const uint8_t* mask, int32_t H, int32_t W,
                                       float edge_weight, float* stats, void* stream) {
    if (!synth || !real || !mask || !stats) return DIFFUS_E_NULL;
    if (H < 1 || W < 1) return DIFFUS_E_SHAPE;
    return cuda_rc(launch_masked_mse_edge_fwd(synth, real, mask, H, W, edge_weight, stats, (cudaStream_t)stream));
}

int32_t diffus_masked_mse_edge_backward(const float* synth, const float* real, const uint8_t* mask, int32_t H, int32_t W,
                                        float edge_weight, const float* stats, const float* grad_loss, float* grad_synth,
                                        void* stream) {
    if (!synth || !real || !mask || !stats || !grad_loss || !grad_synth) return DIFFUS_E_NULL;
    if (H < 1 || W < 1) return DIFFUS_E_SHAPE;
    return cuda_rc(launch_masked_mse_edge_bwd(synth, real, mask, H, W, edge_weight, stats, grad_loss, grad_synth, (cudaStream_t)stream));
}

int64_t diffus_ssim_workspace_bytes(int32_t H, int32_t W, int32_t ksize) {
    if (ksize < 1 || ksize > 33 || H < ksize || W < ksize) return 0;
    return ssim_workspace_bytes(H, W, ksize);
}

static int32_t check_ssim(const float* synth, const float* real, int32_t H, int32_t W, int32_t ksize, float sigma, void* workspace,
                          int64_t workspace_bytes) {
    if (!synth || !real) return DIFFUS_E_NULL;
    if (ksize < 1 || H < ksize || W < ksize || !(sigma > 0.f)) return DIFFUS_E_SHAPE;
    if (ksize > 33 || !(ksize & 1)) return DIFFUS_E_UNSUPPORTED;
    if (!workspace || workspace_bytes < ssim_workspace_bytes(H, W, ksize)) return DIFFUS_E_WORKSPACE;
    return DIFFUS_OK;
}

int32_t diffus_ssim_loss_forward(const float* synth, const float* real, int32_t H, int32_t W, int32_t ksize, float sigma, float k1,
                                 float k2, int32_t normalize, float* loss, void* workspace, int64_t workspace_bytes, void* stream) {
    if (!loss) return DIFFUS_E_NULL;
    int32_t e = check_ssim(synth, real, H, W, ksize, sigma, workspace, workspace_bytes);
    if (e) return e;
    return cuda_rc(launch_ssim_fwd(synth, real, H, W, ksize, sigma, k1, k2, normalize, loss, workspace, (cudaStream_t)stream));
}

int32_t diffus_ssim_loss_backward(const float* synth, const float* real, int32_t H, int32_t W, int32_t ksize, float sigma,
                                  int32_t normalize, const float* grad_loss, float* grad_synth, void* workspace,
                                  int64_t workspace_bytes, void* stream) {
    if (!grad_loss || !grad_synth) return DIFFUS_E_NULL;
    int32_t e = check_ssim(synth, real, H, W, ksize, sigma, workspace, workspace_bytes);
    if (e) return e;
    return cuda_rc(launch_ssim_bwd(synth, real, H, W, ksize, sigma, normalize, grad_loss, grad_synth, workspace, (cudaStream_t)stream));
}

int32_t diffus_brain_mask(const float* volume, const int32_t dim[3], float threshold, int32_t iterations, uint8_t* mask,
                          uint8_t* scratch, void* stream) {
    if (!volume || !dim || !mask || !scratch) return DIFFUS_E_NULL;
    if (dim[0] < 1 || dim[1] < 1 || dim[2] < 1 || iterations < 0 || iterations > 64) return DIFFUS_E_SHAPE;
    return cuda_rc(launch_brain_mask(volume, dim, threshold, iterations, mask, scratch, (cudaStream_t)stream));
}

int32_t diffus_masked_zscore(const float* volume, const uint8_t* mask, int64_t n, float* out, void* workspace,
                             int64_t workspace_bytes, void* stream) {
    if (!volume || !mask || !out) return DIFFUS_E_NULL;
    if (n < 1) return DIFFUS_E_SHAPE;
    if (!workspace || workspace_bytes < 64) return DIFFUS_E_WORKSPACE;
    return cuda_rc(launch_masked_zscore(volume, mask, n, out, workspace, (cudaStream_t)stream));
}

int64_t diffus_brick_elems(const int32_t dim[3]) {
    if (!dim) return 0;
    int64_t nbi = (dim[0] + BRICK_I - 1) / BRICK_I, nbj = (dim[1] + BRICK_J - 1) / BRICK_J,
            nbk = (dim[2] + BRICK_K - 1) / BRICK_K;
    return nbi * nbj * nbk * 32;
}

int32_t diffus_volume_to_bricks(const float* linear, const int32_t dim[3], float* bricks, void* stream) {
    if (!linear || !dim || !bricks) return DIFFUS_E_NULL;
    if (dim[0] < 1 || dim[1] < 1 || dim[2] < 1) return DIFFUS_E_SHAPE;
    return cuda_rc(launch_to_bricks(linear, dim, bricks, (cudaStream_t)stream));
}

int32_t diffus_bricks_to_volume(const float* bricks, const int32_t dim[3], float* linear, void* stream) {
    if (!linear || !dim || !bricks) return DIFFUS_E_NULL;
    if (dim[0] < 1 || dim[1] < 1 || dim[2] < 1) return DIFFUS_E_SHAPE;
    return cuda_rc(launch_from_bricks(bricks, dim, linear, (cudaStream_t)stream));
}

int64_t diffus_quad_elems(const int32_t dim[3]) {
    if (!dim) return 0;
    int64_t nqi = (dim[0] + QUAD_B - 1) / QUAD_B, nqj = (dim[1] + QUAD_B - 1) / QUAD_B, nqk = (dim[2] + QUAD_B - 1) / QUAD_B;
    return nqi * nqj * nqk * 8 * 4;
}

int32_t diffus_volume_to_quads(const float* linear, const int32_t dim[3], float* quads, void* stream) {
    if (!linear || !dim || !quads) return DIFFUS_E_NULL;
    if (dim[0] < 1 || dim[1] < 1 || dim[2] < 1) return DIFFUS_E_SHAPE;
    if ((uintptr_t)quads & 15) return DIFFUS_E_UNSUPPORTED;
    return cuda_rc(launch_to_quads(linear, dim, quads, (cudaStream_t)stream));
}

static bool overlap(const float* a, const float* b, int64_t n) {
    const uintptr_t x = (uintptr_t)a, y = (uintptr_t)b, bytes = (uintptr_t)n * sizeof(float);
    return x < y + bytes && y < x + bytes;
}

int32_t diffus_volume_gaussian_blur(const float* src, const int32_t dim[3], float sigma, float truncate, float* dst, float* scratch,
                                    void* stream) {
    if (!src || !dim || !dst || !scratch) return DIFFUS_E_NULL;
    if (dim[0] < 1 || dim[1] < 1 || dim[2] < 1) return DIFFUS_E_SHAPE;
    if (!std::isfinite(sigma) || sigma < 0.f || !std::isfinite(truncate) || truncate <= 0.f) return DIFFUS_E_SHAPE;
    if ((double)dim[0] * dim[1] * dim[2] >= (double)((int64_t)1 << 60)) return DIFFUS_E_UNSUPPORTED;   // int64 byte offsets
    const int64_t n = (int64_t)dim[0] * dim[1] * dim[2];
    if (overlap(src, dst, n) || overlap(src, scratch, n) || overlap(dst, scratch, n)) return DIFFUS_E_SHAPE;
    // scipy: an axis with sigma <= 1e-15 is skipped; else radius = int(truncate * sigma + 0.5)
    const double rr = (double)sigma <= 1e-15 ? 0.0 : (double)truncate * (double)sigma + 0.5;
    if (rr >= BLUR_MAX_RADIUS + 1) return DIFFUS_E_UNSUPPORTED;
    return cuda_rc(launch_gaussian_blur(src, dim, sigma, (int)rr, dst, scratch, (cudaStream_t)stream));
}

// The layered array: width = dim[2] (p2, fastest), height = dim[1], layers = dim[0].
static cudaError_t copy_linear_to_array(cudaArray_t arr, const float* linear, const int32_t dim[3], cudaStream_t st) {
    cudaMemcpy3DParms cp = {};
    cp.srcPtr = make_cudaPitchedPtr((void*)linear, (size_t)dim[2] * sizeof(float), (size_t)dim[2], (size_t)dim[1]);
    cp.dstArray = arr;
    cp.extent = make_cudaExtent((size_t)dim[2], (size_t)dim[1], (size_t)dim[0]);
    cp.kind = cudaMemcpyDeviceToDevice;
    return cudaMemcpy3DAsync(&cp, st);
}

int32_t diffus_volume_texture_create(const float* linear, const int32_t dim[3], uint64_t* texture_object,
                                     uint64_t* array_handle, void* stream) {
    if (!linear || !dim || !texture_object || !array_handle) return DIFFUS_E_NULL;
    if (dim[0] < 1 || dim[1] < 1 || dim[2] < 1) return DIFFUS_E_SHAPE;
    if (dim[0] > 2048 || dim[1] > 32768 || dim[2] > 32768) return DIFFUS_E_UNSUPPORTED;
    cudaChannelFormatDesc fmt = cudaCreateChannelDesc<float>();
    cudaExtent ext = make_cudaExtent((size_t)dim[2], (size_t)dim[1], (size_t)dim[0]);
    cudaArray_t arr = nullptr;
    cudaError_t e = cudaMalloc3DArray(&arr, &fmt, ext, cudaArrayLayered | cudaArrayTextureGather);
    if (e != cudaSuccess) {                  // some drivers list the gather flag for plain 2-D arrays only
        (void)cudaGetLastError();
        e = cudaMalloc3DArray(&arr, &fmt, ext, cudaArrayLayered);
    }
    if (e != cudaSuccess) return (int32_t)e;
    e = copy_linear_to_array(arr, linear, dim, (cudaStream_t)stream);
    cudaTextureObject_t tex = 0;
    if (e == cudaSuccess) {
        cudaResourceDesc res = {};
        res.resType = cudaResourceTypeArray;
        res.res.array.array = arr;
        cudaTextureDesc td = {};
        td.addressMode[0] = td.addressMode[1] = td.addressMode[2] = cudaAddressModeClamp;
        td.filterMode = cudaFilterModePoint;
        td.readMode = cudaReadModeElementType;
        td.normalizedCoords = 0;
        e = cudaCreateTextureObject(&tex, &res, &td, nullptr);
    }
    if (e != cudaSuccess) {
        cudaFreeArray(arr);
        return (int32_t)e;
    }
    *texture_object = (uint64_t)tex;
    *array_handle = (uint64_t)(uintptr_t)arr;
    return DIFFUS_OK;
}

int32_t diffus_volume_texture_update(uint64_t array_handle, const float* linear, const int32_t dim[3], void* stream) {
    if (!array_handle || !linear || !dim) return DIFFUS_E_NULL;
    if (dim[0] < 1 || dim[1] < 1 || dim[2] < 1) return DIFFUS_E_SHAPE;
    return cuda_rc(copy_linear_to_array((cudaArray_t)(uintptr_t)array_handle, linear, dim, (cudaStream_t)stream));
}

int32_t diffus_volume_texture_destroy(uint64_t texture_object, uint64_t array_handle) {
    cudaError_t e = cudaSuccess;
    if (texture_object) e = cudaDestroyTextureObject((cudaTextureObject_t)texture_object);
    if (array_handle) {
        cudaError_t e2 = cudaFreeArray((cudaArray_t)(uintptr_t)array_handle);
        if (e == cudaSuccess) e = e2;
    }
    return cuda_rc(e);
}

int32_t diffus_gather_probe(const float* buf, int64_t n_floats, int32_t reads_per_thread, int64_t n_threads, uint32_t seed,
                            float* sink, void* stream) {
    if (!buf || !sink) return DIFFUS_E_NULL;
    if (n_floats < 8 || n_floats / 8 >= ((int64_t)1 << 32) || reads_per_thread < 8 || reads_per_thread % 8 || n_threads < 256 ||
        n_threads % 256 || n_threads / 256 >= ((int64_t)1 << 31))
        return DIFFUS_E_SHAPE;
    return cuda_rc(launch_gather_probe(buf, n_floats, reads_per_thread, n_threads, seed, sink, (cudaStream_t)stream));
}

int32_t diffus_fan_directions(const float* median, const float* hint, int64_t n_poses, int64_t n_rays, double opening_angle,
                              float* out, void* stream) {
    if (!median || !hint || !out) return DIFFUS_E_NULL;
    if (n_poses < 1 || n_rays < 1 || n_poses >= ((int64_t)1 << 31)) return DIFFUS_E_SHAPE;
    return cuda_rc(launch_fan_directions(median, hint, n_poses, n_rays, opening_angle, out, (cudaStream_t)stream));
}

int32_t diffus_fan_directions_backward(const float* median, const float* hint, const float* grad_directions, int64_t n_poses,
                                       int64_t n_rays, double opening_angle, float* grad_median, float* grad_hint, void* stream) {
    if (!median || !hint || !grad_directions || !grad_median || !grad_hint) return DIFFUS_E_NULL;
    if (n_poses < 1 || n_rays < 1 || n_poses >= ((int64_t)1 << 31)) return DIFFUS_E_SHAPE;
    return cuda_rc(launch_fan_directions_bwd(median, hint, grad_directions, n_poses, n_rays, opening_angle, grad_median, grad_hint,
                                             (cudaStream_t)stream));
}

static int32_t check_probe(int32_t kind, int64_t n_poses, int64_t n_rays, double opening_angle, double radius, double width) {
    if (n_poses < 1 || n_rays < 1 || n_poses >= ((int64_t)1 << 31) || n_poses * n_rays >= ((int64_t)1 << 31)) return DIFFUS_E_SHAPE;
    if (kind == DIFFUS_PROBE_CONVEX) {
        if (!std::isfinite(opening_angle) || !std::isfinite(radius) || radius < 0.0) return DIFFUS_E_SHAPE;
    } else if (kind == DIFFUS_PROBE_LINEAR) {
        if (!std::isfinite(width) || width <= 0.0) return DIFFUS_E_SHAPE;
    } else {
        return DIFFUS_E_ENUM;
    }
    return DIFFUS_OK;
}

int32_t diffus_probe_rays(int32_t kind, const float* centre, const float* median, const float* hint, int64_t n_poses, int64_t n_rays,
                          double opening_angle, double radius, double width, float* origins, float* directions, void* stream) {
    if (!centre || !median || !hint || !origins || !directions) return DIFFUS_E_NULL;
    int32_t e = check_probe(kind, n_poses, n_rays, opening_angle, radius, width);
    if (e) return e;
    return cuda_rc(launch_probe_rays(kind, centre, median, hint, n_poses, n_rays, opening_angle, radius, width, origins, directions,
                                     (cudaStream_t)stream));
}

int32_t diffus_probe_rays_backward(int32_t kind, const float* centre, const float* median, const float* hint, const float* grad_origins,
                                   const float* grad_directions, int64_t n_poses, int64_t n_rays, double opening_angle, double radius,
                                   double width, float* grad_centre, float* grad_median, float* grad_hint, void* stream) {
    if (!centre || !median || !hint || !grad_origins || !grad_directions || !grad_centre || !grad_median || !grad_hint)
        return DIFFUS_E_NULL;
    int32_t e = check_probe(kind, n_poses, n_rays, opening_angle, radius, width);
    if (e) return e;
    return cuda_rc(launch_probe_rays_bwd(kind, centre, median, hint, grad_origins, grad_directions, n_poses, n_rays, opening_angle,
                                         radius, width, grad_centre, grad_median, grad_hint, (cudaStream_t)stream));
}

}  // extern "C"
