/*
 * diffus_b200.h -- C ABI of the B200-native DiffUS B-mode renderer hot path.
 *
 * The reference (gduguey/DiffUS) is pure Python and has no FFI of its own; its boundary
 * is the Python call surface of src/renderer.py, src/cone.py and src/impedance.py.  Each
 * entry point below names the reference interface it replaces (file:line relative to
 * the reference root).  The Python host package (diffus_b200/) binds these symbols with
 * ctypes and wraps them in torch.library custom ops + autograd; INTEGRATION.md shows the
 * binding a maintainer of the reference would add.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless the name says host; all tensors are
 *     dense, row-major, caller-owned; sizes are element counts;
 *   - `stream` is a cudaStream_t passed as void* (0 = legacy default stream);
 *   - functions only enqueue work: they never allocate device memory, never synchronise
 *     and keep no global state (re-entrant across streams and devices);
 *   - return 0 on success, a negative DIFFUS_E_* for rejected arguments, or a positive
 *     cudaError_t if a launch failed;
 *   - there is no CPU implementation behind this ABI.
 */
#ifndef DIFFUS_B200_H
#define DIFFUS_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DIFFUS_ABI_VERSION 1

/* error codes (negative = bad argument) */
#define DIFFUS_OK 0
#define DIFFUS_E_NULL (-1)       /* a required pointer is NULL            */
#define DIFFUS_E_SHAPE (-2)      /* non-positive or inconsistent sizes    */
#define DIFFUS_E_ENUM (-3)       /* unknown sampler / layout / dtype tag  */
#define DIFFUS_E_WORKSPACE (-4)  /* workspace missing or too small        */
#define DIFFUS_E_UNSUPPORTED (-5)

/* sampler: how impedance is read at a ray point */
#define DIFFUS_SAMPLER_NEAREST 0   /* src/renderer.py:751-759 (HEAD)                          */
#define DIFFUS_SAMPLER_TRILINEAR 1 /* grid_sample(bilinear, border, align_corners=True): the
                                      reference's notebook-era sampler, src/renderer.py:802-815
                                      grid construction; the only pose-differentiable form    */

/* volume layout in HBM */
#define DIFFUS_LAYOUT_LINEAR 0 /* C-contiguous [p0][p1][p2], exactly the torch tensor        */
#define DIFFUS_LAYOUT_BRICK 1  /* 4x4x2-voxel bricks of 128 B made by diffus_volume_to_bricks */
#define DIFFUS_LAYOUT_QUAD 2   /* one float4 per voxel = the voxel and its +p1, +p2, +p1+p2 neighbours (clamped at
                                  the faces), 2x2x2 voxels per 128 B, made by diffus_volume_to_quads: a trilinear
                                  cell is two 16-byte loads.  4x the footprint; read-only (see grad_volume)        */
#define DIFFUS_LAYOUT_TEXTURE 3 /* a layered 2-D CUDA array behind a texture object made by diffus_volume_texture_create
                                  (layer = p0, y = p1, x = p2; clamp addressing, point sampling): a trilinear cell is two
                                  tld4 texel gathers, address arithmetic and border clamp done by the texture unit, 1x the
                                  footprint.  DiffusVolume.data carries the 64-bit texture object; read-only            */

/* dtype tags for the probe pose (the reference's `points` dtype follows torch promotion,
   src/renderer.py:124, and is cast to float32 at :751) */
#define DIFFUS_POSE_F32 0 /* sources/directions are float32 arrays                            */
#define DIFFUS_POSE_F64 1 /* both are float64 arrays; see `product_f32`                        */
#define DIFFUS_POSE_F32_PER_RAY 2 /* float32; sources are (P,R,3): one origin per ray (linear and convex array probes).
                                     Ray i of pose p samples sources[p][i] + k * directions[.][i].  Accepted by every entry point
                                     that takes a DiffusRenderArgs; a library that predates it answers DIFFUS_E_ENUM.  There is no
                                     float64 per-ray form.                                                                   */

typedef struct DiffusVolume {
    const float* data; /* impedance volume, float32                                          */
    int32_t dim[3];    /* extent along point component 0,1,2  (volume[p0][p1][p2])           */
    int32_t layout;    /* DIFFUS_LAYOUT_*                                                    */
} DiffusVolume;

/* One batched render: P poses x R rays x S samples.  Replaces
 * UltrasoundRenderer.plot_beam_frame (src/renderer.py:201-275) with artifacts=False, i.e.
 * trace_ray (:89-180) + custom_nearest_sampler (:741-819) + compute_reflection_coeff
 * (:27-33) + the start crop / median (:237-245) + compute_echo_traces (:439-457, whose
 * per-depth dense solves are evaluated as a 2x2 transfer-matrix prefix product) + the
 * exp(-alpha k) attenuation (:256-259), for a leading batch of probe poses. */
typedef struct DiffusRenderArgs {
    DiffusVolume volume;
    const void* sources;        /* (P,3) float32 or float64 per pose_dtype; (P,R,3) float32 for DIFFUS_POSE_F32_PER_RAY */
    const void* directions;     /* (P,R,3) or, if dir_pose_stride == 0, (R,3) shared by poses */
    int32_t pose_dtype;         /* DIFFUS_POSE_*                                             */
    int32_t product_f32;        /* POSE_F64 only: directions were float32, so k*dir rounds to
                                   float32 before the float64 add (torch promotion)          */
    int64_t n_poses;            /* P >= 1                                                    */
    int64_t n_rays;             /* R >= 1                                                    */
    int64_t dir_pose_stride;    /* elements between poses in `directions`: R*3 or 0          */
    int32_t n_samples;          /* S >= 2 samples per ray (1-voxel steps)                    */
    int32_t start;              /* columns cropped from the front, 0 <= start <= S-2; when > 0
                                   the first kept reflection coefficient of every ray of a pose
                                   is replaced by the lower median over that pose's rays     */
    int32_t sampler;            /* DIFFUS_SAMPLER_*                                          */
    float attenuation;          /* alpha: frame[k] = echo[k] * exp(-alpha k), k from 0 after crop */
    float* frame;               /* out (P,R,S-start); may be NULL when seg_prefix is given: a
                                   prefix-only run (no frame is formed or written, the last 512-column
                                   segment is not walked)                                       */
    float* seg_prefix;          /* out, optional: (P,R,ceil((S-start)/512)-1,4) transfer-matrix
                                   prefixes at every 512th column, consumed by the backward;
                                   may be NULL (always unused when S-start <= 512)           */
    void* workspace;            /* diffus_render_workspace_bytes() bytes, needed iff start>0 */
    int64_t workspace_bytes;
} DiffusRenderArgs;

/* Backward of the render above (what torch autograd computes through the reference,
 * SURVEY.md 3.2): given d loss / d frame, accumulate d loss / d volume (index_put_
 * accumulate semantics of src/renderer.py:758's backward) and, for the trilinear sampler,
 * d loss / d source and d loss / d directions.  Any of the three outputs may be NULL. */
typedef struct DiffusRenderBwdArgs {
    DiffusRenderArgs fwd;       /* same inputs as the forward; fwd.frame is only written in the
                                   fused-loss mode below and may be NULL;
                                   fwd.seg_prefix = the buffer the forward filled (required
                                   when diffus_render_bwd_needs_prefix() says so)             */
    const float* grad_frame;    /* (P,R,S-start)                                             */
    float* grad_volume;         /* QUAD and TEXTURE volumes: a BRICK buffer.  Otherwise the
                                   same layout as fwd.volume (LINEAR (D,H,W), or diffus_brick_elems()
                                   floats for BRICK), ACCUMULATED into (caller zero-fills)    */
    float* grad_sources;        /* (P,3) overwritten; trilinear only.  DIFFUS_POSE_F32_PER_RAY: (P,R,3), overwritten */
    float* grad_directions;     /* (P,R,3) overwritten; trilinear only (per pose, also when
                                   the directions were shared)                                */
    /* Fused forward + MSE loss + backward (one gather pass): when `target` is not NULL,
     * grad_frame is ignored and the kernel itself renders the frame and uses
     * d loss / d frame = grad_scale * (frame - target).  Optional outputs: fwd.frame (the
     * rendered frames) and loss[0] = loss_scale * sum((frame - target)^2).  With the mean
     * over n = P*R*(S-start) elements: grad_scale = 2/n, loss_scale = 1/n.               */
    const float* target;        /* (P,R,S-start) or NULL                                     */
    float grad_scale;
    float loss_scale;
    float* loss;                /* 1 float or NULL                                           */
    void* workspace;            /* diffus_render_bwd_workspace_bytes() bytes                 */
    int64_t workspace_bytes;
} DiffusRenderBwdArgs;

int32_t diffus_abi_version(void);
const char* diffus_error_string(int32_t code);

int64_t diffus_render_workspace_bytes(const DiffusRenderArgs* args);
int32_t diffus_render_forward(const DiffusRenderArgs* args, void* stream);
int64_t diffus_render_bwd_workspace_bytes(const DiffusRenderBwdArgs* args);
/* 1 when diffus_render_backward needs fwd.seg_prefix for these arguments, 0 when it does not (S-start <= 512, or rays of
 * 513..2048 columns with a pose gradient and no volume gradient: one CTA walks the two to four 512-column passes of such a
 * ray together, one warp each, and forms the prefixes itself -- no forward pre-pass), negative error code for invalid arguments.  Reads only
 * the shapes, enums and which output pointers are set. */
int32_t diffus_render_bwd_needs_prefix(const DiffusRenderBwdArgs* args);
int32_t diffus_render_backward(const DiffusRenderBwdArgs* args, void* stream);

/* Gauss-Newton system of each pose in one forward-mode pass: with res = frame - target and J the derivative of the frame
 * w.r.t. a rigid twist xi = (v, w) of the pose about its source (sources + v, directions rotated by Rot(w)),
 * or -- DIFFUS_POSE_F32_PER_RAY -- about the pose's PIVOT c_p, the float64 mean of its R origins: a sample moves as
 *   p_k = c_p + v + Rot(w) (s_i - c_p + k d_i),  i.e. origins c_p + v + Rot(w) (s_i - c_p) and directions Rot(w) d_i,
 *   loss[p] = sum res^2,   jtr[p] (6) = J^T res,   jtj[p] (6x6, full symmetric) = J^T J
 * over the R x (S-start) elements of pose p.  (2/n) jtr is the gradient of the mean-squared loss over n elements in twist
 * coordinates.  start > 0: the median-replaced coefficient's tangent is the mean of the tangents of the rays tied with the
 * median.  Trilinear sampler and float32 poses only (the nearest sampler has no pose derivative): anything else returns
 * DIFFUS_E_UNSUPPORTED.  Outputs are overwritten; the result is bit-identical from run to run (fixed-order sums). */
typedef struct DiffusGaussNewtonArgs {
    DiffusRenderArgs fwd;       /* the render; fwd.frame, fwd.seg_prefix and fwd.workspace are unused */
    const float* target;        /* (P,R,S-start)                                             */
    float* loss;                /* (P)                                                       */
    float* jtr;                 /* (P,6)                                                     */
    float* jtj;                 /* (P,6,6)                                                   */
    void* workspace;            /* diffus_render_gauss_newton_workspace_bytes() bytes        */
    int64_t workspace_bytes;
} DiffusGaussNewtonArgs;

int64_t diffus_render_gauss_newton_workspace_bytes(const DiffusGaussNewtonArgs* args);
int32_t diffus_render_gauss_newton(const DiffusGaussNewtonArgs* args, void* stream);

/* Gauss-Newton system of a whole tracked sweep: ONE rigid twist xi = (v, w) about ONE pivot c moves every sample of every pose,
 *   p_k = c + v + Rot(w) (s_i - c + k d_i),  s_i = the pose's source, or the ray's own origin for DIFFUS_POSE_F32_PER_RAY,
 * and the residuals of all P x R x (S-start) elements go into one system:
 *   loss[0] = sum res^2,   jtr (6) = J^T res,   jtj (6x6, full symmetric) = J^T J,   all float64.
 * With A_p = [[I, -[c_p - c]x], [0, I]] it is sum_p A_p^T (system of pose p about its own source / pivot c_p) A_p.  pivot: 3
 * doubles on the device, or NULL for the float64 mean of all P*R ray origins.  Validation, the median and NaN rules are those of
 * diffus_render_gauss_newton; the sums over rays run in a fixed order (bit-identical from run to run). */
typedef struct DiffusGaussNewtonSweepArgs {
    DiffusRenderArgs fwd;       /* the render; fwd.frame, fwd.seg_prefix and fwd.workspace are unused */
    const float* target;        /* (P,R,S-start)                                             */
    const double* pivot;        /* 3, device; NULL = mean of all ray origins                 */
    double* loss;               /* 1                                                         */
    double* jtr;                /* 6                                                         */
    double* jtj;                /* 6x6                                                       */
    void* workspace;            /* diffus_render_gauss_newton_sweep_workspace_bytes() bytes  */
    int64_t workspace_bytes;
} DiffusGaussNewtonSweepArgs;

int64_t diffus_render_gauss_newton_sweep_workspace_bytes(const DiffusGaussNewtonSweepArgs* args);
int32_t diffus_render_gauss_newton_sweep(const DiffusGaussNewtonSweepArgs* args, void* stream);

/* Clamped nearest-voxel indices of every ray point: the x, y, z int64 outputs of
 * custom_nearest_sampler (src/renderer.py:754-756, :816-819), cropped like
 * plot_beam_frame's return (:275).  Outputs are (P,R,S-start) int64. */
int32_t diffus_ray_indices(const DiffusRenderArgs* args, int64_t* x, int64_t* y, int64_t* z,
                           void* stream);

/* Sampled impedances along the rays, no propagation: the `values` output of
 * UltrasoundRenderer.trace_ray (src/renderer.py:89-180).  out is (P,R,S) (start ignored). */
int32_t diffus_trace_values(const DiffusRenderArgs* args, float* out, void* stream);
/* custom_nearest_sampler on explicit points (src/renderer.py:741-819): points (n,3) float32 voxel coordinates
 * -> values (n) and, if x, y, z are given, the clamped nearest-voxel indices (n each, int64). */
int32_t diffus_sample_points(const DiffusVolume* volume, const float* points, int64_t n, int32_t sampler,
                             float* values, int64_t* x, int64_t* y, int64_t* z, void* stream);
/* Backward of diffus_trace_values (autograd through the reference's sampler, src/renderer.py:758 / grid_sample): grad_values
 * (P,R,S) -> grad_volume (layout of args->volume, ACCUMULATED), and for the trilinear sampler grad_sources
 * (P,3) + grad_directions (P,R,3) (both or neither).  workspace: P*R*12 bytes (256-aligned) for pose gradients.
 * DIFFUS_POSE_F32_PER_RAY: grad_sources is (P,R,3) and no workspace is needed. */
int32_t diffus_trace_values_backward(const DiffusRenderArgs* args, const float* grad_values,
                                     float* grad_volume, float* grad_sources, float* grad_directions,
                                     void* workspace, int64_t workspace_bytes, void* stream);

/* compute_echo_traces (src/renderer.py:439-457, through propagate_full_rays_batched :412-436
 * and prop_single_ray :367-410) on explicit reflection coefficients refl (B,N):
 * echo (B,N+1) = [0, d0^(1), ..., d0^(N)], NaN -> 0.  Backward: grad_refl (B,N) overwritten. */
int32_t diffus_echo_forward(const float* refl, int64_t n_rays, int32_t n_interfaces, float* echo,
                            void* stream);
int32_t diffus_echo_backward(const float* refl, const float* grad_echo, int64_t n_rays,
                             int32_t n_interfaces, float* grad_refl, void* stream);

/* Fans for a batch of poses: generate_cone_directions (src/cone.py:242-259) generalised to
 * a leading pose dimension.  median (P,2) float64 (first two components of the median
 * direction), out (P,R,3) float32; float64 trigonometry then a float32 cast, like the
 * reference. */
int32_t diffus_cone_directions(const double* median, int64_t n_poses, int64_t n_rays,
                               double opening_angle, float* out, void* stream);

/* Fans in an arbitrary plane from pose PARAMETERS: generate_cone_directions (src/cone.py:242-259) generalised from the
 * z = 0 plane.  median (P,3) and hint (P,3) float32: m^ = median/|median|, u^ = hint made orthogonal to m^ and
 * normalised; out (P,R,3) float32, ray i = cos(a_i) m^ + sin(a_i) u^, a = linspace(-angle/2, angle/2, R), float64
 * arithmetic like the reference.  The backward maps d loss / d directions (P,R,3) to d loss / d median and
 * d loss / d hint (P,3 each, overwritten), so a pose-recovery step moves 9 floats per pose instead of 3R. */
int32_t diffus_fan_directions(const float* median, const float* hint, int64_t n_poses, int64_t n_rays,
                              double opening_angle, float* out, void* stream);
int32_t diffus_fan_directions_backward(const float* median, const float* hint, const float* grad_directions,
                                       int64_t n_poses, int64_t n_rays, double opening_angle,
                                       float* grad_median, float* grad_hint, void* stream);

/* Array probes from pose PARAMETERS, one origin per ray (render them with DIFFUS_POSE_F32_PER_RAY).  centre, median, hint
 * (P,3) float32; m^ and u^ as in diffus_fan_directions; origins and directions out (P,R,3) float32.
 *   DIFFUS_PROBE_CONVEX (opening_angle, radius rho >= 0): d_i = cos(a_i) m^ + sin(a_i) u^ with a = linspace(-angle/2,
 *     angle/2, R), formed exactly like diffus_fan_directions, and origin_i = centre + rho d_i (float64, then float32): the
 *     elements sit on an arc of radius rho and fire along its normals.  rho = 0 is the sector probe, bit for bit.
 *   DIFFUS_PROBE_LINEAR (width w > 0): d_i = m^ for every ray, origin_i = centre + t_i u^, t = linspace(-w/2, w/2, R).
 * The backward maps d loss / d origins and d loss / d directions (P,R,3 each) to d loss / d centre, median and hint (P,3
 * each, overwritten); float64 sums in a fixed order.  DIFFUS_E_SHAPE for a negative or non-finite radius, a width <= 0 or
 * not finite, a non-finite opening angle (convex), DIFFUS_E_ENUM for an unknown kind. */
#define DIFFUS_PROBE_CONVEX 0
#define DIFFUS_PROBE_LINEAR 1
int32_t diffus_probe_rays(int32_t kind, const float* centre, const float* median, const float* hint, int64_t n_poses,
                          int64_t n_rays, double opening_angle, double radius, double width, float* origins,
                          float* directions, void* stream);
int32_t diffus_probe_rays_backward(int32_t kind, const float* centre, const float* median, const float* hint,
                                   const float* grad_origins, const float* grad_directions, int64_t n_poses, int64_t n_rays,
                                   double opening_angle, double radius, double width, float* grad_centre,
                                   float* grad_median, float* grad_hint, void* stream);

/* ImpedanceEstimator (src/impedance.py:6-17): Linear(1,32)-ReLU-Linear(32,32)-ReLU-Linear(32,1).
 * params is the 1153-float concatenation [W1(32x1) b1(32) W2(32x32 row-major out,in) b2(32)
 * W3(1x32) b3(1)] in nn.Linear layout.  out[i] = out_scale * mlp(x[i]); when mask != NULL
 * voxels with mask[i] == 0 get `fill` instead (compute_impedance_volume, :46-54). */
#define DIFFUS_MLP_NPARAMS 1153
int32_t diffus_mlp_forward(const float* params, const float* x, const uint8_t* mask,
                           int64_t n, float out_scale, float fill, float* out, void* stream);
/* Same with an explicit execution path.  PIECEWISE: a ReLU network of ONE scalar is a piecewise-linear function of it (at most
 * 1088 breakpoints, ~60 in practice); every CTA builds the table of regions in float64 from the 1153 parameters and a voxel
 * costs a binary search and one fused multiply-add -- an HBM-bound pass, no dense contraction left (falls back to the layered
 * evaluation for weights with more than 256 regions).  CUDA_CORES evaluates the layers, layer 2 (M x 32 x 32) as fp32 FMAs.
 * AUTO = PIECEWISE for n >= 1024, CUDA cores below. */
#define DIFFUS_MLP_PATH_AUTO 0
#define DIFFUS_MLP_PATH_CUDA_CORES 1
/* 2 is rejected (DIFFUS_E_ENUM): it selected a removed tensor-core path and must not be reused. */
#define DIFFUS_MLP_PATH_PIECEWISE 3
int32_t diffus_mlp_forward_ex(const float* params, const float* x, const uint8_t* mask,
                              int64_t n, float out_scale, float fill, float* out, int32_t path,
                              void* stream);
/* grad_params (1153) is ACCUMULATED into (caller zero-fills): d/dparams of
 * sum_i grad_out[i] * out_scale * mlp(x[i]) over unmasked i.  workspace:
 * diffus_mlp_bwd_workspace_bytes(n) bytes. */
int64_t diffus_mlp_bwd_workspace_bytes(int64_t n);
int32_t diffus_mlp_backward(const float* params, const float* x, const uint8_t* mask,
                            const float* grad_out, int64_t n, float out_scale,
                            float* grad_params, void* workspace, int64_t workspace_bytes,
                            void* stream);
/* Same with an explicit path (DIFFUS_MLP_PATH_*).  PIECEWISE: inside a region d mlp / d params is affine in x, so the pass
 * over the volume only accumulates sum g and sum g x per region (float64 bins, no atomics) and a second small kernel turns
 * the moments into the 1153 gradients. */
int32_t diffus_mlp_backward_ex(const float* params, const float* x, const uint8_t* mask,
                               const float* grad_out, int64_t n, float out_scale,
                               float* grad_params, void* workspace, int64_t workspace_bytes,
                               int32_t path, void* stream);

/* d / d x of sum_i grad_out[i] * out_scale * mlp(x[i]): grad_x[i] = grad_out[i] * out_scale * mlp'(x[i]) (0 where masked) --
 * the input gradient the reference's nn.Sequential (src/impedance.py:10-17) hands to autograd.  mlp' is the slope of the linear
 * piece x[i] lies in (piecewise-linear table; layered evaluation above 256 pieces). */
int32_t diffus_mlp_input_grad(const float* params, const float* x, const uint8_t* mask, const float* grad_out,
                              int64_t n, float out_scale, float* grad_x, void* stream);

/* Scan conversion: differentiable_splat (src/renderer.py:694-737).  c0,c1,c2 are the three coordinate
 * arrays (float32, n each -- the reference casts x, y, z to float32, :709-710), intensities n float32.
 * The two axes of largest variance are picked on the device; pixels are rounded and clamped; duplicate
 * pixels keep the sample with the highest index (the reference's non-accumulating indexed write); image
 * and hit mask are blurred with the normalised (int(6 sigma)|1)^2 Gaussian; out is (W,H) =
 * (blur(image) / (blur(mask) + 1e-8))^T.  Backward: grad_out (W,H) -> grad_intensities (n), every
 * duplicate receiving its pixel's gradient, as torch's index_put_ backward does. */
int64_t diffus_splat_workspace_bytes(int32_t H, int32_t W);
int32_t diffus_splat_forward(const float* c0, const float* c1, const float* c2, const float* intensities,
                             int64_t n, int32_t H, int32_t W, float sigma, float* out, void* workspace,
                             int64_t workspace_bytes, void* stream);
int32_t diffus_splat_backward(const float* c0, const float* c1, const float* c2, const float* intensities,
                              int64_t n, int32_t H, int32_t W, float sigma, const float* grad_out,
                              float* grad_intensities, void* workspace, int64_t workspace_bytes,
                              void* stream);

/* ---- training-loop pieces around the path (SURVEY.md 8 row f3; reference notebooks) ------------------------------- */

/* torch.optim.Adam step (the optimiser of src/impedance.py:26-35 and of the training notebooks; no amsgrad) on n <= 65536
 * parameters in ONE launch: g = grad_scale * grads (+ weight_decay * p), moments, bias correction, update, step counter.
 * state = [exp_avg (n) | exp_avg_sq (n) | step (1)] floats, zero-filled by the caller before the first step. */
int32_t diffus_adam_step(float* params, const float* grads, float* state, int64_t n, float lr, float beta1, float beta2,
                         float eps, float weight_decay, float grad_scale, void* stream);

/* One slice of a LINEAR or BRICK volume, `index` along `axis` (0, 1, 2), as a dense row-major 2-D array over the two other
 * axes: scatter = 0 copies volume -> slice, scatter = 1 copies slice -> volume.  ImpedanceLearner.training_forward's slice
 * mode (notebooks/[DEMO] Train MRI to Impedance MLP - GPU.ipynb cell 16: Z_vol = x.clone(); Z_vol[:, :, k] = mlp(x[:, :, k])). */
int32_t diffus_volume_slice(float* volume, const int32_t dim[3], int32_t layout, int32_t axis, int32_t index, float* slice,
                            int32_t scatter, void* stream);

/* rotate_around_apex (src/renderer.py:655-692): x_rot = cos (x - shift) - sin z + apex0, z_rot = sin (x - shift) + cos z + apex1
 * (the reference hard-wires shift = 128), one rounding per operation like the reference's torch expression. */
int32_t diffus_rotate_around_apex(const float* x, const float* z, int64_t n, float cos_a, float sin_a, float shift, float apex0,
                                  float apex1, float* x_rot, float* z_rot, void* stream);

/* The 1-D convolution of compute_gaussian_pulse (src/renderer.py:459-479: F.conv1d of the echo lines with one pulse, a
 * cross-correlation): out[b][o] = sum_t w[t] in[b][o + t - pad], zero outside the row, out is (rows, n_in + 2 pad - taps + 1).
 * taps <= 128.  The backward w.r.t. the rows: grad_in (rows, n_in) from grad_out (rows, n_out). */
int32_t diffus_conv1d_rows_forward(const float* in, int64_t rows, int32_t n_in, const float* w, int32_t taps, int32_t pad,
                                   float* out, void* stream);
int32_t diffus_conv1d_rows_backward(const float* grad_out, int64_t rows, int32_t n_in, const float* w, int32_t taps, int32_t pad,
                                    float* grad_in, void* stream);

/* Log compression (north_star's "log-compressed B-mode"; the reference's only form is process_rf_to_bmode,
 * notebooks/[DEMO] Renderer Alternatives.ipynb cell 14: log1p(envelope) / max).
 * diffus_log_compress_*: out = log1p(|img|) / max(log1p(|img|)) over n pixels, and its backward (the maximum's gradient is
 * spread evenly over its ties, torch's rule); max_out (1 float) may be NULL.
 * diffus_rf_to_bmode: the notebook function itself on (n_rays, n_samples) RF lines: envelope = |analytic signal| with the
 * analytic signal of scipy.signal.hilbert along the samples -- its imaginary part is the circular convolution with
 * hilbert_kernel = Im(ifft(h)) (n_samples floats, h = scipy's one-sided spectrum weights; host-computed) -- then log1p and
 * division by the maximum over the whole array.  workspace: 4 bytes. */
int32_t diffus_log_compress_forward(const float* img, int64_t n, float* out, float* max_out, void* stream);
int32_t diffus_log_compress_backward(const float* img, const float* grad_out, int64_t n, float* grad_img, void* stream);
int32_t diffus_rf_to_bmode(const float* profiles, int64_t n_rays, int32_t n_samples, const float* hilbert_kernel, float* out,
                           void* workspace, int64_t workspace_bytes, void* stream);

/* Losses of the training notebooks on (H, W) images, forward and backward w.r.t. the synthetic image.
 * masked MSE + edge ([DEMO] Train MRI to Impedance MLP.ipynb cell 19, UltrasoundSynthesisModel.loss / gradient_loss):
 *   loss = mean((a - b)^2 over mask) + edge_weight * mean(| |a[:,1:] - a[:,:-1]| - |b[:,1:] - b[:,:-1]| | over mask[:,1:]);
 *   stats (3 floats) = [loss, count(mask), count(mask[:,1:])], written by the forward and read by the backward.
 * 1 - SSIM ([DEMO] Train MRI to Impedance MLP - GPU.ipynb cell 16): with normalize != 0 the synthetic image is first mapped
 *   to (s - min) / (max - min + 1e-8); SSIM is piq.ssim's algorithm (Gaussian window ksize x ksize, sigma, VALID filtering,
 *   k1, k2, data_range 1, mean over the map; piq is not vendored by the reference: defaults 11, 1.5, 0.01, 0.03).
 *   The backward needs the workspace the forward filled. */
int32_t diffus_masked_mse_edge_forward(const float* synth, const float* real, const uint8_t* mask, int32_t H, int32_t W,
                                       float edge_weight, float* stats, void* stream);
int32_t diffus_masked_mse_edge_backward(const float* synth, const float* real, const uint8_t* mask, int32_t H, int32_t W,
                                        float edge_weight, const float* stats, const float* grad_loss, float* grad_synth,
                                        void* stream);
int64_t diffus_ssim_workspace_bytes(int32_t H, int32_t W, int32_t ksize);
int32_t diffus_ssim_loss_forward(const float* synth, const float* real, int32_t H, int32_t W, int32_t ksize, float sigma,
                                 float k1, float k2, int32_t normalize, float* loss, void* workspace, int64_t workspace_bytes,
                                 void* stream);
int32_t diffus_ssim_loss_backward(const float* synth, const float* real, int32_t H, int32_t W, int32_t ksize, float sigma,
                                  int32_t normalize, const float* grad_loss, float* grad_synth, void* workspace,
                                  int64_t workspace_bytes, void* stream);

/* MRI preprocessing in front of the MLP (src/utils.py:12-39, called from compute_impedance_volume,
 * src/impedance.py:46-47).  diffus_brain_mask: create_brain_mask = (volume > threshold), `iterations`
 * binary dilations then `iterations` binary erosions (scipy defaults: 6-neighbour cross, border value 0;
 * the reference uses 2); mask and scratch hold D*H*W bytes each.  diffus_masked_zscore:
 * zscore_normalize = (volume - mean) / (std + 1e-8), mean and unbiased std over voxels with mask != 0;
 * workspace >= 64 bytes. */
int32_t diffus_brain_mask(const float* volume, const int32_t dim[3], float threshold, int32_t iterations,
                          uint8_t* mask, uint8_t* scratch, void* stream);
int32_t diffus_masked_zscore(const float* volume, const uint8_t* mask, int64_t n, float* out,
                             void* workspace, int64_t workspace_bytes, void* stream);

/* LINEAR (D,H,W) -> BRICK copy of a volume (and back, for gradients). dst holds
 * diffus_brick_elems(dim) floats. */
int64_t diffus_brick_elems(const int32_t dim[3]);
int32_t diffus_volume_to_bricks(const float* linear, const int32_t dim[3], float* bricks, void* stream);
int32_t diffus_bricks_to_volume(const float* bricks, const int32_t dim[3], float* linear, void* stream);
/* LINEAR -> QUAD copy; the quad buffer holds diffus_quad_elems(dim) FLOATS (4 per padded voxel, 16-byte aligned). */
int64_t diffus_quad_elems(const int32_t dim[3]);
int32_t diffus_volume_to_quads(const float* linear, const int32_t dim[3], float* quads, void* stream);

/* Isotropic Gaussian smoothing of a (D,H,W) float32 volume: scipy.ndimage.gaussian_filter(src, sigma, mode='nearest',
 * truncate=truncate) -- weights exp(-x^2 / (2 sigma^2)) over x = -r..r, r = int(truncate * sigma + 0.5), normalised to sum 1
 * in float64 and rounded to float32; taps beyond a face repeat the edge voxel (the renderer's border rule), also when r
 * exceeds a dimension.  sigma <= 1e-15 (scipy skips the axes) or r = 0 is an exact copy.  Three separable passes in fp32,
 * p2 src -> dst, p1 dst -> scratch, p0 scratch -> dst; bit-identical from run to run.  dst and scratch hold D*H*W floats
 * each and may not overlap src or each other.  Returns DIFFUS_E_SHAPE for sigma < 0, truncate <= 0 or either not finite,
 * DIFFUS_E_UNSUPPORTED for r > 64.  The scale space of coarse-to-fine pose recovery. */
int32_t diffus_volume_gaussian_blur(const float* src, const int32_t dim[3], float sigma, float truncate, float* dst,
                                    float* scratch, void* stream);

/* TEXTURE layout.  The ONLY entry points of this library that allocate and free device memory (a CUDA array of
 * dim[0] layers x dim[1] x dim[2] float32 texels and a texture object): create once per volume, update after the
 * LINEAR tensor changed (one device-to-device copy enqueued on `stream`), destroy when done.  `*texture_object` is what
 * goes into DiffusVolume.data (cast to a pointer) with layout = DIFFUS_LAYOUT_TEXTURE; `*array_handle` is opaque.
 * Limits: dim[0] <= 2048 layers, dim[1], dim[2] <= 32768. */
int32_t diffus_volume_texture_create(const float* linear, const int32_t dim[3], uint64_t* texture_object,
                                     uint64_t* array_handle, void* stream);
int32_t diffus_volume_texture_update(uint64_t array_handle, const float* linear, const int32_t dim[3], void* stream);
int32_t diffus_volume_texture_destroy(uint64_t texture_object, uint64_t array_handle);

/* Measurement aid for the roofline (SURVEY 8d), not part of the render path: every thread issues
 * `reads_per_thread` independent 4-byte loads at pseudo-random 32-byte-sector-aligned positions of buf (n_floats
 * floats) and stores their sum in sink[thread].  Over a 64 MiB buffer this is the L2 -> SM random-sector rate the
 * gather-bound march competes with; over a buffer larger than L2 it is the HBM random-sector rate. */
int32_t diffus_gather_probe(const float* buf, int64_t n_floats, int32_t reads_per_thread, int64_t n_threads,
                            uint32_t seed, float* sink, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* DIFFUS_B200_H */
