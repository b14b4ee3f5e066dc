/*
 * ffb200.h -- C ABI of libffb200.so, the B200 (sm_100a) hot path of Fireflies.
 *
 * The reference (Henningson/Fireflies) is pure Python/PyTorch and exposes no FFI; its
 * drop-in boundary is the Python API (SURVEY.md section 8(b)).  This header is the boundary
 * *behind* that API: every entry point below replaces the body of one or more reference
 * functions, cited as path:line relative to the reference tree.  The Python package
 * `fireflies_b200` binds these with ctypes (fireflies_b200/_native.py); INTEGRATION.md shows
 * the stub a reference maintainer would add.
 *
 * Conventions
 *   - plain C types only; every pointer is a DEVICE pointer on the current CUDA device unless
 *     the parameter name ends in `_host`; the caller owns every buffer, kernels never allocate;
 *   - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream); every call is
 *     asynchronous with respect to the host;
 *   - return value: 0 = OK, >0 = cudaError_t from a launch/runtime call, <0 = argument error
 *     (FFB_E_*); ffb_last_error_string() describes the last failure on the calling thread;
 *   - no global mutable state; re-entrant across streams;
 *   - all floating point is IEEE fp32 ("f32") except the NURBS evaluator (fp64, section 5); index outputs are int32.
 *
 * Texture orientation: "natural" = [ts1, ts0] row-major, rows pair with points[:,1] and columns
 * with points[:,0] -- the orientation of rasterize_points(...).sum(0)
 * (fireflies/graphics/rasterization.py:18-30).  "transposed" = [ts0, ts1], the orientation
 * baked_sum_2 returns (fireflies/graphics/rasterization.py:318).
 */
#ifndef FFB200_H
#define FFB200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define FFB_VERSION 100

#if defined(__GNUC__)
#define FFB_API __attribute__((visibility("default")))
#else
#define FFB_API
#endif

#define FFB_E_ARG      (-1)   /* invalid argument (null pointer, non-positive size, ...)   */
#define FFB_E_WORKSPACE (-2)  /* workspace too small                                       */
#define FFB_E_LIMIT    (-3)   /* size beyond a compiled limit (see message)                */
#define FFB_E_UNSUPPORTED (-4) /* the fused path does not cover this case; use the unfused calls */

FFB_API int         ffb_version(void);
FFB_API const char* ffb_last_error_string(void);

/* ------------------------------------------------------------------------------------------
 * 1. Laser splat  (fireflies/graphics/rasterization.py)
 * ------------------------------------------------------------------------------------------ */

/* Reduction windows.  num_std > 0 selects the footprint-limited ("baked") semantics of
 * baked_sum / baked_sum_2 / baked_softor / baked_softor_2 (rasterization.py:164-472):
 * footprint = odd(floor(sqrt(sigma)) * num_std), clipped exactly like the reference slices.
 * num_std == 0 selects the dense semantics of rasterize_points + sum/softor
 * (rasterization.py:7-37,156-161): every texel, evaluated up to the radius beyond which
 * exp(-(d^2/sigma)^2) is exactly 0 in fp32 (sum) or 1-g rounds to exactly 1 (softor). */
typedef struct ffb_splat_desc {
    int32_t B;              /* scene samples                                                */
    int32_t N;              /* points per sample                                            */
    int32_t ts0, ts1;       /* texture_size[0] (columns, pairs with p[:,0]), [1] (rows)     */
    float   sigma;          /* the reference's `sigma` (divides d^2; NOT squared again)     */
    int32_t num_std_sum;    /* 4 = baked_sum default; 0 = dense                             */
    int32_t num_std_softor; /* 5 = baked_softor default; 0 = dense                          */
    int64_t pts_batch_stride; /* elements between samples in `pts`; 0 = one pattern shared  */
} ffb_splat_desc;

/* Bytes of scratch the splat calls need for this descriptor (binning tables). */
FFB_API size_t ffb_splat_workspace_bytes(const ffb_splat_desc* d);

/* Bins the points of every sample into texture tiles and computes each point's integer clip
 * window.  Must precede ffb_splat_fwd/ffb_splat_bwd on the same workspace (same stream order).
 *   pts         [B,N,2] f32 in [0,1] (x,y) -- or [N,2] with pts_batch_stride = 0
 *   windows_out NULL or int32 [Bp,N,2,2,3]: per point, per reduction (0 = sum, 1 = softor), per
 *               axis, the reference's (wo, rs, re) slice triple (rasterization.py:199-230);
 *               Bp = B, or 1 when the pattern is shared.  Only defined for baked reductions. */
FFB_API int ffb_splat_prepare(const ffb_splat_desc* d, const float* pts, void* workspace, size_t workspace_bytes,
                      int32_t* windows_out, void* stream);

/* Fused splat + reduce, forward.  Replaces rasterize_points+sum/softor and the baked_* family.
 *   out_sum     NULL or f32 [B,ts1,ts0] (natural) / [B,ts0,ts1] if sum_transposed
 *   out_softor  NULL or f32 [B,ts1,ts0] */
FFB_API int ffb_splat_fwd(const ffb_splat_desc* d, const float* pts, const void* workspace,
                  float* out_sum, int sum_transposed, float* out_softor, void* stream);

/* Backward of ffb_splat_fwd w.r.t. pts (the autograd the reference gets from torch,
 * SURVEY.md 8(a) a7).  d_pts [B,N,2] f32 is OVERWRITTEN (zeroed, then accumulated).
 *   g_sum        NULL or upstream gradient of out_sum, same layout as out_sum
 *   g_softor     NULL or upstream gradient of out_softor
 *   saved_softor NULL or the out_softor that ffb_splat_fwd wrote for these points (what torch autograd
 *                keeps for prod's backward): the per-texel product is then read back as 1 - out_softor
 *                instead of being rebuilt by a first pass over the candidates */
FFB_API int ffb_splat_bwd(const ffb_splat_desc* d, const float* pts, const void* workspace,
                  const float* g_sum, int sum_transposed, const float* g_softor, const float* saved_softor,
                  float* d_pts, void* stream);

/* Fused backward of the only optimisation loop the reference ships (test_point_reg,
 * fireflies/graphics/rasterization.py:586-607: `loss = L1Loss(softored, summed); loss.backward()`):
 * per-sample loss = mean |out_softor - out_sum| over the two textures AS STORED (same memory index), and
 * d loss / d pts, in one pass over the forward's outputs -- the texture gradients are formed in registers
 * instead of being written by ffb_l1_loss_fwd_bwd and read back by ffb_splat_bwd.
 *   out_sum, out_softor  what ffb_splat_fwd wrote for these points (both required)
 *   sum_transposed       layout of out_sum as in ffb_splat_fwd; with 1 the textures must be square
 *                        (the reference pairs softor[ts1,ts0] with baked_sum_2's [ts0,ts1] elementwise)
 *   loss_out f32 [B] and d_pts f32 [B,N,2] are OVERWRITTEN.
 * Returns FFB_E_UNSUPPORTED when the textures cannot be described to the TMA unit (base not 16-byte
 * aligned, sides not multiples of 4) or the descriptor needs the general kernels; callers then use
 * ffb_l1_loss_fwd_bwd + ffb_splat_bwd. */
FFB_API int ffb_splat_bwd_l1(const ffb_splat_desc* d, const float* pts, const void* workspace,
                     const float* out_sum, int sum_transposed, const float* out_softor,
                     float* loss_out, float* d_pts, void* stream);

/* sum over the sample axis: out[N*2] = sum_b in[b, N*2]  (fixed order -> deterministic);
 * used to fold per-sample pattern gradients before the allreduce. */
FFB_API int ffb_reduce_over_samples(const float* in, int32_t B, int64_t row_elems, float* out, void* stream);

/* One level of the same fold for texture-sized rows: out[g, :] = sum of samples 8g .. 8g+7 (fixed order), out is
 * [ceil(B/8), row_elems].  Applied repeatedly it sums B upstream texture gradients at streaming bandwidth (the
 * shared-pattern backward: one pattern for all scenes of a step, the backward being linear in the upstream gradients).
 * Rows must be 16-byte aligned multiples of 4 elements (FFB_E_UNSUPPORTED otherwise). */
FFB_API int ffb_reduce_sample_groups(const float* in, int32_t B, int64_t row_elems, float* out, void* stream);

/* The path's only exchange (SURVEY.md 8(e)) fused with the fold that precedes it: out[row_elems] = sum over ALL
 * ranks of sum_b in[b, :], one kernel, over NVLink peer memory (no NCCL call).  recv_bufs[r] / flag_bufs[r] are host
 * arrays of `world` DEVICE pointers into symmetric memory of rank r: recv f32 [2][world][row_elems] (double buffered
 * by epoch parity), flags u32 [world][ceil(row_elems/32)] zero-initialised once.  `epoch` is 1, 2, 3, ... -- the same
 * on every rank for the same step.  Each CTA pushes its partial sums into every peer's slot [rank], publishes a flag,
 * waits for the peers' flags of the same CTA and adds the slots in rank order (bit-identical result on all ranks).
 * err_flag (device int32) is set when a peer did not arrive within the spin bound.  row_elems <= 37888, world <= 8. */
FFB_API int ffb_fold_allreduce(const float* in, int32_t B, int64_t row_elems, float* const* recv_bufs, uint32_t* const* flag_bufs,
                       int32_t rank, int32_t world, uint32_t epoch, float* out, int32_t* err_flag, void* stream);

/* API-compatibility dense splat: rasterize_points (rasterization.py:7-37) -> [N,ts1,ts0],
 * and its backward given the upstream gradient of that tensor. */
FFB_API int ffb_splat_dense_fwd(const float* pts, int32_t N, int32_t ts0, int32_t ts1, float sigma,
                        float* out, void* stream);
FFB_API int ffb_splat_dense_bwd(const float* pts, int32_t N, int32_t ts0, int32_t ts1, float sigma,
                        const float* g_out, float* d_pts, void* stream);
/* The same for points given in texel units (rasterize_points_in_non_ndc, fireflies/graphics/rasterization.py:38-63:
 * no multiplication by texture_size). */
FFB_API int ffb_splat_dense_px_fwd(const float* pts, int32_t N, int32_t ts0, int32_t ts1, float sigma,
                           float* out, void* stream);
FFB_API int ffb_splat_dense_px_bwd(const float* pts, int32_t N, int32_t ts0, int32_t ts1, float sigma,
                           const float* g_out, float* d_pts, void* stream);

/* ---- line and depth rasterisers (SURVEY.md 8(f) row 2) ------------------------------------------------
 * lines f32 [L,2,2] = (start, end) x (x, y) in units of the texture size (16-byte aligned); the squared
 * point-to-segment distance d2 gives g = exp(-(d2*d2)/(sigma*sigma))  (rasterize_lines,
 * fireflies/graphics/rasterization.py:107-153; the reference's in-place scaling of its argument, :122-123,
 * is not reproduced: `lines` is read-only here).
 *   ffb_lines_dense_fwd/bwd   the reference's dense [L,ts1,ts0] tensor and its backward (d_lines [L,2,2],
 *                             OVERWRITTEN) -- API compatibility.
 *   ffb_lines_reduce_fwd/bwd  sum and/or soft-OR over the lines in one pass (what test_line_reg, :684-697,
 *                             and the epipolar regulariser reduce the dense tensor to): outputs [ts1,ts0];
 *                             the backward takes the upstream gradients of those (NULL = not used). */
FFB_API int ffb_lines_dense_fwd(const float* lines, int32_t L, int32_t ts0, int32_t ts1, float sigma, float* out, void* stream);
FFB_API int ffb_lines_dense_bwd(const float* lines, int32_t L, int32_t ts0, int32_t ts1, float sigma, const float* g_out,
                        float* d_lines, void* stream);
FFB_API int ffb_lines_reduce_fwd(const float* lines, int32_t L, int32_t ts0, int32_t ts1, float sigma, float* out_sum,
                         float* out_softor, void* stream);
FFB_API int ffb_lines_reduce_bwd(const float* lines, int32_t L, int32_t ts0, int32_t ts1, float sigma, const float* g_sum,
                         const float* g_softor, float* d_lines, void* stream);

/* rasterize_depth (fireflies/graphics/rasterization.py:66-104): the dense point splat of pts [N,2] divided by
 * its per-point maximum over the frame and scaled by depth [N] -> out [N,ts1,ts0]; its backward w.r.t. pts
 * and depth (scratch: f32 [N,3]; d_pts [N,2] / d_depth [N] may be NULL, both OVERWRITTEN);
 * ffb_depth_softor_fwd = one level of subsampled_point_raster (:538-549): soft-OR over the points -> [ts1,ts0]. */
FFB_API int ffb_depth_dense_fwd(const float* pts, const float* depth, int32_t N, int32_t ts0, int32_t ts1, float sigma, float* out,
                        void* stream);
FFB_API int ffb_depth_dense_bwd(const float* pts, const float* depth, int32_t N, int32_t ts0, int32_t ts1, float sigma,
                        const float* g_out, float* scratch, float* d_pts, float* d_depth, void* stream);
FFB_API int ffb_depth_softor_fwd(const float* pts, const float* depth, int32_t N, int32_t ts0, int32_t ts1, float sigma, float* out,
                         void* stream);

/* mean |a-b| and its gradients (torch.nn.L1Loss as used by test_point_reg, rasterization.py:591-599).
 *   a is natural [B,ts1,ts0]; b is natural or transposed ([B,ts0,ts1]) per b_transposed.
 *   loss_out f32 [B] (OVERWRITTEN); g_a / g_b (may be NULL) receive d loss_b / d a, d b in the
 *   layouts of a and b. */
FFB_API int ffb_l1_loss_fwd_bwd(const float* a, const float* b, int b_transposed, int32_t B, int32_t ts0, int32_t ts1,
                        float* loss_out, float* g_a, float* g_b, void* stream);

/* ------------------------------------------------------------------------------------------
 * 3. Sampling  (fireflies/sampling)
 * ------------------------------------------------------------------------------------------ */

#define FFB_MODE_TRAIN     0  /* counter-based Philox4x32-10 draws                              */
#define FFB_MODE_EVAL      1  /* deterministic stepping, sampling/base.py:64-74 incl. its aliasing */
#define FFB_MODE_INJECTED  2  /* variates supplied by the caller (parity tests / torch's RNG stream) */

#define FFB_SAMPLER_UNIFORM        0  /* UniformSampler          sampling/uniform.py:16-19: u*(max-min)+min per component */
#define FFB_SAMPLER_SCALAR_TO_VEC3 1  /* UniformScalarToVec3Sampler sampling/uniform_scalar_to_vec3.py:18-38: 1 draw, written 3x */
#define FFB_SAMPLER_GAUSSIAN       2  /* GaussianSampler         sampling/gaussian_distribution.py:19-20: mean + std*z, unclamped */

/* One sampler row.  `dim` is the number of state components (1 or 3).  The eval fields are the
 * in/out state of Sampler.sample_eval: `cur` = _current_step, `aliased` = _current_step is the
 * same tensor as _min_range (after the first wrap), in which case stepping also moves vmin. */
typedef struct ffb_sampler {
    int32_t kind;           /* FFB_SAMPLER_*                                                 */
    int32_t dim;            /* 1 or 3                                                        */
    int32_t aliased;        /* eval state                                                    */
    float   step;           /* eval_step_size (0.01)                                         */
    float   vmin[3], vmax[3], cur[3];
    float   mean[3], std[3];/* FFB_SAMPLER_GAUSSIAN only                                     */
} ffb_sampler;

/* Draws B successive samples from each of S samplers: out[b,s,0:3] (unused components = 0;
 * SCALAR_TO_VEC3 rows carry the draw in all three).
 *   samplers    DEVICE array [S]; in FFB_MODE_EVAL its eval state is advanced B times in place
 *   seed, sample0  FFB_MODE_TRAIN: Philox key / global index of sample 0 of this call; a draw
 *               depends only on (seed, sample0+b, s, component) -- never on B, the GPU or rank
 *   variates    FFB_MODE_INJECTED: f32 [B,S,3] uniform variates in [0,1) (standard normal ones
 *               for GAUSSIAN rows); else NULL */
FFB_API int ffb_sample(ffb_sampler* samplers, int32_t S, int32_t B, int32_t mode, uint64_t seed, uint64_t sample0,
               const float* variates, float* out, void* stream);

/* randomBetweenTensors (utils/math.py:170-175) with the torch.rand variates supplied:
 * out[i] = u[i]*(b[i]-a[i])+a[i], three separately rounded fp32 ops like torch.  All f32 [n]. */
FFB_API int ffb_uniform_between(const float* a, const float* b, const float* u, int64_t n, float* out, void* stream);

/* AnimationSampler frame indices (sampling/animation.py:27-45), int32 out[b,m].
 * train: min + floor(u*(max-min)) with Philox (python's random.randint stream is not reproducible
 * on a device; the injected path takes host-drawn indices instead); eval: min..max INCLUSIVE walk
 * continuing from cur[m] (in/out, device). */
FFB_API int ffb_sample_anim_index(const int32_t* amin, const int32_t* amax, int32_t* cur, int32_t M, int32_t B, int32_t mode,
                          uint64_t seed, uint64_t sample0, int32_t* out, void* stream);

/* ------------------------------------------------------------------------------------------
 * 2. Per-entity compose + vertex transforms  (fireflies/entity, fireflies/utils/math.py)
 * ------------------------------------------------------------------------------------------ */

#define FFB_ENTITY_PLAIN  0   /* (T+C) @ R @ W          entity/base.py:220-234                */
#define FFB_ENTITY_MESH   1   /* (T+C) @ R @ S @ W      entity/mesh.py:141-150                */

typedef struct ffb_entity {
    int32_t kind;           /* FFB_ENTITY_*                                                  */
    int32_t parent;         /* row of the parent entity, -1 = root (entity/base.py:239-244); must be < own row:
                               a row whose parent does not precede it gets NaN matrices (loud, not a dropped parent) */
    int32_t randomizable;   /* 0: local = W  (randomize() returns early, entity/base.py:221-222) */
    int32_t s_translation;  /* sampler rows feeding this entity; -1 = zeros / zeros / ones    */
    int32_t s_rotation;
    int32_t s_scale;
    float   centroid[3];    /* entity/base.py:51-54                                          */
    float   _pad;
    float   world[16];      /* row-major _world                                              */
} ffb_entity;

/* out_world[b,e] = parent chain of ((T+C) @ R [@ S] @ W) built from sampled[b, s_*, :].
 * Rotation = Pitch(r2) @ Yaw(r1) @ Roll(r0) with fp64 trig rounded to fp32 (utils/math.py:24-60,
 * entity/base.py:194-207).   entities DEVICE [E]; sampled f32 [B,S,3]; out_world f32 [B,E,16]. */
FFB_API int ffb_compose_world(const ffb_entity* entities, int32_t E, int32_t B, const float* sampled, int32_t S,
                      float* out_world, void* stream);

/* Batched transform_points (utils/math.py:220-228) over up to FFB_MAX_MESHES meshes per call, with
 * optional animation-frame gather (entity/mesh.py:158-165,183-198):
 *   out[b, voff_m + v] = persp_div(world[b, entity_m] @ [src_m[v], 1])
 *   src_m = frames_m[anim_idx[b,m]] if frames_m else verts + 3*voff_m.
 * The mesh table is passed BY VALUE (host struct). */
#define FFB_MAX_MESHES 32
typedef struct ffb_mesh_table {
    int32_t M;
    int32_t voff[FFB_MAX_MESHES + 1];   /* vertex offsets into verts / out rows              */
    int32_t entity[FFB_MAX_MESHES];     /* row of `world` per mesh                           */
    int32_t nframes[FFB_MAX_MESHES];    /* 0 = not animated                                  */
    const float* frames[FFB_MAX_MESHES];/* DEVICE f32 [nframes, V_m, 3] or NULL              */
} ffb_mesh_table;

FFB_API int ffb_transform_vertices(const ffb_mesh_table* meshes, const float* verts, int32_t E, int32_t B,
                           const int32_t* anim_idx, const float* world, float* out, void* stream);

/* transform_points / transform_directions for one matrix (utils/math.py:220-235):
 * out[v] = persp_div(T @ [x,y,z,1])  or  (T @ [x,y,z,0])[:3].   T f32 [16] row-major, DEVICE. */
FFB_API int ffb_transform_points(const float* pts, int64_t V, const float* T, int as_directions, float* out, void* stream);
/* its backward w.r.t. pts (torch autograd in the reference; the laser rays are optimised through
 * projectRaysToNDC): d_pts[v] = J(pts[v])^T g_out[v]. */
FFB_API int ffb_transform_points_bwd(const float* pts, int64_t V, const float* T, int as_directions, const float* g_out,
                                     float* d_pts, void* stream);

/* Laser glue (projection/laser.py:199-206, 262-290).  M = K @ FLIP_Y and Minv are DEVICE f32 [16].
 * rays_to_ndc: ndc[n] = persp_div(M @ [ray,1]).
 * clamp_to_fov: clamp ndc xy to [clamp_lo, clamp_hi] (= [1-c, c], the host rounds 1-c in fp64 like
 * python does), un-project through Minv, renormalise. */
FFB_API int ffb_rays_to_ndc(const float* rays, int32_t N, const float* M, float* ndc, void* stream);
FFB_API int ffb_clamp_to_fov(const float* rays, int32_t N, const float* M, const float* Minv, float clamp_lo, float clamp_hi,
                     float* rays_out, void* stream);

/* Laser.randomize_laser_out_of_bounds (M = `_perspective`, bounds (0, 1)) and randomize_camera_out_of_bounds
 * (ndc given, bounds (-1, 1)) -- fireflies/projection/laser.py:208-249 -- in one launch without a host sync.
 * rays f32 [N,3] IN/OUT: a ray whose NDC x or y is >= hi or <= lo is replaced by Minv applied to (u0, u1, -1)
 * (projectNDCPointsToWorld); if any ray was replaced ALL rays are renormalised, otherwise `rays` is untouched
 * (the reference returns before its normalise).  Exactly one of M ([4,4], projects the rays) and ndc ([N,3],
 * coordinates computed by the caller) is non-NULL.  u comes from `variates` ([K,3] rows consumed in ray order,
 * the reference's torch.rand(K, 3)) or, when NULL, from Philox keyed by (seed, ray index, counter).
 * respawned_out (device int32, nullable) receives K. */
FFB_API int ffb_respawn_rays(float* rays, int32_t N, const float* M, const float* ndc, float lo, float hi, const float* Minv,
                     uint64_t seed, uint64_t counter, const float* variates, int32_t* respawned_out, void* stream);

/* ------------------------------------------------------------------------------------------
 * 4. Post-processing  (fireflies/postprocessing)
 * ------------------------------------------------------------------------------------------ */
typedef struct ffb_post_desc {
    int32_t B, H, W;        /* frames [B,H,W] f32                                             */
    int32_t blur_ky, blur_kx; /* 0 = no blur stage; kornia gaussian_blur2d kernel_size (odd, <= 15) */
    float   blur_sy, blur_sx;
    int32_t noise;          /* 0 = no noise stage; 1 = WhiteNoise (white_noise.py:16-20)       */
    float   noise_mean, noise_std;
    uint64_t seed;          /* Philox key for the native noise stream                         */
    uint64_t frame0;        /* global index of frame 0 (stream independent of batching/rank)   */
} ffb_post_desc;

/* out = clip?(noise?(blur?(img))) per frame; gates u8 [B,2] = (blur gate, noise gate) -- the
 * Bernoulli draws of BasePostProcessingFunction.apply (postprocessing/base.py:10-14) made by the
 * caller; NULL = all stages on.  noise_injected NULL or f64 [B,H,W] normal variates already
 * scaled by mean/std, added in fp64 like numpy does (white_noise.py:17; parity tests).  img and out must not alias when a blur stage is present. */
FFB_API int ffb_postprocess(const ffb_post_desc* d, const float* img, const uint8_t* gates,
                    const double* noise_injected, float* out, void* stream);

/* Backward of ffb_postprocess's blur stage w.r.t. its input, per frame: g_in = A^T g_out, A = the separable Gaussian blur
 * with kornia's reflect border that ffb_postprocess applies for d's blur fields (same rules: odd sizes <= 15,
 * kernel/2 < side).  d->noise must be 0; seed / frame0 are ignored; no gates.  g_out, g_in f32 [B,H,W], must not alias. */
FFB_API int ffb_blur_bwd(const ffb_post_desc* d, const float* g_out, float* g_in, void* stream);

/* ApplySilhouette.post_process (fireflies/postprocessing/apply_silhouette.py:17-40) for B frames:
 * out = img * blur11x11,sigma5(disc(cx, cy, r)).  discs int32 [B,3] = (cx, cy, r) per frame -- the caller's
 * random.randint draws (:23-25).  The disc is the analytic set (x-cx)^2 + (y-cy)^2 <= r^2 (the reference
 * rasterises it with cv2.circle: parity with OpenCV's rasteriser is unpinned).  mask_scratch f32 [B,H,W];
 * out may alias img. */
FFB_API int ffb_silhouette(const float* img, const int32_t* discs, int32_t B, int32_t H, int32_t W, float* mask_scratch,
                   float* out, void* stream);

/* Perlin material texture: rand_perlin_2d_octaves + NoiseTextureLerpSampler.sample_train
 * (fireflies/sampling/noise_texture_lerp.py:8-98).  `angles`: per octave o (frequency f = 2^o) the
 * (f*res0+1) x (f*res1+1) uniforms in [0,1) the reference draws with torch.rand, concatenated; H, W must be
 * multiples of res * 2^(octaves-1).  noise_scratch f32 [H,W] receives the octave sum, minmax_scratch
 * (2 x int32) its extrema; out (nullable) f32 [3,H,W] = lerp(color_a, color_b, (noise-min)/(max-min)). */
FFB_API int ffb_perlin_texture(const float* angles, int32_t H, int32_t W, int32_t res0, int32_t res1, int32_t octaves,
                       double persistence, const float* color_a, const float* color_b, float* noise_scratch,
                       int32_t* minmax_scratch, float* out, void* stream);

/* The parameters of one Perlin texture. */
typedef struct ffb_perlin_params {
    int32_t res0, res1;     /* lattice resolution (drawn: res0 = res1 = 2^k)                    */
    int32_t octaves;        /* 1..8 (drawn: 1..4)                                               */
    int32_t _pad;
    double  persistence;    /* octave o has amplitude float32(persistence^o)                    */
    int64_t angle_offset;   /* injected: index in `angles` of the sample's first lattice angle  */
} ffb_perlin_params;

#define FFB_PERLIN_TILE 512 /* Philox mode: H and W multiples of this, the largest res * 2^(octaves-1) it draws (64 * 8) */

/* B Perlin textures in one call, each with its own parameters: ffb_perlin_texture per sample.  noise f32 [B,H,W],
 * minmax int32 [B,2] (ordered-int extrema per sample), out (nullable) f32 [B,3,H,W]; colours f32 [3], shared by the
 * samples.  Every buffer is DEVICE memory; the call enqueues three kernels on `stream` and never waits for the device.
 *   Injected mode (params_host != NULL): params_host HOST [B]; each sample's angles are the concatenated per-octave
 *     (f*res0+1) x (f*res1+1) lattices of ffb_perlin_texture, starting at angles[angle_offset] (angles f32 [n_angles]).
 *     The parameters are checked here, then copied into params_out (DEVICE [B], required), which the kernels read.
 *     The texture of each sample is bit-identical to ffb_perlin_texture fed the same parameters and angles.
 *   Philox mode (params_host == NULL, angles == NULL): H and W multiples of FFB_PERLIN_TILE, 0 <= row <= 65535.
 *     Sample g = sample0 + b of sampler `row` draws, with r = Philox4x32-10(key = seed,
 *     counter = (0, lo32(g), hi32(g), 0x9E700000 | row)):
 *       k           = 1 + (r[0] * 6 >> 32)           res0 = res1 = 2^k        (random.randint(1, 6))
 *       octaves     = 1 + (r[1] * 4 >> 32)                                    (random.randint(1, 4))
 *       persistence = 0.1 + 1.9 * u53, u53 = ((r[2] >> 5) * 2^26 + (r[3] >> 6)) / 2^53, in fp64 (random.uniform(0.1, 2.0))
 *     and the angle of its lattice node n (the index into the concatenation above, octave by octave, row-major) is
 *       u = (w[0] >> 8) / 2^24, w = Philox4x32-10(key = seed, counter = (n, lo32(g), hi32(g), 0x9E710000 | row)).
 *     A texture depends only on (seed, sample0 + b, row): never on B or on how samples are split over calls.
 *     params_out (nullable) DEVICE [B] receives the drawn parameters (angle_offset = 0). */
FFB_API int ffb_perlin_texture_batch(int32_t B, int32_t H, int32_t W, uint64_t seed, uint64_t sample0, int32_t row,
                       const ffb_perlin_params* params_host, const float* angles, int64_t n_angles,
                       ffb_perlin_params* params_out, const float* color_a, const float* color_b, float* noise,
                       int32_t* minmax, float* out, void* stream);

/* ------------------------------------------------------------------------------------------
 * 5. NURBS-curve camera paths and batched intersections  (fireflies/entity/curve.py, utils/intersections.py)
 * ------------------------------------------------------------------------------------------ */

#define FFB_NURBS_MAX_DEGREE 7

/* geomdl==5.3.1 NURBS.Curve.evaluate_single (the evaluator behind fireflies/entity/curve.py:52-53,74; the curve
 * object is built by fireflies/utils/io.py:77-108) for B parameters at once, in fp64 like geomdl's Python floats:
 * linear knot-span walk, the degree+1 non-vanishing basis functions (Piegl & Tiller A2.2), homogeneous sum,
 * perspective divide (A4.1).  ctrlw f64 [n_ctrl,4] = (x*w, y*w, z*w, w); knots f64 [n_ctrl+degree+1], normalised to
 * [0,1] by the caller (geomdl does so on assignment); t f64 [B] in [0,1]; out f64 [B,3].  geomdl is absent from the
 * reference tree: parity with it is unpinned (see oracle/ff_oracle.py). */
FFB_API int ffb_nurbs_curve_eval(const double* ctrlw, const double* knots, int32_t n_ctrl, int32_t degree, const double* t,
                                 int32_t B, double* out, void* stream);

/* Curve.randomize's matrix for B path parameters (fireflies/entity/curve.py:48-96):
 *   out_world[b] = T(C(t_b)) @ toMat4x4(rotation_matrix_from_vectors([0,1,0], d_b)) @ world,
 *   d_b = f32(C(t_b + dt)) - f32(C(t_b)) with x and z negated (dt = 0.001 in the reference).
 * world f32 [16]; out_world / out_rot (sample_rotation) / out_trans (sample_translation) f32 [B,16], each nullable. */
FFB_API int ffb_curve_pose(const double* ctrlw, const double* knots, int32_t n_ctrl, int32_t degree, const double* t, int32_t B,
                           double dt, const float* world, float* out_world, float* out_rot, float* out_trans, void* stream);

/* rayPlane (fireflies/utils/intersections.py:5-12): t_out[i] = ((po_i - o_i) . n_i) / (n_i . d_i), a denominator
 * below 1e-6 in magnitude replaced by denom/denom.  All inputs f32 [N,3]; t_out f32 [N]. */
FFB_API int ffb_ray_plane(const float* origin, const float* direction, const float* plane_origin, const float* plane_normal,
                          int32_t N, float* t_out, void* stream);

/* sphereSphere (fireflies/utils/intersections.py:26-33): hit[i] = |a_i - b_i|^2 <= (ra_i + rb_i)^2.
 * a, b f32 [N,D]; ra, rb f32 [N]; hit u8 [N]. */
FFB_API int ffb_sphere_sphere(const float* a, const float* ra, const float* b, const float* rb, int32_t N, int32_t D, uint8_t* hit,
                              void* stream);

#ifdef __cplusplus
}
#endif
#endif /* FFB200_H */
