/*
 * laenerf_b200.h -- C ABI of liblaenerf_b200.so (hand-written sm_100a CUDA, no torch types).
 *
 * One entry point per function the reference's pybind11 `_backend` modules export for the ray-marched NeRF
 * step (citations are paths under /root/reference):
 *     raymarching/src/bindings.cpp:5-21   (12 functions)
 *     gridencoder/src/bindings.cpp        (3 functions)
 *     ffmlp/src/bindings.cpp              (5 functions)
 *     shencoder/src/bindings.cpp          (2 functions; adjacent row f-1 of SURVEY.md section 8)
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless the name ends in _host; buffers are caller-allocated and the
 *     library never allocates device memory.  Scratch, where needed, is passed in; its size is queried with the
 *     matching *_scratch_bytes function.  Scratch given to lnrf_march_rays_train / lnrf_compact_alive must be
 *     zero-filled before its FIRST use only (the kernels leave their look-back words zeroed again), must not be
 *     shared between the two functions, nor by launches that can overlap.
 *   - `stream` is a cudaStream_t passed as void* (0 = legacy default stream, which is what the reference uses).
 *   - return value: 0 on success, a negative lnrf_status otherwise; lnrf_last_error() returns a thread-local
 *     message (the reference raises RuntimeError through TORCH_CHECK; the Python shim re-raises the same way).
 *   - float tensors are fp32 row-major contiguous exactly as the reference's at::Tensor arguments; `*_f16`
 *     pointers are IEEE binary16.
 *   - zero-initialisation contracts of the reference wrappers are stated per function ("ZERO-IN" = the caller
 *     must pass zero-filled memory as the reference wrapper does; "SELF-ZERO" = the kernel writes every element,
 *     so the caller may pass uninitialised memory and sees what the reference's torch.zeros + kernel produce).
 */
#ifndef LAENERF_B200_H_
#define LAENERF_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#define LNRF_API __attribute__((visibility("default")))
#else
#define LNRF_API
#endif

typedef void* lnrf_stream_t;

typedef enum {
    LNRF_OK = 0,
    LNRF_ERR_INVALID_ARGUMENT = -1,
    LNRF_ERR_CUDA = -2,
    LNRF_ERR_UNSUPPORTED = -3,
    LNRF_ERR_SCRATCH_TOO_SMALL = -4
} lnrf_status;

typedef enum { LNRF_F32 = 0, LNRF_F16 = 1 } lnrf_dtype;

/* Thread-local description of the last failure on this thread ("" if none). */
LNRF_API const char* lnrf_last_error(void);
/* Library/ABI version and the SM architecture the kernels were compiled for (100 => sm_100a). */
LNRF_API int lnrf_version(void);
LNRF_API int lnrf_compiled_arch(void);
/* Number of kernels this library has launched from this process (all threads); used by bench.py gpu_launches. */
LNRF_API uint64_t lnrf_launch_count(void);
/* sizeof(lnrf_render_desc) / sizeof(lnrf_opt_tensor) in this build, so that an FFI mirror of the two descriptor structs
 * (ctypes.Structure, cgo, ...) can be checked before the first call. */
LNRF_API size_t lnrf_sizeof_render_desc(void);
LNRF_API size_t lnrf_sizeof_opt_tensor(void);

/* ---------------------------------------------------------------------------------------------------------
 * raymarching utilities -- replaces raymarching/src/raymarching.cu:148-156, 201-209, 229-232, 257-260, 292-300
 * --------------------------------------------------------------------------------------------------------- */

/* near_far_from_aabb (raymarching.h:7).  rays_o/rays_d [N,3]; aabb [6]; nears/fars [N] (written for all N). */
LNRF_API int lnrf_near_far_from_aabb(const float* rays_o, const float* rays_d, const float* aabb, uint32_t N,
                                     float min_near, float* nears, float* fars, lnrf_stream_t stream);
/* sph_from_ray (raymarching.h:8).  coords [N,2]. */
LNRF_API int lnrf_sph_from_ray(const float* rays_o, const float* rays_d, float radius, uint32_t N, float* coords,
                               lnrf_stream_t stream);
/* morton3D / morton3D_invert (raymarching.h:9-10).  coords [N,3] int32 in [0,1024); indices [N] int32. */
LNRF_API int lnrf_morton3D(const int32_t* coords, uint32_t N, int32_t* indices, lnrf_stream_t stream);
LNRF_API int lnrf_morton3D_invert(const int32_t* indices, uint32_t N, int32_t* coords, lnrf_stream_t stream);
/* packbits (raymarching.h:11).  grid [N*8] fp32; bitfield [N] bytes; bit i of byte n = grid[8n+i] > thresh. */
LNRF_API int lnrf_packbits(const float* grid, uint32_t N, float density_thresh, uint8_t* bitfield,
                           lnrf_stream_t stream);

/* ---------------------------------------------------------------------------------------------------------
 * training march + compositing -- replaces raymarching.cu:482-490, 580-588, 685-693
 * --------------------------------------------------------------------------------------------------------- */

/* march_rays_train (raymarching.h:13).
 *   rays_o, rays_d [N,3]; grid = density bitfield [C*H^3/8]; nears, fars, noises [N];
 *   xyzs, dirs [M,3], deltas [M,2]  SELF-ZERO (rows not covered by a ray are written as zeros);
 *   rays [N,3] int32 = (ray id, point offset, point count) -- all N rows written;
 *   counter [2] int32: counter[0] += total points, counter[1] += N (the caller zeroes it, renderer.py:287-288).
 * Slot assignment is DETERMINISTIC: row n of `rays` is ray n and offsets are the exclusive prefix sum of the
 * per-ray counts in ray-id order, starting at the incoming counter[0] (the reference hands out slots with
 * atomicAdd in warp arrival order -- a run-dependent permutation of this layout, see DESIGN.md).  Rays with
 * offset + count > M write nothing (raymarching.cu:416).
 *   scratch: lnrf_march_rays_train_scratch_bytes(N) bytes, zero before first use. */
LNRF_API size_t lnrf_march_rays_train_scratch_bytes(uint32_t N);
LNRF_API int lnrf_march_rays_train(const float* rays_o, const float* rays_d, const uint8_t* grid, float bound,
                                   float dt_gamma, uint32_t max_steps, uint32_t N, uint32_t C, uint32_t H, uint32_t M,
                                   const float* nears, const float* fars, float* xyzs, float* dirs, float* deltas,
                                   int32_t* rays, int32_t* counter, const float* noises, void* scratch,
                                   size_t scratch_bytes, lnrf_stream_t stream);
/* The same with rays ending where they leave `occupied_box` (device float[6], see lnrf_render_desc.occupied_box; NULL = off):
 * identical samples, counts and offsets -- the walk through the empty rest of the scene box is skipped. */
LNRF_API int lnrf_march_rays_train_clipped(const float* rays_o, const float* rays_d, const uint8_t* density_bitfield, float bound,
                                           float dt_gamma, uint32_t max_steps, uint32_t N, uint32_t C, uint32_t H, uint32_t M,
                                           const float* nears, const float* fars, float* xyzs, float* dirs, float* deltas,
                                           int32_t* rays, int32_t* counter, const float* noises, const float* occupied_box,
                                           void* scratch, size_t scratch_bytes, lnrf_stream_t stream);

/* composite_rays_train_forward (raymarching.h:14).  sigmas [M], rgbs [M,3], deltas [M,2], rays [N,3];
 * weights_sum, depth [N], image [N,3] written at index rays[n,0] for every row n. */
LNRF_API int lnrf_composite_rays_train_forward(const float* sigmas, const float* rgbs, const float* deltas,
                                               const int32_t* rays, uint32_t M, uint32_t N, float T_thresh,
                                               float* weights_sum, float* depth, float* image, lnrf_stream_t stream);
/* composite_rays_train_backward (raymarching.h:15).  grad_sigmas [M], grad_rgbs [M,3]: ZERO-IN when
 * zero_fill == 0 (reference contract, raymarching.py:283-284).  With zero_fill != 0 the kernel itself clears
 * every element no ray covers; this requires the canonical `rays` layout lnrf_march_rays_train produces
 * (ray ranges ascending and contiguous); the fused training tail uses it, the drop-in `composite_rays_train` wrapper keeps
 * `torch.zeros` + zero_fill == 0 because callers may hand it `rays` in any order. */
LNRF_API int lnrf_composite_rays_train_backward(const float* grad_weights_sum, const float* grad_image,
                                                const float* sigmas, const float* rgbs, const float* deltas,
                                                const int32_t* rays, const float* weights_sum, const float* image,
                                                uint32_t M, uint32_t N, float T_thresh, float* grad_sigmas,
                                                float* grad_rgbs, int zero_fill, lnrf_stream_t stream);

/* Row f-5 of SURVEY.md section 8: the tail of the training step behind the network as one launch each way --
 * composite_rays_train (raymarching.h:14-15) + `image + (1 - weights_sum) * bg_color` (nerf/renderer.py:326) +
 * `clamp(depth - nears, min=0) / (fars - nears)` (:328) + the trainer's MSE `criterion(pred, gt).mean(-1).mean()`
 * (nerf/utils.py:592,633).  The reference runs ~12 elementwise / reduction launches here and as many backward.
 *   gt_rgb [N,3]; bg_rgb [N,3] per-pixel background or NULL -> bg_scalar; nears/fars [N] or both NULL (depth unscaled).
 *   outputs: weights_sum, depth [N], image [N,3] (blended), image_raw [N,3] (the composite, kept for the backward),
 *   loss [1] (deterministic: per-block partial sums added in index order by the last block).
 *   scratch: lnrf_composite_loss_scratch_bytes(N) bytes, zero before first use (the kernel re-arms it). */
LNRF_API size_t lnrf_composite_loss_scratch_bytes(uint32_t N);
LNRF_API int lnrf_composite_loss_train_forward(const float* sigmas, const float* rgbs, const float* deltas,
                                               const int32_t* rays, const float* gt_rgb, const float* bg_rgb,
                                               float bg_scalar, const float* nears, const float* fars, uint32_t M,
                                               uint32_t N, float T_thresh, float* weights_sum, float* depth,
                                               float* image, float* image_raw, float* loss, void* scratch,
                                               size_t scratch_bytes, lnrf_stream_t stream);
/* grad_loss [1] on the DEVICE (dL_total/dloss: the AMP loss scale, never read by the host).  dL/dimage and
 * dL/dweights_sum are formed inside the kernel; grad_sigmas [M] / grad_rgbs [M,3] are written completely (the
 * zero_fill contract of lnrf_composite_rays_train_backward: needs the canonical `rays` layout). */
LNRF_API int lnrf_composite_loss_train_backward(const float* grad_loss, const float* sigmas, const float* rgbs,
                                                const float* deltas, const int32_t* rays, const float* gt_rgb,
                                                const float* bg_rgb, float bg_scalar, const float* weights_sum,
                                                const float* image, const float* image_raw, uint32_t M, uint32_t N,
                                                float T_thresh, float* grad_sigmas, float* grad_rgbs,
                                                lnrf_stream_t stream);
/* Both of the above in ONE launch: dL_total/dloss is known before the forward runs (the AMP loss scale, a device
 * scalar), so the warp that composited a ray writes the ray's sample gradients right away, its samples still in L1.
 * Outputs of the forward AND of the backward, bit-identical to the two calls made one after the other. */
LNRF_API int lnrf_composite_loss_train_forward_backward(const float* grad_loss, const float* sigmas, const float* rgbs,
                                                        const float* deltas, const int32_t* rays, const float* gt_rgb,
                                                        const float* bg_rgb, float bg_scalar, const float* nears,
                                                        const float* fars, uint32_t M, uint32_t N, float T_thresh,
                                                        float* weights_sum, float* depth, float* image, float* image_raw,
                                                        float* loss, float* grad_sigmas, float* grad_rgbs, void* scratch,
                                                        size_t scratch_bytes, lnrf_stream_t stream);

/* ---------------------------------------------------------------------------------------------------------
 * inference / distillation march + compositing -- replaces raymarching.cu:929-945, 1145-1159
 * --------------------------------------------------------------------------------------------------------- */

/* march_rays (raymarching.h:17) and march_rays_distill (raymarching.h:18; edit_grid/edit_occ non-NULL).
 *   rays_alive [n_alive] int32 ray ids; rays_t, nears, fars [N]; noises [n_alive] (indexed by slot);
 *   xyzs, dirs [M_rows,3], deltas [M_rows,2], edit_occ [M_rows] bytes (bool): SELF-ZERO over all M_rows rows
 *   (M_rows >= n_alive*n_step is the padded row count the wrapper allocated, raymarching.py:329-336). */
LNRF_API int lnrf_march_rays(uint32_t n_alive, uint32_t n_step, const int32_t* rays_alive, const float* rays_t,
                             const float* rays_o, const float* rays_d, float bound, float dt_gamma, uint32_t max_steps,
                             uint32_t C, uint32_t H, const uint8_t* grid, const float* nears, const float* fars,
                             float* xyzs, float* dirs, float* deltas, const float* noises, uint32_t M_rows,
                             lnrf_stream_t stream);
LNRF_API int lnrf_march_rays_distill(uint32_t n_alive, uint32_t n_step, const int32_t* rays_alive, const float* rays_t,
                                     const float* rays_o, const float* rays_d, float bound, float dt_gamma,
                                     uint32_t max_steps, uint32_t C, uint32_t H, const uint8_t* grid,
                                     const uint8_t* edit_grid, const float* nears, const float* fars, float* xyzs,
                                     float* dirs, float* deltas, uint8_t* edit_occ, const float* noises,
                                     uint32_t M_rows, lnrf_stream_t stream);
/* composite_rays (raymarching.h:19) / composite_rays_distill (raymarching.h:20): in-place on rays_alive, rays_t,
 * weights_sum, depth, image (+ weights_edit_sum, depth_edit). */
LNRF_API int lnrf_composite_rays(uint32_t n_alive, uint32_t n_step, float T_thresh, int32_t* rays_alive, float* rays_t,
                                 const float* sigmas, const float* rgbs, const float* deltas, float* weights_sum,
                                 float* depth, float* image, lnrf_stream_t stream);
LNRF_API int lnrf_composite_rays_distill(uint32_t n_alive, uint32_t n_step, float T_thresh, int32_t* rays_alive,
                                         float* rays_t, const float* sigmas, const float* rgbs, const float* deltas,
                                         float* weights_sum, float* weights_edit_sum, float* depth, float* depth_edit,
                                         const uint8_t* edit_occ, float* image, lnrf_stream_t stream);
/* A ray subset on a PRESCRIBED n_step sequence, all rounds in one pass -- the fix-up pass of the "auto" render schedule
 * (laenerf_b200/nerf.py _fix_schedule_dependent_rays).  Round boundaries reach a ray's sample positions only through rays_t, which
 * composite_rays rebuilds as rays_t + sum of deltas[.][1] (raymarching.cu:1006): additions of numbers the marcher itself produced.
 * So the marcher can run a ray through ALL rounds of a given sequence on its own (each round starting from the t the compositor
 * would have rebuilt), the network runs once over the samples, and the compositor walks them in order and stops where
 * raymarching.cu:948-1035 would.  Bit-identical to lnrf_render_rounds with the same nstep_seq.
 *   march: offsets == NULL -> count only (counts[ray] = samples until the ray leaves the volume or the sequence ends);
 *          else write the ray's samples at row offsets[ray] (exclusive prefix sum of counts).  edit_grid != NULL: also edit_occ.
 *          caps (optional, [n_rays]): most samples to march per ray -- with offsets = prefix sum of the caps the counting pass and the
 *          walk behind a ray's death are spared; a ray that has not died within its cap must be redone without one.
 *          occupied_box (optional): as in lnrf_render_desc.
 *   composite: per-ray outputs indexed by the subset position; ray_steps[ray] = completed samples (where the ray dies). */
LNRF_API int lnrf_march_rays_prescribed(uint32_t n_rays, const float* rays_o, const float* rays_d, const float* nears,
                                        const float* fars, float bound, float dt_gamma, uint32_t max_steps, uint32_t C, uint32_t H,
                                        const uint8_t* density_bitfield, const uint8_t* edit_bitfield, const int32_t* nstep_seq,
                                        uint32_t nstep_len, const int32_t* offsets, int32_t* counts, float* xyzs, float* dirs,
                                        float* deltas, uint8_t* edit_occ, const int32_t* caps, const float* occupied_box,
                                        lnrf_stream_t stream);
LNRF_API int lnrf_composite_rays_prescribed(uint32_t n_rays, float T_thresh, const int32_t* offsets, const int32_t* counts,
                                            const float* nears, const float* sigmas, const float* rgbs, const float* deltas,
                                            const uint8_t* edit_occ, float* weights_sum, float* weights_edit_sum, float* depth,
                                            float* depth_edit, float* image, int32_t* ray_steps, lnrf_stream_t stream);

/* Device-side replacement for `rays_alive = rays_alive[rays_alive >= 0]` (renderer.py:375): stable compaction of
 * the non-negative entries of rays_alive[0..n_alive) into out (which must not alias rays_alive); the count is
 * written to n_out (device int32[1]).  scratch: lnrf_compact_alive_scratch_bytes(n_alive) bytes, zero before first
 * use (the kernel leaves it zeroed).  Row f-3 of SURVEY.md section 8. */
LNRF_API size_t lnrf_compact_alive_scratch_bytes(uint32_t n_alive);
LNRF_API int lnrf_compact_alive(const int32_t* rays_alive, uint32_t n_alive, int32_t* out, int32_t* n_out, void* scratch,
                                size_t scratch_bytes, lnrf_stream_t stream);

/* ---------------------------------------------------------------------------------------------------------
 * hash-grid encoder -- replaces gridencoder/src/gridencoder.cu:448-503, 639-645 (gridencoder.h:12-15)
 * --------------------------------------------------------------------------------------------------------- */

/* layout of the per-level feature axis in outputs / grad */
typedef enum {
    LNRF_GRID_LBC = 0, /* [L, B, C]: what the reference kernel writes (gridencoder.cu:388) */
    LNRF_GRID_BLC = 1  /* [B, L*C]: what grid.py:57 returns after its permute copy -- written directly */
} lnrf_grid_layout;

/* grid_encode_forward.  inputs [B,D] fp32 in [0,1]; embeddings [offsets[L], C] (dtype emb_dtype);
 * offsets_host [L+1] int32 on the HOST (the reference passes a device tensor; the shim keeps a host copy);
 * outputs in emb_dtype, layout out_layout; dy_dx optional ([B, L*D*C], emb_dtype) or NULL.
 * S = log2(per_level_scale), H = base_resolution, gridtype 0 hash / 1 tiled, interp 0 linear / 1 smoothstep.
 * Supported: D in {2,3}, C in {1,2,4,8}, L <= 32. */
LNRF_API int lnrf_grid_encode_forward(const float* inputs, const void* embeddings, const int32_t* offsets_host,
                                      void* outputs, uint32_t B, uint32_t D, uint32_t C, uint32_t L, float S,
                                      uint32_t H, void* dy_dx, uint32_t gridtype, int align_corners, uint32_t interp,
                                      lnrf_dtype emb_dtype, lnrf_grid_layout out_layout, lnrf_stream_t stream);
/* grid_encode_backward.  grad in emb_dtype with layout grad_layout; grad_embeddings [offsets[L], C] emb_dtype
 * ZERO-IN (grid.py:77); dy_dx/grad_inputs optional (grad_inputs [B,D] emb_dtype). */
LNRF_API int lnrf_grid_encode_backward(const void* grad, const float* inputs, const void* embeddings,
                                       const int32_t* offsets_host, void* grad_embeddings, uint32_t B, uint32_t D,
                                       uint32_t C, uint32_t L, float S, uint32_t H, const void* dy_dx,
                                       void* grad_inputs, uint32_t gridtype, int align_corners, uint32_t interp,
                                       lnrf_dtype emb_dtype, lnrf_grid_layout grad_layout, lnrf_stream_t stream);
/* grad_total_variation: accumulates into grad in place. inputs [B,D] in emb_dtype as in the reference. */
LNRF_API int lnrf_grad_total_variation(const void* inputs, const void* embeddings, void* grad,
                                       const int32_t* offsets_host, float weight, uint32_t B, uint32_t D, uint32_t C,
                                       uint32_t L, float S, uint32_t H, uint32_t gridtype, int align_corners,
                                       lnrf_dtype emb_dtype, lnrf_stream_t stream);
/* Test hook: the per-level `scale` (exp2f(level*S)*H - 1) exactly as the device evaluates it; scales [L] fp32. */
LNRF_API int lnrf_grid_level_scales(uint32_t L, float S, uint32_t H, float* scales, lnrf_stream_t stream);

/* ---------------------------------------------------------------------------------------------------------
 * fully fused MLP (tcgen05 / TMEM) -- replaces ffmlp/src/ffmlp.cu:635-709, 721-740, 749-895 (ffmlp.h)
 * --------------------------------------------------------------------------------------------------------- */

/* Weights are the reference's flat fp16 vector: [hidden,in] + (num_layers-1) x [hidden,hidden] + [out,hidden],
 * each row-major (ffmlp.cu:632).  B must be a multiple of 128 (the shim pads, ffmlp.py:157-159); hidden_dim 64
 * (the width every LAENeRF net uses) ; input_dim a multiple of 16 up to 64; output_dim == 16 (padded).
 * activation ids as ffmlp.py:89-96 (0 relu, 3 sigmoid ... 6 none).
 * ffmlp_forward: inputs [B,in], forward_buffer [num_layers,B,hidden] (saved activations), outputs [B,out]. */
LNRF_API int lnrf_ffmlp_forward(const void* inputs_f16, const void* weights_f16, uint32_t B, uint32_t input_dim,
                                uint32_t output_dim, uint32_t hidden_dim, uint32_t num_layers, uint32_t activation,
                                uint32_t output_activation, void* forward_buffer_f16, void* outputs_f16,
                                lnrf_stream_t stream);
/* ffmlp_inference: no activations saved (inference_buffer is accepted for signature parity and unused). */
LNRF_API int lnrf_ffmlp_inference(const void* inputs_f16, const void* weights_f16, uint32_t B, uint32_t input_dim,
                                  uint32_t output_dim, uint32_t hidden_dim, uint32_t num_layers, uint32_t activation,
                                  uint32_t output_activation, void* inference_buffer_f16, void* outputs_f16,
                                  lnrf_stream_t stream);
/* ffmlp_backward: grad [B,out]; backward_buffer [num_layers,B,hidden] scratch (accepted for parity; the fused
 * kernel keeps dL/dhidden on chip and only uses it when non-NULL for debugging); grad_inputs [B,in] or NULL
 * (calc_grad_inputs); grad_weights flat fp16 like weights (written, not accumulated);
 * wgrad_scratch: lnrf_ffmlp_wgrad_scratch_bytes(...) bytes of fp32 partial sums (any contents). */
LNRF_API size_t lnrf_ffmlp_wgrad_scratch_bytes(uint32_t input_dim, uint32_t output_dim, uint32_t hidden_dim,
                                               uint32_t num_layers);
LNRF_API int lnrf_ffmlp_backward(const void* grad_f16, const void* inputs_f16, const void* weights_f16,
                                 const void* forward_buffer_f16, uint32_t B, uint32_t input_dim, uint32_t output_dim,
                                 uint32_t hidden_dim, uint32_t num_layers, uint32_t activation,
                                 uint32_t output_activation, int calc_grad_inputs, void* backward_buffer_f16,
                                 void* grad_inputs_f16, void* grad_weights_f16, void* wgrad_scratch,
                                 size_t wgrad_scratch_bytes, lnrf_stream_t stream);
/* allocate_splitk / free_splitk (ffmlp.cu:721-740): the reference creates side streams for its split-K wgrad
 * GEMMs.  The fused backward needs none; both are kept as no-ops so that the binding surface is identical. */
LNRF_API int lnrf_allocate_splitk(size_t size);
LNRF_API int lnrf_free_splitk(void);

/* ---------------------------------------------------------------------------------------------------------
 * spherical-harmonics direction encoder (adjacent row f-1) -- shencoder/src/shencoder.cu:385-439
 * --------------------------------------------------------------------------------------------------------- */
/* inputs [B,3] fp32; outputs [B, degree^2] in out_dtype; degree in 1..8; dy_dx optional [B, 3*degree^2]. */
LNRF_API int lnrf_sh_encode_forward(const float* inputs, void* outputs, uint32_t B, uint32_t degree, void* dy_dx,
                                    lnrf_dtype out_dtype, lnrf_stream_t stream);
/* sh_encode_backward (shencoder.cu:394-397): grad [B, degree^2], dy_dx [B, 3*degree^2], grad_inputs [B,3] fp32,
 * accumulated in place (ZERO-IN, sphere_harmonics.py:49). */
LNRF_API int lnrf_sh_encode_backward(const float* grad, uint32_t B, uint32_t degree, const float* dy_dx,
                                     float* grad_inputs, lnrf_stream_t stream);

/* world-coordinate variants of the hot hash-grid kernels (D = 3, C = 2, [B, L*C] layout): GridEncoder.forward's
 * (x + bound) / (2 * bound) (gridencoder/grid.py:147) is applied inside the kernel with the same two IEEE operations.
 * B_dev (forward, device int32 or NULL): when given, B is only the capacity and the kernel reads the row count there. */
LNRF_API int lnrf_grid_encode_forward_world(const float* inputs_world, float bound, const void* embeddings,
                                            const int32_t* offsets_host, void* outputs, uint32_t B, const int32_t* B_dev,
                                            uint32_t L, float S, uint32_t H, uint32_t gridtype, int align_corners,
                                            uint32_t interp, lnrf_dtype emb_dtype, lnrf_stream_t stream);
LNRF_API int lnrf_grid_encode_backward_world(const void* grad, const float* inputs_world, float bound,
                                             const int32_t* offsets_host, void* grad_embeddings, uint32_t B,
                                             const int32_t* B_dev, uint32_t L, float S, uint32_t H, uint32_t gridtype,
                                             int align_corners, uint32_t interp, lnrf_dtype emb_dtype, lnrf_stream_t stream);

/* ---------------------------------------------------------------------------------------------------------
 * device-driven inference rounds (row f-3) -- the loop of NeRFRenderer.run_cuda / run_cuda_distill
 * (nerf/renderer.py:335-387, 425-470) without a device->host synchronisation per round.
 * --------------------------------------------------------------------------------------------------------- */
typedef struct {
    int32_t* ctl;                 /* device int32[32] control block: [0] n_alive [1] n_step [2] steps marched [3] rows of the
                                     round (n_alive*n_step padded past 128) [4] n_rays [5] max_steps [6] finished [7] rounds
                                     [9] sample slots marched so far [12] the result may depend on the round schedule (see
                                     ray_flags) [13] rays that raised [12] [14] the max_steps cap cut rays off [15] rows of the running compact round; [16..22] internal
                                     (copies of the four fields below) */
    uint32_t n_rays, max_steps;
    /* rays and marching (raymarching.march_rays arguments) */
    const float *rays_o, *rays_d, *nears, *fars;       /* [n_rays,3] x2, [n_rays] x2 */
    const uint8_t* density_bitfield;
    const uint8_t* edit_bitfield;                      /* NULL: plain render; else run_cuda_distill */
    float bound, dt_gamma, T_thresh;
    uint32_t cascade, grid_size;
    const float* first_round_noises;                   /* [n_rays] or NULL (perturb only applies to the first round) */
    /* network (NeRFNetwork.forward, see lnrf_nerf_forward) */
    const void* embeddings_f16;
    const int32_t* offsets_host;
    uint32_t num_levels, base_resolution, gridtype, interpolation;
    int align_corners;
    float level_scale_log2;                            /* S of lnrf_grid_encode_forward */
    const void *w_sigma_f16, *w_color_f16;
    uint32_t num_layers_sigma, num_layers_color;
    float density_scale;
    /* state: two rays_alive buffers [n_rays] (round r reads [r & 1]), rays_t [n_rays] */
    int32_t* rays_alive[2];
    float* rays_t;
    /* per-round sample buffers, n_rays + 128 rows each (or sample_rows, see below) */
    float *xyzs, *dirs, *deltas;                       /* [rows,3], [rows,3], [rows,2] */
    uint8_t* edit_occ;                                 /* [rows] (distillation) or NULL */
    void* enc_f16;                                     /* [rows,32] */
    float *sigmas, *rgbs;                              /* [rows], [rows,3] */
    /* per-ray accumulators [n_rays] (image [n_rays,3]); cleared by lnrf_render_begin */
    float *weights_sum, *depth, *image, *weights_edit_sum, *depth_edit;
    void* scratch;                                     /* lnrf_render_scratch_bytes(n_rays), zero-filled before first use */
    size_t scratch_bytes;
    /* Round schedule.  sample_rows = 0: the reference's, n_step = clamp(n_rays / n_alive, 1, 8) (renderer.py:357), sample buffers
     * of n_rays + 128 rows.  sample_rows > n_rays + 128: the buffers hold that many rows and every round after the first
     * uses n_step = clamp((sample_rows - 128) / n_alive, 1, samples_per_round): the first round (n_step = 1) weeds out the rays that miss,
     * the survivors then take up to samples_per_round samples per round -- several times fewer rounds per frame.  Same per-sample arithmetic; sample
     * positions can differ in the last ulp where a round boundary moves (composite_rays re-sums t from deltas). */
    uint32_t sample_rows;
    uint32_t samples_per_round;   /* cap on n_step after the first round when sample_rows is in force (0: 8; at most 64) */
    /* Making a non-reference schedule exact (all optional, NULL / 0 = off).  ray_steps [n_rays] int32: += the samples a ray completed
     * in each round (cleared by lnrf_render_begin): its total is the sample index at which the ray dies, whatever the schedule.
     * ray_flags [n_rays] uint8: set to 1 for a ray that emitted a delta that is not exactly representable after round 0 -- the
     * only rays whose result depends on where the round boundaries fall (cleared by lnrf_render_begin).  nstep_seq [nstep_len]
     * int32 (device): a prescribed n_step per round instead of either rule above -- with the reference's sequence (which follows
     * from the histogram of ray_steps) a subset of rays is rendered exactly as the reference's full-frame loop renders it. */
    int32_t* ray_steps;
    uint8_t* ray_flags;
    const int32_t* nstep_seq;
    uint32_t nstep_len;
    /* Optional (NULL = off): device float[6] = {lo_x, lo_y, lo_z, hi_x, hi_y, hi_z}, a box that CONTAINS every occupied cell of
     * density_bitfield on every cascade (with a margin of two cells; laenerf_b200/nerf.py occupied_box).  The marcher then ends a
     * ray at min(far, exit of this box): beyond it no cell is occupied, so no sample is ever emitted there -- the walk to the end of
     * the scene box that raymarching.cu:766 does for every ray (and the whole walk of a ray that misses the box) is skipped with
     * the same samples, deltas and rays_t.  The START of a ray is never moved: the t lattice hangs on `near`. */
    const float* occupied_box;
} lnrf_render_desc;
LNRF_API size_t lnrf_render_scratch_bytes(uint32_t n_rays);
/* rays_alive[0] = 0..n_rays-1, rays_t = nears, accumulators = 0, control block = first round. */
LNRF_API int lnrf_render_begin(const lnrf_render_desc* desc_host, lnrf_stream_t stream);
/* Queues rounds first_round .. first_round + n_rounds - 1 (march -> encode -> network -> composite -> compact each).
 * Rounds after the frame has finished are no-ops; read ctl[6] (finished) between calls. */
LNRF_API int lnrf_render_rounds(const lnrf_render_desc* desc_host, uint32_t first_round, uint32_t n_rounds,
                                lnrf_stream_t stream);

/* ---------------------------------------------------------------------------------------------------------
 * fused NeRFNetwork.forward / backward (row f-1 of SURVEY.md section 8) -- nerf/network_ff.py:51-79:
 *     h = sigma_net(enc); sigma = trunc_exp(h[:,0]) (activation.py:5-17); d = SHEncoder(dirs) (degree 4,
 *     shencoder/src/shencoder.cu:27-123); rgb = sigmoid(color_net(cat[d, h[:,1:], 0]))
 * with both FFMLPs (hidden 64; sigma 32 -> 64 x num_layers_sigma -> 16; colour 32 -> 64 x num_layers_color -> 16,
 * weights in the reference's flat layout, ffmlp.cu:632) and all of the elementwise glue in one kernel.
 * --------------------------------------------------------------------------------------------------------- */
/* enc [M,32] fp16 (GridEncoder output), dirs [M,3] fp32, M a multiple of 128.
 * outputs: sigmas [M] fp32 = density_scale * exp(h0) (renderer.py:299), rgbs [M,3] fp32 (fp16-rounded values, as
 * torch.sigmoid on the half output gives).  train != 0 additionally saves forward_buffer [ns+nc, M, 64] fp16
 * (hidden activations: sigma net's first), color_in [M,32] fp16 (the colour net's input rows) and h0 [M] fp16. */
LNRF_API int lnrf_nerf_forward(const void* enc_f16, const float* dirs, const void* w_sigma_f16, const void* w_color_f16,
                               uint32_t M, uint32_t num_layers_sigma, uint32_t num_layers_color, float density_scale,
                               int train, void* forward_buffer_f16, void* color_in_f16, void* h0_f16, float* sigmas,
                               float* rgbs, lnrf_stream_t stream);
/* grad_sigmas [M] / grad_rgbs [M,3] fp32 (what composite_rays_train's backward writes) -> grad_enc [M,32] fp16,
 * grad_w_sigma / grad_w_color flat fp16 (written, or added to when accumulate_wgrad != 0).  dh_scratch [M,16] fp16 and wgrad_scratch
 * (lnrf_nerf_wgrad_scratch_bytes) may hold anything.  Gradients are rounded to fp16 where autograd would
 * hold fp16 tensors in the reference (grad of the .float() casts, dL/dh, dL/denc). */
LNRF_API size_t lnrf_nerf_wgrad_scratch_bytes(uint32_t num_layers_sigma, uint32_t num_layers_color);
LNRF_API int lnrf_nerf_backward(const float* grad_sigmas, const float* grad_rgbs, const float* rgbs, const void* h0_f16,
                                const void* enc_f16, const void* color_in_f16, const void* w_sigma_f16,
                                const void* w_color_f16, const void* forward_buffer_f16, uint32_t M,
                                uint32_t num_layers_sigma, uint32_t num_layers_color, float density_scale,
                                void* grad_enc_f16, void* grad_w_sigma_f16, void* grad_w_color_f16, int accumulate_wgrad,
                                void* dh_scratch_f16, void* wgrad_scratch, size_t wgrad_scratch_bytes,
                                lnrf_stream_t stream);

/* Round 2: the same pair WITHOUT saved hidden activations.  The forward keeps only h = sigma_net(enc) [M,16] fp16 (32 B/sample
 * instead of 704); the backward RECOMPUTES every hidden activation from enc and h on the tensor cores inside one warp-specialised
 * kernel (csrc/nerfbwd.cu: TMA producer warp, MMA warp, two epilogue warpgroups) -- DRAM traffic of the two calls drops from
 * ~366 MB to ~60 MB per 228 k-sample step.  Same values as lnrf_nerf_forward / lnrf_nerf_backward (identical MMAs and rounding points).
 * M_dev (optional, may be NULL): device-side count of live samples (the training marcher's counter[0], the render control block);
 * rows at or beyond ceil(*M_dev / 128) * 128 are padding and are skipped.  h_f16 may be NULL (inference).
 * lnrf_nerf_backward_recompute_supported: 2 <= num_layers_sigma <= num_layers_color and the shared-memory / TMEM budget (LAENeRF's
 * 2 / 3 layers fit); otherwise use lnrf_nerf_forward(train) + lnrf_nerf_backward. */
LNRF_API int lnrf_nerf_forward_lean(const void* enc_f16, const float* dirs, const void* w_sigma_f16, const void* w_color_f16, uint32_t M,
                                    const int32_t* M_dev, uint32_t num_layers_sigma, uint32_t num_layers_color, float density_scale,
                                    void* h_f16, float* sigmas, float* rgbs, lnrf_stream_t stream);
LNRF_API int lnrf_nerf_backward_recompute_supported(uint32_t num_layers_sigma, uint32_t num_layers_color);
LNRF_API int lnrf_nerf_backward_recompute(const float* grad_sigmas, const float* grad_rgbs, const float* rgbs, const void* h_f16,
                                          const void* enc_f16, const float* dirs, const void* w_sigma_f16, const void* w_color_f16,
                                          uint32_t M, const int32_t* M_dev, uint32_t num_layers_sigma, uint32_t num_layers_color,
                                          float density_scale, void* grad_enc_f16, void* grad_w_sigma_f16, void* grad_w_color_f16,
                                          int accumulate_wgrad, void* wgrad_scratch, size_t wgrad_scratch_bytes, lnrf_stream_t stream);
/* accumulate_wgrad of lnrf_nerf_backward_recompute: bit 0 = add to the existing fp16 weight gradients, bit 1 = leave the per-CTA partial
 * sums in wgrad_scratch and let the caller run their fixed-order reduction with this call -- e.g. on another stream beside the
 * hash-grid backward, which does not depend on it (laenerf_b200/nerf.py).  Same M / layer counts / scratch as the backward call. */
LNRF_API int lnrf_nerf_wgrad_reduce(const void* wgrad_scratch, size_t wgrad_scratch_bytes, uint32_t M, uint32_t num_layers_sigma,
                                    uint32_t num_layers_color, void* grad_w_sigma_f16, void* grad_w_color_f16, int accumulate,
                                    lnrf_stream_t stream);

/* ---------------------------------------------------------------------------------------------------------
 * occupancy-grid maintenance (row f-2) -- NeRFRenderer.update_extra_state, nerf/renderer.py:556-649
 * --------------------------------------------------------------------------------------------------------- */
/* Jittered query points of one cascade: xyz = (2 c / (H-1) - 1) * (bound_c - hgs) + (u * 2 - 1) * hgs, hgs = bound_c / H
 * (renderer.py:585-597, torch's rounding sequence), indices = morton3D(c).  coords [N,3] int32 cell coordinates, or
 * NULL for the full grid in meshgrid('ij') order (N == H^3); uniforms [N,3] fp32 in [0,1) (torch.rand). */
LNRF_API int lnrf_occupancy_points(const int32_t* coords, const float* uniforms, uint32_t N, uint32_t H,
                                   float cascade_bound, float* xyzs, int32_t* indices, lnrf_stream_t stream);
/* tmp_grid_cascade[indices[i]] = sigmas[i] (renderer.py:601, 641). */
LNRF_API int lnrf_occupancy_scatter(const float* sigmas, const int32_t* indices, uint32_t N, float* tmp_grid_cascade,
                                    lnrf_stream_t stream);
LNRF_API int lnrf_occupancy_fill(float* grid, uint32_t n, float value, lnrf_stream_t stream);
/* density_grid = max(density_grid * decay, tmp_grid) where both >= 0 (renderer.py:625-626); tmp_grid is reset to -1;
 * mean_out[0] = mean(clamp(density_grid, 0)) (:627), mean_out[1] = min(mean, density_thresh) (:632), both on the device. */
LNRF_API size_t lnrf_occupancy_scratch_bytes(void);
LNRF_API int lnrf_occupancy_ema(float* density_grid, float* tmp_grid, uint32_t n, float decay, float density_thresh,
                                float* mean_out, void* scratch, size_t scratch_bytes, lnrf_stream_t stream);
/* packbits (raymarching.cu:267-300) with the threshold read from device memory; N = number of output bytes. */
LNRF_API int lnrf_packbits_dev(const float* grid, uint32_t N, const float* thresh_dev, uint8_t* bitfield,
                               lnrf_stream_t stream);
/* Box around the occupied cells of a bitfield (every cascade, two cells of margin, world coordinates): box = device float[6] {lo xyz,
 * hi xyz}, +-inf when nothing is occupied.  What lnrf_render_desc.occupied_box / lnrf_march_rays_train_clipped take.  work: device
 * int32[lnrf_occupied_box_work_ints(C)], initialised ONCE to {H, H, H, -1, -1, -1} per cascade followed by 0 (the kernel re-arms it).
 * One launch, no host synchronisation. */
LNRF_API size_t lnrf_occupied_box_work_ints(uint32_t C);
LNRF_API int lnrf_occupied_box(const uint8_t* density_bitfield, uint32_t C, uint32_t H, float bound, int32_t* work, float* box,
                               lnrf_stream_t stream);
/* sigma net only (NeRFNetwork.density, network_ff.py:81-95): sigmas [M] = density_scale * exp(h0); M a multiple of 128. */
LNRF_API int lnrf_nerf_density(const void* enc_f16, const void* w_sigma_f16, uint32_t M, uint32_t num_layers_sigma,
                               float density_scale, float* sigmas, lnrf_stream_t stream);

/* ---------------------------------------------------------------------------------------------------------
 * Adam + AMP glue in one pass (row f-4) -- replaces, per training step of `-O` (nerf/utils.py:1474-1484,
 * main_nerf.py:223: Adam betas (0.9, 0.99) eps 1e-15 under GradScaler): embeddings.half() (grid.py:43-44),
 * the gradient clear, the fp16 -> fp32 gradient cast, GradScaler's inf check / unscale and torch.optim.Adam.
 * --------------------------------------------------------------------------------------------------------- */
typedef struct {
    float* params;      /* [n] fp32 master parameters, updated in place */
    float* exp_avg;     /* [n] fp32 */
    float* exp_avg_sq;  /* [n] fp32 */
    void* grad;         /* [n] gradient, possibly loss-scaled; CLEARED to zero by lnrf_adam_step */
    void* params_f16;   /* [n] fp16 shadow copy rewritten from the updated parameters, or NULL */
    uint64_t n;
    lnrf_dtype grad_dtype;
} lnrf_opt_tensor;
/* tensors_host: HOST array of 1..8 descriptors (device pointers inside).  found_inf: device fp32 scalar, set to
 * 1.0f when any gradient element is inf/nan (never cleared: GradScaler's convention). */
LNRF_API int lnrf_grad_nonfinite_check(const lnrf_opt_tensor* tensors_host, uint32_t count, float* found_inf,
                                       lnrf_stream_t stream);
/* One Adam step on every tensor (torch.optim.Adam, amsgrad off).  grad_scale (device fp32 scalar or NULL): the
 * gradients are divided by it first; found_inf (device scalar or NULL): when non-zero the parameters and moments
 * are left untouched (the gradients are still cleared); step_count: device fp32 scalar = 1-based step number;
 * lr_scale (device fp32 scalar or NULL): multiplies lr (a LambdaLR schedule factor that a CUDA graph can replay). */
LNRF_API int lnrf_adam_step(const lnrf_opt_tensor* tensors_host, uint32_t count, double lr, double beta1, double beta2,
                            double eps, double weight_decay, const float* grad_scale, const float* found_inf,
                            const float* step_count, const float* lr_scale, lnrf_stream_t stream);
/* Ray-sharded training (SURVEY.md section 8e): gradient exchange + Adam + parameter broadcast in ONE kernel over NVLink
 * peer memory.  grad_peers / shadow_peers / flag_peers: HOST arrays of `world` pointers, entry r = rank r's full fp16
 * gradient vector, full fp16 shadow vector and non-finite flag (all peer-mapped into this process, e.g. torch symmetric
 * memory).  This rank owns elements [lo, lo + n): it averages the `world` gradients of that slice, applies Adam to its fp32
 * master / moment slices and stores the new fp16 values into every rank's shadow.  When any flag is non-zero nothing is
 * updated and *found_inf_out = 1.  The caller synchronises the ranks before (gradients and flags complete) and after
 * (shadows visible; gradients may be cleared) the call. */
LNRF_API int lnrf_adam_step_sharded(const void* const* grad_peers_host, void* const* shadow_peers_host,
                                    const float* const* flag_peers_host, uint32_t world, uint64_t lo, uint64_t n,
                                    float* master_shard, float* exp_avg_shard, float* exp_avg_sq_shard, double lr,
                                    double beta1, double beta2, double eps, double weight_decay, const float* grad_scale,
                                    float* found_inf_out, const float* step_count, const float* lr_scale,
                                    lnrf_stream_t stream);
/* fp32 form of lnrf_adam_step_sharded for a network trained without fp16 shadows (the edit-stage style network): grad_peers /
 * param_peers / flag_peers = HOST arrays of `world` pointers to each rank's full fp32 gradient vector, full fp32 parameter vector
 * and non-finite flag.  This rank (`rank`) owns elements [lo, lo + n): it averages the `world` gradients of that slice in the fixed
 * rank order 0 .. world-1 (every rank forms the same bits), unscales by *grad_scale, applies Adam with its fp32 moment slices and
 * stores the new value into every rank's parameter vector -- the parameter vector is the master, no separate copy exists.
 * Learning rate per part of the vector: n_segs (1..8) segments, segment s covers [seg_start[s], seg_start[s+1]) at
 * lr x seg_lr_mult[s]; seg_start (HOST, elements of the full vector) begins at 0, ascends strictly and holds multiples of 8.
 * Skip-on-inf and the caller's synchronisation as for lnrf_adam_step_sharded. */
LNRF_API int lnrf_adam_step_sharded_f32(const float* const* grad_peers_host, float* const* param_peers_host,
                                        const float* const* flag_peers_host, uint32_t world, uint32_t rank, uint64_t lo,
                                        uint64_t n, const uint64_t* seg_start_host, const double* seg_lr_mult_host,
                                        uint32_t n_segs, float* exp_avg_shard, float* exp_avg_sq_shard, double lr,
                                        double beta1, double beta2, double eps, double weight_decay, const float* grad_scale,
                                        float* found_inf_out, const float* step_count, const float* lr_scale,
                                        lnrf_stream_t stream);
/* The same for a loop that alternates TWO gradient buffers (and two flag words) between consecutive steps: while the ranks read this
 * step's buffer, the kernel clears the buffer the previous step used (other_grad_f16, other_n elements; its readers passed this step's
 * opening barrier long ago), zeroes that step's flag word (other_flag), and performs GradScaler.update() on the live words at its end.
 * The closing "clear + update" launch and the flag memset ahead of the inf check disappear; the barrier after the kernel stays (the
 * peers' stores into this rank's table).  Scale and step number of THIS step are read from `snapshot` ([1], [2]), which
 * lnrf_grad_nonfinite_check_snapshot fills ahead of the opening barrier. */
LNRF_API int lnrf_adam_step_sharded_pipelined(const void* const* grad_peers_host, void* const* shadow_peers_host,
                                              const float* const* flag_peers_host, uint32_t world, uint64_t lo, uint64_t n,
                                              float* master_shard, float* exp_avg_shard, float* exp_avg_sq_shard, double lr,
                                              double beta1, double beta2, double eps, double weight_decay, const float* snapshot,
                                              const float* lr_scale, void* other_grad_f16, uint64_t other_n, float* other_flag,
                                              float* grad_scale, int32_t* growth_tracker, float* found_inf, float* step_count,
                                              float growth_factor, float backoff_factor, int32_t growth_interval,
                                              lnrf_stream_t stream);
/* lnrf_grad_nonfinite_check into flag_out, plus snapshot[1] = *grad_scale (1 when NULL), snapshot[2] = *step_count. */
LNRF_API int lnrf_grad_nonfinite_check_snapshot(const lnrf_opt_tensor* tensors_host, uint32_t count, float* flag_out,
                                                const float* grad_scale, const float* step_count, float* snapshot,
                                                lnrf_stream_t stream);
/* The same with the rank synchronisation inside the kernels instead of two barrier launches around it.  flag_peers: each
 * rank's peer-mapped buffer of >= 32 fp32 words -- word 0 is the non-finite flag, words 8..15 / 16..23 are written by ranks
 * 0..7 ("my gradient is complete" / "my stores into your table are complete", as epoch numbers); all zero before the first
 * step.  sync_state: two LOCAL device uint32 words (completed epoch, block ticket), zero before the first step.  The kernel
 * waits for every rank's gradient before reading it and announces the end of its stores; lnrf_exchange_finish -- the next
 * launch on the stream -- waits for every rank's announcement, then clears this rank's gradient (n elements).  Waits trap
 * after ~4 s instead of hanging. */
LNRF_API int lnrf_adam_step_sharded_sync(const void* const* grad_peers_host, void* const* shadow_peers_host,
                                         const float* const* flag_peers_host, uint32_t world, uint32_t rank, uint64_t lo,
                                         uint64_t n, float* master_shard, float* exp_avg_shard, float* exp_avg_sq_shard,
                                         double lr, double beta1, double beta2, double eps, double weight_decay,
                                         const float* grad_scale, float* found_inf_out, const float* step_count,
                                         const float* lr_scale, uint32_t* sync_state, lnrf_stream_t stream);
LNRF_API int lnrf_exchange_finish(const float* my_flags, uint32_t world, const uint32_t* sync_state, void* grad_f16,
                                  uint64_t n, lnrf_stream_t stream);
/* GradScaler.update() (growth / backoff of the loss scale from found_inf) fused with the step bookkeeping:
 * step_count += 1 unless the step was skipped, found_inf re-armed to 0.  scale / growth_tracker may be NULL
 * (no loss scaling). */
/* Round 2: the three calls above (non-finite check, Adam, GradScaler.update) as ONE launch.  Every block checks the gradient chunks
 * it is about to update, the blocks meet at a grid-wide barrier (the grid is capped at what is resident at once), read the combined
 * flag and run the update; the block that finishes last applies the scale growth / backoff, advances step_count when the step was
 * not skipped and re-arms found_inf.  grad_scale may be NULL (no GradScaler: nothing is unscaled, the check still guards the step).
 * sync_words: 3 zero-initialised device uint32 owned by the caller (left zero / advanced consistently by every call). */
LNRF_API int lnrf_adam_amp_step(const lnrf_opt_tensor* tensors_host, uint32_t count, double lr, double beta1, double beta2,
                                double eps, double weight_decay, float* grad_scale, int32_t* growth_tracker, float* found_inf,
                                float* step_count, const float* lr_scale, float growth_factor, float backoff_factor,
                                int32_t growth_interval, uint32_t* sync_words, lnrf_stream_t stream);
/* Closing launch of the barrier-bracketed sharded step: clears the local fp16 gradient (n elements, a multiple of 8) and applies
 * GradScaler.update() (as lnrf_amp_update) in the same launch. */
LNRF_API int lnrf_exchange_tail(void* grad_f16, uint64_t n, float* scale, int32_t* growth_tracker, float* found_inf,
                                float* step_count, float growth_factor, float backoff_factor, int32_t growth_interval,
                                lnrf_stream_t stream);
LNRF_API int lnrf_amp_update(float* scale, int32_t* growth_tracker, float* found_inf, float* step_count,
                             float growth_factor, float backoff_factor, int32_t growth_interval, lnrf_stream_t stream);
/* lnrf_grad_nonfinite_check and lnrf_amp_update in ONE launch that runs AHEAD of lnrf_adam_step: the last block out freezes what
 * this step's optimizer kernel must see into snapshot[0..2] = {found_inf, the scale the gradients carry, step_count before the
 * increment} and then performs GradScaler.update().  Pass &snapshot[1], &snapshot[0], &snapshot[2] to lnrf_adam_step as
 * grad_scale, found_inf, step_count.  snapshot: 8 floats on the device, zero before first use ([4] is a ticket the kernel re-arms). */
LNRF_API int lnrf_grad_nonfinite_check_amp_update(const lnrf_opt_tensor* tensors_host, uint32_t count, float* grad_scale,
                                                  int32_t* growth_tracker, float* found_inf, float* step_count,
                                                  float growth_factor, float backoff_factor, int32_t growth_interval,
                                                  float* snapshot, lnrf_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* LAENERF_B200_H_ */
