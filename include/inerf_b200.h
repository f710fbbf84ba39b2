/*
 * inerf_b200.h -- C-ABI of libinerf_b200.so, the B200 (sm_100a) implementation
 * of Instance-NeRF's instance-field render / train hot path.
 *
 * Drop-in boundary: every entry point replaces one function of the reference's
 * pybind FFI (L0 in SURVEY.md section 8b).  Paths below are relative to
 * /root/reference/instance_nerf/.
 *
 * Conventions
 *   - plain C pointers to DEVICE memory, explicit sizes, no torch types;
 *   - the caller allocates every output (the reference's Python wrappers do the
 *     same: raymarching/raymarching.py:205-208, 260-262, 323-326);
 *   - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream,
 *     which is what the reference launches on: raymarching.cu:154,488,586);
 *   - every function returns 0 on success, a NEGATIVE inerf_status on a bad
 *     argument and a POSITIVE cudaError_t if the launch failed.  Nothing throws.
 *     (The reference's raymarching functions check nothing; gridencoder /
 *     shencoder TORCH_CHECK and throw: gridencoder.cu:446-462.)
 */
#ifndef INERF_B200_H
#define INERF_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef enum inerf_status {
    INERF_OK = 0,
    INERF_ERR_NULL = -1,        /* required pointer is NULL */
    INERF_ERR_SIZE = -2,        /* size / count out of range */
    INERF_ERR_UNSUPPORTED = -3, /* configuration the kernels do not implement */
    INERF_ERR_WORKSPACE = -4,   /* workspace too small */
    INERF_ERR_ALIGN = -5        /* pointer not aligned as required */
} inerf_status;

typedef enum inerf_dtype { INERF_F32 = 0, INERF_F16 = 1 } inerf_dtype;

/* Library / ABI version (major*1000 + minor). */
int inerf_version(void);
/* Human-readable text for a return code (static storage). */
const char *inerf_error_string(int code);

/* ------------------------------------------------------------------ utils -- */

/* raymarching/src/raymarching.h:7  near_far_from_aabb (kernel raymarching.cu:91-145) */
int inerf_near_far_from_aabb(const float *rays_o, const float *rays_d, const float *aabb, uint32_t N,
                             float min_near, float *nears, float *fars, void *stream);
/*
 * nerf/utils.py:56-140 get_rays (Python / ~10 torch kernels in the reference; no FFI function there):
 * poses [B,4,4] row-major cam2world, intrinsics (fx, fy, cx, cy), image H x W.  `inds` = int64 [N] flat pixel indices
 * (row*W + col) shared by every pose, or NULL with N == H*W for the full frame.  Writes rays_o, rays_d [B,N,3].
 * With aabb != NULL the slab test of near_far_from_aabb is fused: nears, fars [B*N] (bit-identical to a separate call).
 */
int inerf_get_rays(const float *poses, uint32_t B, float fx, float fy, float cx, float cy, uint32_t H, uint32_t W,
                   const long long *inds, uint32_t N, float *rays_o, float *rays_d, const float *aabb, float min_near,
                   float *nears, float *fars, void *stream);
/* raymarching.h:8  sph_from_ray (raymarching.cu:162-198) */
int inerf_sph_from_ray(const float *rays_o, const float *rays_d, float radius, uint32_t N, float *coords,
                       void *stream);
/* raymarching.h:9  morton3D (raymarching.cu:214-232) */
int inerf_morton3D(const int32_t *coords, uint32_t N, int32_t *indices, void *stream);
/* raymarching.h:10 morton3D_invert (raymarching.cu:237-260) */
int inerf_morton3D_invert(const int32_t *indices, uint32_t N, int32_t *coords, void *stream);
/* raymarching.h:11 packbits (raymarching.cu:267-300); N = number of output BYTES (C*H^3/8) */
int inerf_packbits(const float *grid, uint32_t N, float density_thresh, uint8_t *bitfield, void *stream);

/* ------------------------------------------------------- training marching -- */

/*
 * raymarching.h:13 march_rays_train (raymarching.cu:311-490).
 *
 * The reference reserves sample ranges with atomicAdd, so its output order is
 * racy.  This library is deterministic: count -> exclusive scan -> write.
 * `rays` comes out sorted by ray id with offsets = exclusive prefix sum of the
 * counts, i.e. exactly the canonical form of the reference's stream.
 *
 * Two-phase use (lets the host size xyzs/dirs/deltas exactly instead of
 * zero-filling N*max_steps rows as raymarching.py:205-207 does), every ray walked ONCE:
 *   inerf_march_rays_train_count_t  walks, writes rays[N,3], adds (total, N) to counter[2] and records the
 *                                   parameter t of every sample in t_scratch;
 *   inerf_march_rays_train_expand   rebuilds the samples of every ray with offset+count <= M from t alone (one warp
 *                                   per ray, coalesced stores) -- the reference walks every ray a second time (:403-479).
 * inerf_march_rays_train does both with the reference's argument list plus the workspace.
 * t_scratch: caller-owned float[inerf_march_scratch_floats(N, max_steps)] = [N, max_steps], uninitialised.
 */
size_t inerf_march_scratch_floats(uint32_t N, uint32_t max_steps);
int inerf_march_rays_train_count_t(const float *rays_o, const float *rays_d, const uint8_t *grid, float bound,
                                   float dt_gamma, uint32_t max_steps, uint32_t N, uint32_t C, uint32_t H,
                                   const float *nears, const float *fars, int32_t *rays, int32_t *counter,
                                   const float *noises, float *t_scratch, void *stream);
int inerf_march_rays_train_expand(const float *rays_o, const float *rays_d, float bound, float dt_gamma, uint32_t max_steps,
                                  uint32_t N, uint32_t C, uint32_t H, uint32_t M, const float *nears, float *xyzs, float *dirs,
                                  float *deltas, const int32_t *rays, const float *noises, const float *t_scratch,
                                  void *stream);
int inerf_march_rays_train(const float *rays_o, const float *rays_d, const uint8_t *grid, float bound, float dt_gamma,
                           uint32_t max_steps, uint32_t N, uint32_t C, uint32_t H, uint32_t M, const float *nears,
                           const float *fars, float *xyzs, float *dirs, float *deltas, int32_t *rays,
                           int32_t *counter, const float *noises, float *t_scratch, void *stream);

/* --------------------------------------------------- training compositing -- */

/* raymarching.h:14 composite_rays_train_forward (raymarching.cu:500-588) */
int inerf_composite_rays_train_forward(const float *sigmas, const float *rgbs, const float *deltas,
                                       const int32_t *rays, uint32_t M, uint32_t N, float T_thresh,
                                       float *weights_sum, float *depth, float *image, void *stream);
/* raymarching.h:15 composite_rays_train_backward (raymarching.cu:601-693); grad_* pre-zeroed by the caller */
int inerf_composite_rays_train_backward(const float *grad_weights_sum, const float *grad_image, const float *sigmas,
                                        const float *rgbs, const float *deltas, const int32_t *rays,
                                        const float *weights_sum, const float *image, uint32_t M, uint32_t N,
                                        float T_thresh, float *grad_sigmas, float *grad_rgbs, void *stream);
/* raymarching.h:17 composite_rays_with_masks_train_forward (raymarching.cu:705-810) */
int inerf_composite_rays_with_masks_train_forward(const float *sigmas, const float *rgbs, const float *masks,
                                                  const float *deltas, const int32_t *rays, uint32_t M, uint32_t N,
                                                  uint32_t K, float T_thresh, float *weights_sum, float *depth,
                                                  float *image, float *mask_out, void *stream);
/* raymarching.h:18 composite_rays_with_masks_train_backward (raymarching.cu:828-951).
 * grad_masks_acc (the reference's global scratch, raymarching.cu:844) is accepted
 * for signature compatibility and may be NULL: the running sums live in registers. */
int inerf_composite_rays_with_masks_train_backward(const float *grad_weights_sum, const float *grad_image,
                                                   const float *grad_mask_out, const float *sigmas, const float *rgbs,
                                                   const float *masks, const float *deltas, const int32_t *rays,
                                                   const float *weights_sum, const float *image, const float *mask_out,
                                                   uint32_t M, uint32_t N, uint32_t K, float T_thresh,
                                                   float *grad_sigmas, float *grad_rgbs, float *grad_masks_acc,
                                                   float *grad_masks, void *stream);

/* Same backward for a DENSE sample stream (every row of the gradient buffers belongs to exactly one ray of `rays`, as the
 * count -> scan -> expand marcher produces it): the kernel writes the zero gradients of the samples behind a ray's
 * termination itself, so grad_sigmas / grad_rgbs / grad_masks may be uninitialised memory (no memset of 16 + 4K bytes per
 * sample), and grad_sigmas / grad_rgbs may be NULL when the caller does not need them (instance stage: the sigma and colour
 * nets are frozen, nerf/utils.py:1242-1246).  K == 0: composite_rays_train_backward (raymarching.h:16).  K <= 64. */
int inerf_composite_rays_with_masks_train_backward_dense(const float *grad_weights_sum, const float *grad_image,
                                                         const float *grad_mask_out, const float *sigmas, const float *rgbs,
                                                         const float *masks, const float *deltas, const int32_t *rays,
                                                         const float *weights_sum, const float *image, const float *mask_out,
                                                         uint32_t M, uint32_t N, uint32_t K, float T_thresh,
                                                         float *grad_sigmas, float *grad_rgbs, float *grad_masks, void *stream);

/* -------------------------------------------------------------- inference -- */

/* raymarching.h:20 march_rays (raymarching.cu:958-1073); xyzs/dirs/deltas pre-zeroed by the caller */
int inerf_march_rays(uint32_t n_alive, uint32_t n_step, const int32_t *rays_alive, const float *rays_t,
                     const float *rays_o, const float *rays_d, float bound, float dt_gamma, uint32_t max_steps,
                     uint32_t C, uint32_t H, const uint8_t *grid, const float *nears, const float *fars, float *xyzs,
                     float *dirs, float *deltas, const float *noises, void *stream);
/* raymarching.h:21 composite_rays (raymarching.cu:1076-1172) */
int inerf_composite_rays(uint32_t n_alive, uint32_t n_step, float T_thresh, int32_t *rays_alive, float *rays_t,
                         const float *sigmas, const float *rgbs, const float *deltas, float *weights_sum,
                         float *depth, float *image, void *stream);
/* raymarching.h:22 composite_rays_with_masks (raymarching.cu:1175-1280) */
int inerf_composite_rays_with_masks(uint32_t n_alive, uint32_t n_step, uint32_t K, float T_thresh,
                                    int32_t *rays_alive, float *rays_t, const float *sigmas, const float *rgbs,
                                    const float *masks, const float *deltas, float *weights_sum, float *depth,
                                    float *image, float *mask_out, void *stream);
/* Device-side stream compaction replacing `rays_alive[rays_alive >= 0]`
 * (nerf/mask_renderer.py:370): stable, writes the survivors to `out` and their
 * number to n_out[0].  `out` must not alias `rays_alive`. */
int inerf_compact_alive(const int32_t *rays_alive, uint32_t n_alive, int32_t *out, int32_t *n_out, void *stream);

/* ------------------------------------------------------------ grid encoder -- */

/*
 * gridencoder/src/gridencoder.h:12 grid_encode_forward (gridencoder.cu:87-242, 445-468).
 *   inputs      float [B, D] in [0, 1]
 *   embeddings  [offsets[L], C] of `dtype`
 *   offsets     int32 [L + 1]
 *   outputs     `dtype`; out_layout 0 = [L, B, C] (what the reference kernel
 *               writes, grid.py:47), 1 = [B, L*C] (what grid.py:57 permutes to)
 *   dy_dx       optional [B, L*D*C] of `dtype`, or NULL
 *   S = log2(per_level_scale), H = base resolution, gridtype 0 = hash / 1 = tiled,
 *   interp 0 = linear / 1 = smoothstep.  D in {2,3}, C in {1,2,4,8}.
 */
int inerf_grid_encode_forward(const float *inputs, const void *embeddings, const int32_t *offsets, void *outputs,
                              uint32_t B, uint32_t D, uint32_t C, uint32_t L, float S, uint32_t H, void *dy_dx,
                              uint32_t gridtype, int align_corners, uint32_t interp, int dtype, int out_layout,
                              void *stream);
/*
 * gridencoder.h:13 grid_encode_backward (gridencoder.cu:245-337, 470-500).
 *   grad            `dtype`, grad_layout 0 = [L, B, C] (grid.py:75), 1 = [B, L*C]
 *   grad_embeddings `dtype`, pre-zeroed by the caller (grid.py:77), accumulated atomically
 *   dy_dx / grad_inputs optional (NULL on the instance-field path, grid.py:156)
 */
int inerf_grid_encode_backward(const void *grad, const float *inputs, const void *embeddings, const int32_t *offsets,
                               void *grad_embeddings, uint32_t B, uint32_t D, uint32_t C, uint32_t L, float S,
                               uint32_t H, const void *dy_dx, void *grad_inputs, uint32_t gridtype,
                               int align_corners, uint32_t interp, int dtype, int grad_layout, void *stream);
/*
 * gridencoder.h:15 grad_total_variation (gridencoder.cu:504-642): adds the total-variation gradient of the grid vertices
 * hit by `inputs` (float [B, D] in [0, 1]; points outside are skipped) into `grad` (same shape / dtype as `embeddings`).
 * D in {2, 3}, C in {1, 2, 4, 8}.
 */
int inerf_grad_total_variation(const float *inputs, const void *embeddings, void *grad, const int32_t *offsets, float weight,
                               uint32_t B, uint32_t D, uint32_t C, uint32_t L, float S, uint32_t H, uint32_t gridtype,
                               int align_corners, int dtype, void *stream);

/* -------------------------------------------------------------- SH encoder -- */

/* shencoder/src/shencoder.h:9 sh_encode_forward (shencoder.cu:28-129, 386-417).
 * inputs float [B, 3], outputs float [B, degree^2], degree in [1, 8]; dy_dx optional [B, 3*degree^2]
 * (supported for degree <= 4). */
int inerf_sh_encode_forward(const float *inputs, float *outputs, uint32_t B, uint32_t D, uint32_t degree,
                            float *dy_dx, void *stream);
/* shencoder.h:10 sh_encode_backward (shencoder.cu:359-382, 419-438) */
int inerf_sh_encode_backward(const float *grad, const float *inputs, uint32_t B, uint32_t D, uint32_t degree,
                             const float *dy_dx, float *grad_inputs, void *stream);

/* --------------------------------------------------- fused instance field -- */

/*
 * One launch for NeRFNetwork.forward (nerf/network_mask.py:119-158): both hash
 * encoders, SH degree 4, sigma-net 32->64->16, colour-net 31->64->64->3 and
 * mask-net 47->64->64->K on tcgen05 tensor cores (fp16 operands, fp32 TMEM
 * accumulators, one fp16 rounding per layer as under torch autocast).
 *
 * `weights` is the packed fp16 blob produced by inerf_field_pack_weights from
 * the fp32 nn.Linear matrices ([out, in] row-major, network_mask.py:48,69,90).
 */
typedef struct inerf_field_desc {
    const void *table_packed;  /* fp16 [offsets[L], 4]: (encoder.embeddings c0 c1, encoder_mask.embeddings c0 c1)
                                  interleaved per entry by inerf_field_pack_tables: one 8-byte gather per corner
                                  serves both encoders (they share level geometry, network_mask.py:34,76) */
    const int32_t *offsets;    /* int32 [L + 1] (shared by both encoders)      */
    const void *weights;       /* packed fp16 blob, inerf_field_weights_bytes(K) bytes */
    uint32_t L;                /* 16 */
    uint32_t H;                /* base resolution 16 */
    float S;                   /* log2(per_level_scale) */
    float bound;               /* scene bound: x01 = (x + bound) / (2 bound) */
    uint32_t K;                /* num_instances, 1..64 */
    float density_scale;       /* mask_renderer.py:273 */
    const int32_t *n_valid;    /* optional device int32: rows >= *n_valid of a sample stream are padding and are not
                                  evaluated (fixed-size streams of a CUDA-graph-captured training step); NULL = all B rows */
} inerf_field_desc;

/* emb_sigma / emb_mask: device [n_entries, 2] of `dtype` (INERF_F32 parameters or INERF_F16) -> packed fp16 [n_entries, 4] */
int inerf_field_pack_tables(const void *emb_sigma, const void *emb_mask, int dtype, uint64_t n_entries, void *packed,
                            void *stream);
size_t inerf_field_weights_bytes(uint32_t K);
/* host-side packing (CPU pointers): w_* are fp32 row-major [out, in] */
int inerf_field_pack_weights(const float *sigma0, const float *sigma1, const float *color0, const float *color1,
                             const float *color2, const float *mask0, const float *mask1, const float *mask2,
                             uint32_t K, void *packed_host);
/* xyzs/dirs float [B,3]; sigmas float [B]; rgbs float [B,3]; masks float [B,K] (NULL = skip mask-net) */
int inerf_field_forward(const inerf_field_desc *desc, const float *xyzs, const float *dirs, uint32_t B,
                        float *sigmas, float *rgbs, float *masks, void *stream);

/*
 * Training forward: inerf_field_forward that also keeps, per sample, the mask-net input row
 * (32 mask-table features | 15 geo features | 0) as fp16 [B, 48] in `x0_save` (16-byte aligned) for the backward.
 */
int inerf_field_forward_train(const inerf_field_desc *desc, const float *xyzs, const float *dirs, uint32_t B,
                              float *sigmas, float *rgbs, float *masks, void *x0_save, void *stream);
/*
 * Backward of the instance head in ONE launch (instance stage of MaskTrainer, nerf/utils.py:1242-1246: sigma / colour
 * nets frozen).  Replaces autograd through mask_net (network_mask.py:150-154: 6 cuBLAS GEMMs + ReLU / cat backward)
 * and kernel_grid_backward of encoder_mask (gridencoder.cu:245-337).
 *   weights_bwd  packed fp16 blob from inerf_field_pack_weights_bwd (inerf_field_bwd_weights_bytes() bytes, device)
 *   x0           fp16 [B, 48] saved by inerf_field_forward_train
 *   grad_logits  float [B, K]  = dL/d(mask logits) per sample (output of composite_rays_with_masks_train_backward)
 *   grad_table   float [offsets[L], 2], grad_w0 float [64, 47], grad_w1 float [64, 64], grad_w2 float [K, 64]:
 *                ACCUMULATED into (atomics), so the caller zeroes them (or passes .grad buffers to accumulate).
 */
size_t inerf_field_bwd_weights_bytes(void);
/* Same packing as inerf_field_pack_weights (+ _bwd when packed_bwd != NULL) from DEVICE fp32 matrices into DEVICE blobs,
 * one launch on `stream`, no host round trip (the trainable weights change every optimizer step). */
int inerf_field_pack_weights_device(const float *sigma0, const float *sigma1, const float *color0, const float *color1,
                                    const float *color2, const float *mask0, const float *mask1, const float *mask2,
                                    uint32_t K, void *packed_fwd, void *packed_bwd, void *stream);
int inerf_field_pack_weights_bwd(const float *mask0, const float *mask1, const float *mask2, uint32_t K, void *packed_host);
int inerf_field_backward_mask(const inerf_field_desc *desc, const void *weights_bwd, const float *xyzs, const void *x0,
                              const float *grad_logits, uint32_t B, float *grad_table, float *grad_w0, float *grad_w1,
                              float *grad_w2, void *stream);

/* ---- stage-1 (RGB-sigma) training: Trainer.train_step (nerf/utils.py:536-632) on network.py:96-127 ----------------------
 * inerf_field_forward_train_rgb = inerf_field_forward with the instance head off, plus `xs_save` fp16 [B, 64]: the inputs of
 * sigma_net (32 table features) and color_net (SH16 | geo15 | 0) per sample.
 * inerf_field_backward_rgb replaces, in ONE launch, what autograd runs for that network: 10 GEMMs, the ReLU / sigmoid /
 * trunc_exp (activation.py:13-17) backward kernels and kernel_grid_backward of `encoder` (gridencoder.cu:245-337).
 *   sigmas / rgbs          the forward outputs (sigma unscaled), grad_sigmas / grad_rgbs their gradients (float [B], [B,3])
 *   grad_table             float [offsets[L], 2] (encoder.embeddings.grad)
 *   grad_ws0 [64,32], grad_ws1 [16,64], grad_wc0 [64,31], grad_wc1 [64,64], grad_wc2 [3,64]   (nn.Linear layout)
 * All gradient outputs are ACCUMULATED into (atomics): the caller zeroes them or passes .grad buffers. */
size_t inerf_field_rgb_bwd_weights_bytes(void);
int inerf_field_pack_weights_rgb_bwd_device(const float *sigma0, const float *sigma1, const float *color0, const float *color1,
                                            const float *color2, void *packed_bwd, void *stream);
int inerf_field_forward_train_rgb(const inerf_field_desc *desc, const float *xyzs, const float *dirs, uint32_t B, float *sigmas,
                                  float *rgbs, void *xs_save, void *stream);
int inerf_field_backward_rgb(const inerf_field_desc *desc, const void *weights_bwd, const float *xyzs, const void *xs,
                             const float *sigmas, const float *rgbs, const float *grad_sigmas, const float *grad_rgbs,
                             uint32_t B, float *grad_table, float *grad_ws0, float *grad_ws1, float *grad_wc0,
                             float *grad_wc1, float *grad_wc2, void *stream);

/*
 * Whole-frame inference render in ONE persistent launch, replacing the host
 * loop of NeRFMaskRenderer.run_cuda (nerf/mask_renderer.py:322-381):
 * march -> encode -> MLP -> composite per 128-ray tile, ray state in registers,
 * no sample stream in HBM.  Outputs are the un-normalised accumulators the
 * reference loop produces before mask_renderer.py:376-377.
 * `work_counter` is caller-owned scratch, int32[4], 8-byte aligned; the call
 * zeroes it, uses [0] as the ray cursor and leaves the number of 128-row tiles
 * it evaluated in [1] and the number of samples it composited in [2..3] (one
 * uint64), which bench.py reads for the roofline and the tile fill rate.
 */
int inerf_render_fused(const inerf_field_desc *desc, const float *rays_o, const float *rays_d, const float *nears,
                       const float *fars, const uint8_t *bitfield, uint32_t N, uint32_t C, uint32_t H,
                       float dt_gamma, uint32_t max_steps, float T_thresh, float *weights_sum, float *depth,
                       float *image, float *mask_out, int32_t *work_counter, void *stream);

/* Same with the first step of every ray jittered as the reference's run_cuda does for perturb=True (mask_renderer.py:334-337 ->
 * raymarching.cu:1004: t = near + clamp(near * dt_gamma, dt_min, dt_max) * noises[ray]); noises float [N] in [0, 1), NULL = none. */
int inerf_render_fused_perturb(const inerf_field_desc *desc, const float *rays_o, const float *rays_d, const float *nears,
                               const float *fars, const float *noises, const uint8_t *bitfield, uint32_t N, uint32_t C, uint32_t H,
                               float dt_gamma, uint32_t max_steps, float T_thresh, float *weights_sum, float *depth,
                               float *image, float *mask_out, int32_t *work_counter, void *stream);

/* --------------------------------------------------------------- loss tail -- */

/*
 * MaskTrainer.train_step's loss on the composited maps (nerf/utils.py:1310-1314 cross-entropy over labelled pixels,
 * label -1 = unlabelled; nerf/utils.py:1262-1285 depth-aware label smoothness on patch x patch pixel blocks, batch order
 * patch-major as produced by get_rays, nerf/utils.py:83-100).  logits float [N, K], depth float [N], labels int64 [N],
 * N a multiple of patch^2 (patch = 1: cross-entropy only).  acc6 = 6 floats of caller-owned scratch kept for the backward.
 * Backward writes grad_logits [N, K] = upstream[0] * dloss/dlogits (upstream NULL = 1); no gradient goes to depth
 * (the compositor drops grad_depth, raymarching.py:342).
 */
int inerf_mask_loss(const float *logits, const float *depth, const long long *labels, uint32_t N, uint32_t K,
                    uint32_t patch, float reg_weight, float *acc6, float *loss_out, void *stream);
int inerf_mask_loss_backward(const float *logits, const float *depth, const long long *labels, uint32_t N, uint32_t K,
                             uint32_t patch, float reg_weight, const float *acc6, const float *upstream,
                             float *grad_logits, void *stream);

/* ------------------------------------------------------ occupancy grid EMA -- */

/*
 * nerf/mask_renderer.py:532-540 as two launches without host syncs:
 *   grid[i] = max(grid[i]*decay, tmp[i]) where both >= 0; sum(clamp(grid,0)) -> mean_out[0] (pre-zeroed),
 *   then packbits with thresh = min(mean, density_thresh).
 */
int inerf_occupancy_ema(float *density_grid, const float *tmp_grid, uint32_t n_cells, float decay,
                        double *sum_out, void *stream);
int inerf_occupancy_pack(const float *density_grid, uint32_t n_cells, const double *sum_in, float density_thresh,
                         uint8_t *bitfield, float *mean_out, void *stream);

/* ------------------------------------------- occupancy grid: sampling front -- */

/*
 * nerf/mask_renderer.py:466-527 (update_extra_state, the part before the EMA) and :389-452 (mark_untrained_grid) as
 * device code: no meshgrid / randint / nonzero / index_put, no host read.
 *
 * A "sweep" is C * per_cascade samples; sample s belongs to cascade c = s / per_cascade and to the cell with Morton
 * index cells[s] (cells == NULL: cell s % G^3, the full sweep of the first 16 updates, per_cascade = G^3).  Its point is
 * the cell centre `(2 * coord / (G - 1) - 1) * (bound_c - bound_c / G)` plus `(u * 2 - 1) * bound_c / G` per axis
 * (:480-487), u = noise[s, :] when noise != NULL (parity tests inject the reference's rand_like draws) else a
 * counter-based generator keyed by `seed`.
 *
 *   inerf_occupancy_sample_cells  partial update (:498-513): per cascade N uniform cells + N cells drawn with
 *                                 replacement from the occupied ones (density_grid[c] > 0), compacted in torch.nonzero
 *                                 order on the device -> cells [C, 2N].  uniform_cells [C, N] / occ_picks [C, N]
 *                                 (positions in the occupied list) inject the draws; NULL = generator.  scratch:
 *                                 int32[inerf_occupancy_sample_scratch_ints(C, G)], caller-owned.
 *   inerf_occupancy_points        the sweep's points xyzs [C * per_cascade, 3] and flat cell indices c * G^3 + cell
 *                                 (for networks the fused sweep does not cover, and for tests).
 *   inerf_occupancy_density       fused: point -> hash encode -> sigma-net (tcgen05) -> tmp_grid[c, cell] =
 *                                 sigma * desc->density_scale, one launch.  tmp_grid [C, G^3] is only written at the
 *                                 sampled cells (pre-fill with -1 for a partial sweep: inerf_fill_f32).
 *   inerf_mark_untrained_grid     density_grid[c, cell] = -1 for every cell whose centre no camera sees (c2w poses
 *                                 [B, 4, 4] row-major, pinhole fx fy cx cy, margin 2 * bound_c / G); *n_marked
 *                                 (optional, pre-zeroed) counts them.
 */
size_t inerf_occupancy_sample_scratch_ints(uint32_t C, uint32_t G);
int inerf_occupancy_sample_cells(const float *density_grid, uint32_t C, uint32_t G, uint32_t N,
                                 const int32_t *uniform_cells, const int32_t *occ_picks, uint64_t seed, int32_t *cells,
                                 int32_t *scratch, void *stream);
int inerf_occupancy_points(uint32_t C, uint32_t G, float bound, const int32_t *cells, uint32_t per_cascade,
                           const float *noise, uint64_t seed, float *xyzs, int32_t *flat_index, void *stream);
int inerf_occupancy_density(const inerf_field_desc *desc, uint32_t C, uint32_t G, const int32_t *cells,
                            uint32_t per_cascade, const float *noise, uint64_t seed, float *tmp_grid, void *stream);
int inerf_mark_untrained_grid(const float *poses, uint32_t B, float fx, float fy, float cx, float cy, uint32_t C,
                              uint32_t G, float bound, float *density_grid, uint32_t *n_marked, void *stream);
int inerf_fill_f32(float *p, uint32_t n, float value, void *stream);

/* ------------------------------------------------------------- optimizer -- */

/*
 * The Adam step the reference trainer takes on the trainable parameters (main_nerf_mask.py:182,
 * torch.optim.Adam(betas=(0.9, 0.99), eps=1e-15); no weight decay / amsgrad), fused with the AMP unscale and with
 * clearing the gradient: one pass over param / grad / exp_avg / exp_avg_sq (fp32 [n], 16-byte aligned) instead of
 * zero_grad + unscale + Adam.  `step` is a device float holding the number of steps taken so far; grad_scale and
 * found_inf are GradScaler's device scalars (NULL = 1 / 0).  found_inf != 0 leaves parameters and moments unchanged
 * (the gradient is cleared either way).  grad_div (> 0) divides the gradient once more: data-parallel training passes the
 * world size, so the SUM all-reduce needs no separate averaging pass (1 = single GPU, bit-identical to no division).
 * Call inerf_adam_advance(step, found_inf) once after all tensors of a step.
 */
int inerf_adam_step(float *param, float *grad, float *exp_avg, float *exp_avg_sq, uint64_t n, float lr, float beta1,
                    float beta2, float eps, const float *step, const float *grad_scale, const float *found_inf,
                    float grad_div, void *stream);
int inerf_adam_advance(float *step, const float *found_inf, void *stream);

/* ---- 3D-mask projection (scripts/project_3d_masks.py:135-266) ------------------------------------------------------------
 * The labelled voxels of the predicted 3D masks (generate_predicted_grid, :108-131: labels int32 [nx, ny, nz], 0 = none) seen
 * from a camera: every ray (rays_o / rays_d as inerf_get_rays builds them for that pose) walks the grid of cells centred on the
 * reference's points (grid_pts_coord, :72-83; bbox_host = room_bbox as 6 HOST floats: min xyz, max xyz) with an exact 3D DDA;
 * out_label[r] = first non-zero label along ray r (0: none), out_t[r] (may be NULL) = ray parameter where that cell is entered.
 * Replaces the PyTorch3D point rasteriser of the reference (nearest labelled point per pixel). */
int inerf_project_labels(const float *rays_o, const float *rays_d, uint32_t N, const int32_t *labels, uint32_t nx, uint32_t ny,
                         uint32_t nz, const float *bbox_host, int32_t *out_label, float *out_t, void *stream);

/* ---- volume extraction: the trained fields on a voxel grid ------------------------------------------------------------------
 * The grid geometry and label convention of inerf_project_labels, so that an extracted label volume projects unchanged.
 *
 * Voxel (i,j,k) of an X x Y x Z grid over bbox (6 HOST floats: lo xyz, hi xyz) -> its point
 *   p = lo + ((float)i / (float)X) * (hi - lo)        (per axis; fp32; one IEEE op each, in this order)
 * = projection.voxel_points / grid_pts_coord, the cell centres inerf_project_labels walks.
 * occupied (optional, u8 [X*Y*Z]): 1 where the point's occupancy cell is set in `bitfield` (NULL bitfield: all 1).  The cell
 * is the one the marcher tests for a sample at p with dt = 0: cascade = clamped exponent of max|p|, then the cell of p in it.
 * Every axis is 1..2048, X*Y*Z < 2^31, lo < hi on every axis and the bbox lies inside [-bound, bound]^3.
 */
int inerf_volume_points(const float *bbox_host, uint32_t X, uint32_t Y, uint32_t Z, const uint8_t *bitfield, uint32_t C,
                        uint32_t H, float bound, float *xyzs, uint8_t *occupied, void *stream);

size_t inerf_extract_scratch_ints(uint32_t X, uint32_t Y, uint32_t Z);
/* The fields at every voxel, outputs C order [X,Y,Z](,3), each optional (at least one):
 *   sigma  = density * desc->density_scale           (the sigma run_cuda composites and density_grid stores)
 *   rgb    = colour for the single view direction view_dir_host (3 HOST floats; required iff rgb != NULL)
 *   label  = 1 + argmax_k logits  if the voxel is live and sigma >= sigma_thresh, else 0
 * Field values are bit-identical to inerf_field_forward at the voxel's point (d = view_dir), sigma multiplied by
 * density_scale in fp32; the argmax runs over the fp16-rounded logits it stores, lowest index on ties.
 * bitfield != NULL: a voxel whose occupancy cell is empty is NOT evaluated: sigma 0, rgb 0, label 0.
 * bitfield == NULL: every voxel is evaluated.
 * n_live (optional, device int32): number of voxels evaluated.  scratch: caller-owned, uninitialised,
 * int32[inerf_extract_scratch_ints(X, Y, Z)]; required iff bitfield != NULL.  Every output element is written once. */
int inerf_extract_volume(const inerf_field_desc *desc, const float *bbox_host, uint32_t X, uint32_t Y, uint32_t Z,
                         const uint8_t *bitfield, uint32_t C, uint32_t H, const float *view_dir_host, float sigma_thresh,
                         float *sigma, float *rgb, int32_t *label, int32_t *scratch, int32_t *n_live, void *stream);

/* ---- mesh export: marching cubes over a float volume ------------------------------------------------------------------------
 * v: device float [X,Y,Z] in C order, sample (i,j,k) at the voxel point of inerf_volume_points:
 *   p = lo + ((float)i / (float)X) * (hi - lo)        (per axis; bbox_host = 6 HOST floats lo xyz, hi xyz; finite, lo < hi)
 * Inside means v > iso (NaN: outside).  The table (csrc/mc_table.h, generated by scripts/gen_mc_table.py) cuts every run of
 * inside corners on a cube face off by its own segment, so neighbouring cubes agree and the surface is closed where it does
 * not reach the volume's border; triangle normals (right-hand rule) point toward v < iso.
 *   vertices   one per lattice edge whose two samples differ in inside-ness, owned by its lower sample; ordered by that
 *              sample's C-order index, then by axis (x, y, z).  Along the edge's axis the vertex sits at s = (float)i + t,
 *              t = fminf(fmaxf((iso - va) / (vb - va), 0), 1), world coordinate lo + (s / (float)X) * (hi - lo); the other two
 *              coordinates are the sample's own.  fp32, one IEEE op each, in this order (a vertex with t = 0 is the voxel
 *              point bit for bit; the clamp gives a NaN sample the lower end).
 *   triangles  int32 [F,3] vertex indices, ordered by cube (C order of its lower corner) and then by table order.
 * Every output position is a prefix sum over C order (no atomics): the same bytes on every run.
 * Every axis is 2..2048, X*Y*Z < 2^31, and 3*X*Y*Z and 5*(X-1)*(Y-1)*(Z-1) (the most vertices / triangles a volume can
 * yield) < 2^31, so that every index and count fits int32.
 * Two calls: inerf_mesh_count leaves (V, F) in counts[2] (device int32) and its per-sample state in scratch (caller-owned,
 * uninitialised, int32[inerf_mesh_scratch_ints(X, Y, Z)]; 0 = sizes out of range); the caller sizes verts float [V,3] and
 * tris int32 [F,3] and calls inerf_mesh_emit with the same v, sizes, iso and scratch (F == 0: nothing to emit). */
size_t inerf_mesh_scratch_ints(uint32_t X, uint32_t Y, uint32_t Z);
int inerf_mesh_count(const float *v, uint32_t X, uint32_t Y, uint32_t Z, float iso, int32_t *scratch, int32_t *counts, void *stream);
int inerf_mesh_emit(const float *v, uint32_t X, uint32_t Y, uint32_t Z, const float *bbox_host, float iso, int32_t *scratch,
                    float *verts, int32_t *tris, void *stream);

/* ---- frame finalisation (MaskTrainer.test / evaluate_one_epoch, nerf/utils.py:1425-1431, 1461-1485, 1624-1634) ----------------
 * rgb[N,3] / depth_u8[N] = (x * 255) truncated to uint8 (saturating), label[N] = argmax_k logits[N,K] (= the reference's
 * softmax + argmax; lowest index on ties; K <= 256).  depth / depth_u8 and logits / label may be NULL in pairs. */
int inerf_frame_to_u8(const float *image, const float *depth, const float *logits, uint32_t N, uint32_t K, uint8_t *rgb,
                      uint8_t *depth_u8, uint8_t *label, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* INERF_B200_H */
