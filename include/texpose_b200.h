/* texpose_b200 -- C ABI of the B200 (sm_100a) kernels behind TexPose's per-ray NeRF render hot path.
 *
 * The reference (HanzhiC/TexPose) is pure Python/PyTorch and has no FFI of its own (SURVEY.md section 8b):
 * the drop-in boundary is its Python call surface, and every entry point below replaces the aten-op
 * sequence of one reference function (cited per declaration, paths relative to the reference checkout).
 * INTEGRATION.md shows the ctypes binding and the reference-side patch.
 *
 * Conventions
 *   - all pointers are DEVICE pointers into caller-owned memory unless marked "host"; the library never
 *     allocates or frees device memory and keeps no mutable global state;
 *   - tensors are dense row-major fp32 unless a leading dimension (`ld*`, in elements) is given;
 *   - every call takes the caller's cudaStream_t as `void* stream`, enqueues asynchronously and never
 *     synchronises;
 *   - return value: 0 ok; <0 argument/shape/alignment/arch/workspace error (TP_ERR_*); >0 a cudaError_t;
 *   - no CPU fallback and no backend dispatch: a device that is not sm_100 yields TP_ERR_ARCH from the
 *     tensor-core entry points.
 */
#ifndef TEXPOSE_B200_H_
#define TEXPOSE_B200_H_
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define TP_VERSION 100

/* epilogues of tp_linear_forward */
#define TP_ACT_NONE 0
#define TP_ACT_RELU 1
#define TP_ACT_TRUNK_LAST_STL 2   /* row 0 -> softplus -> aux0 = density[S,2] col 0; rows 1.. -> relu -> Y[:, n-1] */
#define TP_ACT_TRUNK_LAST_PLAIN 3 /* same with aux0 = density[S] */
#define TP_ACT_RGB_STATIC 4       /* sigmoid -> Y = rgb[S,3,2] slot 0 */
#define TP_ACT_TRANS_OUT 5        /* rows 0-2 sigmoid -> Y = rgb[S,3,2] slot 1; row 3 softplus -> aux0 = density[S,2] col 1;
                                     row 4 softplus -> aux1 = uncert[S] */
#define TP_ACT_SIGMOID 6

int tp_version(void);
/* 1 when the current device is compute capability 10.x (tcgen05/TMEM available), else 0. */
int tp_device_is_sm100(void);

/* ---- rays / sampling (K1) ------------------------------------------------------------------------------- */

/* K^-1 [B,3,3] and pose^-1 [B,3,4] of B views in one launch (camera.py:267 `cam_intr.inverse()`, camera.py:38-44
 * Pose.invert): intr [B,3,3], pose [B,3,4] = [R|t].  K^-1 = fp64 cofactor formula rounded to fp32 (last-bit differences from
 * torch's LU-based inverse; the fp32 parity mode keeps torch's call); pose^-1 = [R^T | (-R^T) t]. */
int tp_view_matrices(const float* intr, const float* pose, int B, float* kinv, float* pose_inv, void* stream);

/* camera.get_center_and_ray (camera.py:292-314) + Graph.ray_batch_sample (model/nerf_adapt_st_gan.py:702-710).
 * kinv [B,3,3] = intr.inverse(), pose_inv [B,3,4] = Pose().invert(pose) (host-side torch calls, a1 in SURVEY 8a).
 * ray_idx: NULL -> all H*W pixels (R must equal H*W); else int64 [B,R] pixel indices.  pix_offset 0.5. */
int tp_raygen(const float* kinv, const float* pose_inv, int B, int H, int W, float pix_offset, const int64_t* ray_idx,
              int R, float* center, float* ray, void* stream);

/* RaySampler.get_rays (tools/ray_sampler.py:39-69): coords [B,P,2] in [-1,1] (x,y), bilinear ramp lookup, no +0.5. */
int tp_patch_rays(const float* kinv, const float* pose_inv, const float* coords, int B, int P, int H, int W,
                  float* center, float* ray, void* stream);

/* F.grid_sample(image[B,C,H,W], coords[B,P,2], bilinear, zeros, align_corners=True) -> out [B,C,P]
 * (RaySampler.get_bounds / get_image, tools/ray_sampler.py:12-37). */
int tp_grid_sample_bilinear(const float* image, const float* coords, int B, int C, int H, int W, int P, float* out,
                            void* stream);

/* Graph.ray_batch_sample on an arbitrary [B,HW,C] tensor (model/nerf_adapt_st_gan.py:702-710). */
int tp_gather_rows(const float* src, const int64_t* idx, int B, int64_t HW, int C, int R, float* out, void* stream);

/* camera.aabb_ray_intersection (camera.py:415-433; compute_box.py:69-87).  aabb_* [3] or, if aabb_batched, [B,3].
 * Bit-exact incl. NaN propagation for axis-parallel rays.  valid: uint8 [B,n]. */
int tp_aabb_intersect(const float* aabb_min, const float* aabb_max, int aabb_batched, const float* ray_o,
                      const float* ray_d, int B, int64_t n_per_batch, float* t_near, float* t_far, uint8_t* valid,
                      void* stream);

/* Graph.sample_depth, metric parametrisation (model/nerf_adapt_st_gan.py:682-700).
 * mode 0: rand [n_rays,N] supplied (the torch.rand draw); 1: midpoint 0.5 (sample_stratified false);
 * 2: in-kernel Philox4x32-10 jitter keyed by (seed, sample index).  out [n_rays,N]. */
int tp_sample_depth(const float* z_near, const float* z_far, const float* rand, int64_t n_rays, int N, int mode,
                    uint64_t seed, float* out, void* stream);

/* compute_box.py:266-271 + data/lm.py:349-350 fused: full-frame rays -> slab test -> misses zeroed ->
 * zeros replaced by the background range.  z_near/z_far [B,H*W]; valid may be NULL. */
int tp_box_range(const float* kinv, const float* pose_inv, int B, int H, int W, const float* aabb_min,
                 const float* aabb_max, int aabb_batched, float bg_near, float bg_far, float* z_near, float* z_far,
                 uint8_t* valid, void* stream);

/* 'render' range source: 0.8/1.2 x depth, zeros -> background (data/lm.py:352-356). */
int tp_depth_guided_range(const float* depth, int64_t n, float bg_near, float bg_far, float* z_near, float* z_far,
                          void* stream);

/* compute_surfelinfo.normal_from_depth (compute_surfelinfo.py:37-55).  depth [B,H,W] -> normal [B,3,H,W]. */
int tp_normal_from_depth(const float* kinv, const float* pose_inv, const float* depth, int B, int H, int W,
                         float* normal, void* stream);

/* ---- mask-prior frames (render_by_slices, model/nerf_adapt_st_gan.py:633-680, modes other than 'val') ---------------------- */

/* Object-pixel ray list of B views for the list mode of the render launches (tp_render_fused_forward_list,
 * tp_tc32_render_forward_list): mask [B,HW] fp32, object pixel = mask > 0 (the reference's test, :655).  list [list_cap] int64
 * receives, view after view, the entries q = b*HW + pixel of the view's object pixels in ascending order (`nonzero`'s order),
 * each view's run padded to a multiple of u = 256 / N entries (one super-tile of the lock-step kernel, two tiles of the staged
 * one: no tile holds rays of two views) with pad entries ~(b*HW) (negative; rendered as pixel 0 of view b, never stored); an
 * empty view has no entries.  DEVICE outputs: n_slots [1] = the number of entries, counts [B] = object pixels per view.  Nothing
 * is read back; three launches, no atomics (the order is deterministic).  N in {32, 64, 128};
 * list_cap >= tp_mask_ray_list_capacity(B, HW, N); workspace >= tp_mask_ray_list_workspace(B, HW) bytes, 8-byte aligned. */
int64_t tp_mask_ray_list_capacity(int B, int64_t HW, int N);
int64_t tp_mask_ray_list_workspace(int B, int64_t HW);
int tp_mask_ray_list(const float* mask, int B, int64_t HW, int N, int64_t* list, int64_t list_cap, int64_t* n_slots,
                     int64_t* counts, void* workspace, int64_t ws_bytes, void* stream);

/* The defaults of :657-667 at the background pixels (mask <= 0) of pixels [pix0, pix1) of every view: rgb, rgb_static,
 * rgb_transient [B*HW,3] = 0; depth, opacity, opacity_static, opacity_transient [B*HW] = 0; uncert [B*HW] = min_uncert;
 * alpha_static, alpha_transient [B*HW*N] = 1; density [B*HW*N,2] = 1 (N a multiple of 4; these three 16-byte aligned).  Object
 * pixels are never touched.  Any output may be NULL and may address a peer GPU's memory (the frame layout of a FrameGather window). */
int tp_mask_defaults(const float* mask, int B, int64_t HW, int64_t pix0, int64_t pix1, int N, float min_uncert, float* rgb,
                     float* rgb_static, float* rgb_transient, float* depth, float* opacity, float* opacity_static,
                     float* opacity_transient, float* uncert, float* alpha_static, float* alpha_transient, float* density,
                     void* stream);

/* ---- compositing (K3) ----------------------------------------------------------------------------------- */

/* NeRF.composite, static/transient/joint chains (layers/nerf_static_transient_light.py:168-212).
 * ray [R,3]; rgb [R,N,3,2]; density [R,N,2]; depth [R,N]; uncert [R,N].
 * outputs: rgb, rgb_static, rgb_transient [R,3]; depth, opacity(3x), uncert [R]; prob, alpha_static, alpha_transient [R,N]. */
int tp_composite_stl_forward(const float* ray, const float* rgb, const float* density, const float* depth,
                             const float* uncert, int64_t R, int N, float min_uncert, float* o_rgb,
                             float* o_rgb_static, float* o_rgb_transient, float* o_depth, float* o_opacity,
                             float* o_opacity_static, float* o_opacity_transient, float* o_prob, float* o_uncert,
                             float* o_alpha_static, float* o_alpha_transient, void* stream);

/* Backward of the above w.r.t. rgb, density, uncert samples.  Any g_* may be NULL (= zero gradient).
 * depth/ray receive no gradient (they come from no_grad rays + rand in the reference). */
int tp_composite_stl_backward(const float* ray, const float* rgb, const float* density, const float* depth,
                              const float* uncert, int64_t R, int N, const float* g_rgb, const float* g_rgb_static,
                              const float* g_rgb_transient, const float* g_depth, const float* g_opacity,
                              const float* g_opacity_static, const float* g_opacity_transient, const float* g_prob,
                              const float* g_uncert, const float* g_alpha_static, const float* g_alpha_transient,
                              float* d_rgb, float* d_density, float* d_uncert, void* stream);

/* NeRF.composite of the plain model (layers/nerf.py:117-136).  rgb [R,N,3]; density [R,N]. */
int tp_composite_plain_forward(const float* ray, const float* rgb, const float* density, const float* depth,
                               int64_t R, int N, int use_bg, float bgcolor, float* o_rgb, float* o_depth,
                               float* o_opacity, float* o_prob, void* stream);
int tp_composite_plain_backward(const float* ray, const float* rgb, const float* density, const float* depth,
                                int64_t R, int N, int use_bg, float bgcolor, const float* g_rgb, const float* g_depth,
                                const float* g_opacity, const float* g_prob, float* d_rgb, float* d_density,
                                void* stream);

/* ---- MLP, fp32 SIMT parity path + generic layer backward (K2 fp32 / K2b) ---------------------------------- */

/* NeRF.positional_encoding with the raw coordinates prepended (layers/nerf_static_transient_light.py:81-82,217-223):
 * enc[s, 0:3+6L] for x = center[s/N] + ray[s/N] * depth[s] (camera.py:317-322). */
int tp_points_encode(const float* center, const float* ray, const float* depth, int64_t S, int N, int L, float* enc,
                     int64_t ld, void* stream);
/* same for explicit points x [S,3]. */
int tp_positional_encode(const float* x, int64_t S, int L, float* enc, int64_t ld, void* stream);
/* per-ray view direction encoding; normalize!=0 applies F.normalize first (nerf_static_transient_light.py:155-157). */
int tp_view_encode(const float* ray, int64_t R, int L, int normalize, float* enc, int64_t ld, void* stream);

/* One nn.Linear (+ activation) on a segmented input: row s of X is the concatenation of nseg (<=4) segments,
 * segment i contributing seg_cols[i] columns read at seg_ptr[i][(s / seg_group[i]) * seg_ld[i] + c].
 * seg_* are HOST arrays.  W [Nout, Ktot] with leading dimension ldw; bias [Nout] or NULL.  See TP_ACT_*. */
int tp_linear_forward(const float* const* seg_ptr, const int64_t* seg_ld, const int64_t* seg_group,
                      const int32_t* seg_cols, int nseg, const float* W, int64_t ldw, const float* bias, int64_t S,
                      int Nout, int act, float* Y, int64_t ldy, float* aux0, float* aux1, void* stream);

/* dX[:, 0:K1] = (dY W[:, 0:K1]) masked by xact > 0 (xact NULL = no mask). */
int tp_linear_backward_input(const float* dY, int64_t lddy, const float* W, int64_t ldw, int64_t S, int Nout, int K1,
                             const float* xact, int64_t ldx, float* dX, int64_t lddx, void* stream);

/* dW [Nout,Ktot] (=/+=) dY^T X, db [Nout] (=/+=) colsum(dY); split-K with a fixed-order second stage. */
int64_t tp_linear_backward_weight_workspace(int64_t S, int Nout, int Ktot);
int tp_linear_backward_weight(const float* dY, int64_t lddy, const float* const* seg_ptr, const int64_t* seg_ld,
                              const int64_t* seg_group, const int32_t* seg_cols, int nseg, int64_t S, int Nout,
                              float* dW, float* db, int accumulate, float* workspace, int64_t workspace_floats,
                              void* stream);

/* out[g, :] = sum of dY rows of group g (rows g*group .. ); workspace >= min(256, ceil(group/512)) * ceil(S/group) * Nout floats. */
int tp_group_colsum(const float* dY, int64_t lddy, int64_t S, int64_t group, int Nout, float* out, float* workspace,
                    int64_t workspace_floats, void* stream);

/* gradients w.r.t. the output layers' pre-activations from the stored outputs (sigmoid / softplus). */
int tp_stl_output_grad(const float* rgb, const float* density, const float* uncert, const float* g_rgb,
                       const float* g_density, const float* g_uncert, int64_t S, float* dz_rgb, float* dz_trans,
                       float* dz_sigma, void* stream);
int tp_plain_output_grad(const float* rgb, const float* density, const float* g_rgb, const float* g_density, int64_t S,
                         float* dz_rgb, float* dz_sigma, void* stream);
int tp_trunk_last_grad(const float* dz_sigma, const float* d_feat, int64_t ldd, const float* feat, int64_t ldf,
                       int64_t S, int F, float* dz, int64_t ldz, void* stream);

/* ---- MLP, bf16 tensor-core path (K2): fused encode + trunk + both heads on tcgen05/TMEM ---------------------- */

/* Number / size of the packed weight chunks the fused kernel streams (fixed by the canonical architecture:
 * 8x256 trunk with skip at 4, 3x256 heads; options/nerf_lm_adapt_gan.yaml:9-18). */
int tp_tc_num_chunks(void);
int64_t tp_tc_chunk_bytes(void);
/* Bytes of L2-resident scratch the forward needs (parked trunk features: SMs x 2 tiles x 64 KB). */
int64_t tp_tc_scratch_bytes(void);
/* Byte offset, inside that scratch, of the cycle counters a -DTP_FWD_PROF build of the library leaves behind (debugging aid). */
int64_t tp_tc_prof_offset(void);

/* Packs fp32 nn.Linear weights (and the static biases, which ride on a constant-1 input column) into the bf16 SMEM
 * images of the chunks.  chunk_desc: DEVICE int64 [n_chunks,10] rows {W device pointer (0 = none), ld, row0, rows_valid,
 * col0, cols_valid, n_layout (256|16), bias device pointer (0 = none), bias k-column, transpose}; packed: n_chunks*chunk_bytes.
 * n_layout 16 (the output stages, <= 8 rows): rows 0..7 of the chunk hold bf16(W), rows 8..15 bf16(W - bf16(W)); the kernel
 * adds the two accumulator columns, so the output layers see their weights to ~16 mantissa bits. */
int tp_tc_pack_weights(const int64_t* chunk_desc, int n_chunks, void* packed, void* stream);

/* Both heads' image biases in one launch (per-image constants folded into a bias; fp32):
 * out_rgb[b,:] = b_rgb + W_rgb[:, col_rgb:col_rgb+n_light] light[b],
 * out_trans[b,:] = b_trans + W_trans[:, col_trans:col_trans+n_trans] trans[b]  (256 outputs each). */
int tp_tc_image_biases(const float* W_rgb, int64_t ld_rgb, int col_rgb, int n_light, const float* b_rgb, const float* light,
                       const float* W_trans, int64_t ld_trans, int col_trans, int n_trans, const float* b_trans,
                       const float* trans, int B, float* out_rgb, float* out_trans, void* stream);
/* out[r,:] = imgbias[r / rays_per_image] + W[:, col0:col0+3+6L] [u, enc(u)], u = ray[r]/|ray[r]|  (256 outputs; fp32):
 * the view-direction part of mlp_rgb[0] (layers/nerf_static_transient_light.py:104-117), once per ray. */
int tp_tc_ray_bias(const float* ray, int64_t R, int64_t rays_per_image, int L_view, const float* W, int64_t ldw,
                   int col0, const float* imgbias, float* out, void* stream);

/* NeRF.forward_samples of the static/transient/light model (layers/nerf_static_transient_light.py:76-166), bf16
 * operands / fp32 accumulate.  center, ray [rays,3]; depth [S] (S = rays*N); per_image = samples per image.
 * biasbuf: 16 floats {trunk7 b[0], rgb3 b[0:3], trans3 b[0:5], 0...} (the 256-wide stages' biases live in `packed`).
 * Outputs rgb [S,3,2], density [S,2], uncert [S].  save: NULL, or tp_tc_save_bytes(S) bytes receiving, per 128-sample
 * tile, the bf16 tile images [7][32 k8][128 rows][8] of {trunk feature, rgb hidden 1-3, transient hidden 1-3} that the
 * backward consumes (training).  flags: 0 = default; bit 17 (0x20000) = static-only rendering (inference launch only): the
 * stage list stops after the rgb head, so the launch does 78 % of the work; rgb[:, :, 1], density[:, 1] and uncert are written
 * as zeros -- for callers that use only the static outputs (rgb_static / depth / opacity_static of Model.evaluate_full,
 * model/nerf_adapt_st_gan.py:341-362) and for the plain layers/nerf.py model.  Any other flag bit is TP_ERR_BAD_ARG. */
int tp_tc_nerf_stl_forward(const float* center, const float* ray, const float* depth, int64_t S, int N,
                           int64_t per_image, const void* packed, const float* biasbuf, const float* raybias,
                           const float* imgbias, float* rgb, float* density, float* uncert, void* scratch,
                           int64_t scratch_bytes, void* save, int flags, void* stream);
int64_t tp_tc_save_bytes(int64_t S);

/* Graph.render after ray selection (model/nerf_adapt_st_gan.py:565-631: get_center_and_ray + ray_batch_sample, sample_depth,
 * forward_samples, composite) as ONE launch of the fused kernel, for inference (no gradient).  Per ray the kernel reads its
 * pixel index (8 B, optional) and its bounds (8 B) and writes 56 B; no depth, point, bias-table, rgb-sample or uncertainty
 * tensor exists in HBM.
 *   kinv [B,9], pose_inv [B,12]: K^-1 and pose^-1 per view (the reference's own host-side inverses, camera.py:292-314);
 *   ray_idx [B,R] int64 pixel indices (p = y*W + x), or NULL: ray r of every view is pixel ray0 + r (a row block of the frame);
 *   z_near / z_far [B,H*W]: full-frame sample bounds, read at the ray's pixel (Graph.ray_batch_sample, :702-710);
 *   N in {32, 64, 128} samples per ray; depth_mode 0 = injected jitter rand [B,R,N] (the reference's torch.rand draw),
 *   1 = midpoints (sample_stratified false), 2 = in-kernel Philox keyed by seed (same stream as tp_sample_depth mode 2);
 *   packed / biasbuf as for tp_tc_nerf_stl_forward; wview [3+6*L_view,256] = columns 256.. of mlp_rgb[0].weight transposed
 *   (view-direction inputs, layers/nerf_static_transient_light.py:111-117); imgbias_rgb / imgbias_trans [B,256] from
 *   tp_tc_image_biases (per-image latents folded into the layer-0 biases).
 * Outputs (any may be NULL = not materialised): rgb, rgb_static, rgb_transient [B*R,3]; depth, opacity, opacity_static,
 * opacity_transient, uncert [B*R] (uncert includes + min_uncert, layers/..light.py:207); alpha_static, alpha_transient [B*R*N];
 * density [B*R*N,2].  Output pointers may address a peer GPU's memory (NVLink stores: the one-frame multi-GPU gather).
 * flags: bit 17 = static only (transient terms zero).  scratch >= tp_tc_scratch_bytes(). */
int tp_render_fused_forward(const float* kinv, const float* pose_inv, int B, int H, int W, float pix_offset,
                            const int64_t* ray_idx, int64_t R, int64_t ray0, const float* z_near, const float* z_far, int N,
                            int depth_mode, const float* rand, uint64_t seed, const void* packed, const float* biasbuf,
                            const float* wview, int L_view, const float* imgbias_rgb, const float* imgbias_trans,
                            float min_uncert, float* rgb, float* rgb_static, float* rgb_transient, float* depth,
                            float* opacity, float* opacity_static, float* opacity_transient, float* uncert,
                            float* alpha_static, float* alpha_transient, float* density, void* scratch,
                            int64_t scratch_bytes, int flags, void* stream);
/* The same launch over an object-pixel list (tp_mask_ray_list): ray j is slot j of `list` [>= *n_slots], n_slots a DEVICE
 * pointer read by the kernel (one CTA per SM: the host does not know the count; n_slots = 0 is a valid launch).  Rank shard_rank
 * of shard_world renders super-tiles [floor(r*T/w), floor((r+1)*T/w)) of the T = n_slots / (256/N) in the list.  A sample's key
 * is s = q*N + k for entry q: per-ray outputs are stored at row q of [B*HW,C] frame buffers, per-sample ones at s, and
 * depth_mode 0 reads a frame-sized rand [B*HW*N] at s -- the key a full-frame launch (ray_idx NULL, ray0 0, R = HW) gives the same
 * sample, for injected rand and Philox alike, so a list-mode sample is bit-identical to that launch's.  Every other argument,
 * flags bit 17 included, as for tp_render_fused_forward. */
int tp_render_fused_forward_list(const float* kinv, const float* pose_inv, int B, int H, int W, float pix_offset,
                                 const int64_t* list, const int64_t* n_slots, int shard_rank, int shard_world,
                                 const float* z_near, const float* z_far, int N, int depth_mode, const float* rand, uint64_t seed,
                                 const void* packed, const float* biasbuf, const float* wview, int L_view,
                                 const float* imgbias_rgb, const float* imgbias_trans, float min_uncert, float* rgb,
                                 float* rgb_static, float* rgb_transient, float* depth, float* opacity, float* opacity_static,
                                 float* opacity_transient, float* uncert, float* alpha_static, float* alpha_transient,
                                 float* density, void* scratch, int64_t scratch_bytes, int flags, void* stream);
/* ---- fp32-parity mode on the tensor cores (K2 split-bf16, csrc/mlp_tc_split.cu) --------------------------------
 * NeRF.forward_samples (layers/nerf_static_transient_light.py:76-166; layers/nerf.py:61-99 as a padded layer list) with every
 * operand carried as hi + lo bf16 and three tcgen05.mma passes per K step (A_hi W_hi + A_hi W_lo + A_lo W_hi, fp32 accumulate):
 * ~16 mantissa bits per operand, for the <= 1e-4 contract the bf16 kernel cannot meet.  The positional encoding is the
 * reference's fp32 arithmetic (sin / cos of the rounded product x * fl(2^k pi)), biases are added in fp32.
 *   image: n_slots x tp_tc32_slot_bytes() from tp_tc32_pack_weights; slot_desc: DEVICE int64 [n_slots,8] rows {W device
 *   pointer (0 = zeros), ld, row0, rows_valid, col0, cols_valid, kind (256: one K = 16 step of a 256-row layer, hi | lo;
 *   16: an output layer of <= 8 rows over K = 256, hi rows 0..7 / lo rows 8..15), 0} in consumption order;
 *   stages: HOST int32 [n_stages,7] rows {a_steps (0 | 16: K steps read from the activation tile), e_steps (0..4: K steps
 *   read from the encoding tile [xyz, enc(xyz)], taken first), kind (0 hidden 256-wide + ReLU, 1 density: softplus of row 0,
 *   2 rgb: sigmoid of rows 0..2, 3 transient: sigmoid x3, softplus x2), bias kind (0 static: bias + bias_off, 1 per ray:
 *   raybias row, 2 per image: imgbias row), bias_off (floats, multiple of 4), flags (1 = reads the activation tile the previous
 *   hidden stage wrote, 2 = reads the parked trunk feature, 4 = its output is the trunk feature (parked), 8 = last stage that
 *   reads the encoding tile), save slot (-1 = none)}; the list is validated (TP_ERR_BAD_ARG / TP_ERR_BAD_SHAPE) before the launch;
 *   precision 0 = the split mode above; 1 = ONE pass with bf16 operands (image packed with precision 1): the bf16 forward for any
 *   stage list (<= 1e-2; tp_tc_nerf_stl_forward stays the fast path of the yaml's architecture).  With precision 1, `save`
 *   [ceil(S/128)][n_save][64 KB] receives the output of every hidden stage that names a save slot as a bf16 tile image
 *   [32 k8][128 rows][8] -- the operands of the tensor-core backward (tp_tc_chain_backward, tp_tc_dw_gemm) -- and slot enc_slot
 *   (-1 = none) the encoding tile [xyz, enc(xyz), 1, 0...]: dz^T of it = the encoding columns of a layer's dW and its bias sum;
 *   bias: fp32 static biases; raybias [rays,256] from tp_tc_ray_bias, imgbias [images,256] from tp_tc_image_biases.
 * Outputs rgb [S,3,2], density [S,2], uncert [S] as tp_tc_nerf_stl_forward.  scratch >= tp_tc32_scratch_bytes().  Range of the
 * split mode: |weights|, |hidden activations| < 65 504 (fp16 hi part); a violation is reported through the status word. */
int64_t tp_tc32_slot_bytes(void);
int64_t tp_tc32_save_bytes(int64_t S, int n_save);      /* save buffer: [tiles][n_save][64 KB] images + [tiles][n_save][4 KB] ReLU bitmasks */
int64_t tp_tc32_scratch_bytes(void);
int64_t tp_tc32_status_offset(void);      /* byte offset, inside scratch, of a 32-bit status word the caller zeroes once: the split
                                           * mode sets bit 0 when a hidden activation exceeds the fp16 range (> 6e4) or is NaN */
int tp_tc32_max_stages(void);
int tp_tc32_pack_weights(const int64_t* slot_desc, int n_slots, int precision, void* image, void* stream);
int tp_tc32_forward(const float* center, const float* ray, const float* depth, int64_t S, int N, int64_t per_image,
                    const void* image, int n_slots, const int32_t* stages, int n_stages, const float* bias,
                    const float* raybias, const float* imgbias, float* rgb, float* density, float* uncert, void* scratch,
                    int64_t scratch_bytes, int precision, void* save, int n_save, int enc_slot, void* stream);
/* The split-mode forward (precision 0 arithmetic, outputs bit-identical to tp_tc32_forward's) of a <= 1e-4 TRAINING step
 * (autograd of layers/nerf.py:61-99 and layers/nerf_static_transient_light.py:104-137 at fp32 parity): `save` (required, n_save >= 1)
 * [ceil(S/128)][2 n_save][64 KB] receives every save-slot activation, and slot enc_slot the encoding tile [xyz, enc(xyz), 1, 0...],
 * as bf16 hi / lo tile images (slot 2k = bf16(x), 2k + 1 = bf16(x - hi)), then [ceil(S/128)][n_save][4 KB] ReLU bitmasks -- the
 * operands of tp_tc_chain_backward_split and of tp_tc_dw_gemm / tp_tc_images_colsum / tp_tc_thin_dw / tp_tc_image_ray_sums, which
 * address hi and lo as ordinary slots.  bf16 rather than the forward's fp16: the backward's operands need fp32's exponent range.
 * Same stage list, checks, scratch and status word as tp_tc32_forward. */
int64_t tp_tc32_split_save_bytes(int64_t S, int n_save);
/* Graph.render after ray selection as ONE launch of the staged kernel, for inference, in either arithmetic (precision 0 split
 * <= 1e-4, 1 single-pass bf16) and for any stage list tp_tc32_forward takes: what tp_raygen + tp_sample_depth + tp_tc_ray_bias +
 * tp_tc32_forward + tp_composite_{plain,stl}_forward compute (pre-training engine, model/nerf_pretrain.py:588-627 with the plain
 * layers/nerf.py model; adaptation engine, model/nerf_adapt_st_gan.py:565-631), with no per-sample tensor and no bias table in HBM.
 *   kinv, pose_inv, B, H, W, pix_offset, ray_idx / R / ray0, z_near / z_far, N in {32, 64, 128}, depth_mode / rand / seed and
 *   min_uncert as for tp_render_fused_forward (rays and depths have the bits of tp_raygen and tp_sample_depth);
 *   image, n_slots, stages, n_stages, bias, precision as for tp_tc32_forward (no save slot is written); a BIAS_RAY stage's row is
 *   imgbias_rgb[view] + wview^T [u, enc(u)] computed in-kernel with tp_tc_ray_bias's bits: wview [3+6*L_view,256] = the view-encoding
 *   columns of the rgb-0 layer, transposed; imgbias_rgb [B,256] and imgbias [B,256] (BIAS_IMAGE stages; may be NULL without one)
 *   from tp_tc_image_biases or the layer-0 biases of the two heads.
 *   chains 3 (static / transient / light, layers/nerf_static_transient_light.py:168-212): outputs as tp_render_fused_forward's,
 *   density [B*R*N,2]; chains 1 (plain model, single-chain compositing of layers/nerf.py:117-136, no background colour): rgb [B*R,3],
 *   depth and opacity [B*R], density [B*R*N] -- the other outputs must be NULL.  Any output may be NULL and may address a peer
 *   GPU's memory.  scratch >= tp_tc32_render_scratch_bytes(); the fp16-range status word is tp_tc32_forward's (same offset). */
int64_t tp_tc32_render_scratch_bytes(void);
int tp_tc32_render_forward(const float* kinv, const float* pose_inv, int B, int H, int W, float pix_offset, const int64_t* ray_idx,
                           int64_t R, int64_t ray0, const float* z_near, const float* z_far, int N, int depth_mode,
                           const float* rand, uint64_t seed, const void* image, int n_slots, const int32_t* stages, int n_stages,
                           const float* bias, const float* wview, int L_view, const float* imgbias_rgb, const float* imgbias,
                           int chains, float min_uncert, float* rgb, float* rgb_static, float* rgb_transient, float* depth,
                           float* opacity, float* opacity_static, float* opacity_transient, float* uncert,
                           float* alpha_static, float* alpha_transient, float* density, void* scratch,
                           int64_t scratch_bytes, int precision, void* stream);
/* tp_tc32_render_forward over an object-pixel list: list, n_slots, shard_rank, shard_world, frame-sized rand and the frame layout
 * of the outputs as tp_render_fused_forward_list (a shard's tiles are twice its super-tiles); n_weight_slots is tp_tc32_forward's
 * n_slots.  chains must be 3 (static / transient / light); every other argument as for tp_tc32_render_forward. */
int tp_tc32_render_forward_list(const float* kinv, const float* pose_inv, int B, int H, int W, float pix_offset, const int64_t* list,
                                const int64_t* n_slots, int shard_rank, int shard_world, const float* z_near, const float* z_far,
                                int N, int depth_mode, const float* rand, uint64_t seed, const void* image, int n_weight_slots,
                                const int32_t* stages, int n_stages, const float* bias, const float* wview, int L_view,
                                const float* imgbias_rgb, const float* imgbias, int chains, float min_uncert, float* rgb,
                                float* rgb_static, float* rgb_transient, float* depth, float* opacity, float* opacity_static,
                                float* opacity_transient, float* uncert, float* alpha_static, float* alpha_transient,
                                float* density, void* scratch, int64_t scratch_bytes, int precision, void* stream);
int tp_tc32_forward_split_save(const float* center, const float* ray, const float* depth, int64_t S, int N, int64_t per_image,
                               const void* image, int n_slots, const int32_t* stages, int n_stages, const float* bias,
                               const float* raybias, const float* imgbias, float* rgb, float* density, float* uncert, void* scratch,
                               int64_t scratch_bytes, void* save, int n_save, int enc_slot, void* stream);

/* ---- tensor-core backward of the two heads on the saved tile images (K2b, bf16 mode) ------------------------- */

/* out[i] (=/+=) sum_z partial[z*count + i], fixed order (second stage of every split reduction). */
int tp_reduce_partials(const float* partial, int splits, int64_t count, float* out, int accumulate, void* stream);

int tp_tc_bwd_num_chunks(void);              /* chunks of the transposed weight image tp_tc_heads_backward streams (34) */
int64_t tp_tc_dz_bytes(int64_t S);           /* bytes of the dz tile images tp_tc_heads_backward writes: ceil(S/128) x 6 x 64 KB */
int tp_tc_dw_splits(int64_t S, int n_jobs);  /* split partials per job that tp_tc_dw_gemm writes */

/* n_jobs (<= 8) weight-gradient GEMMs in one launch: job j computes dz[a_slots[j]]^T x[b_slots[j]] (256x256 fp32) over all
 * samples (staged backward: dz = images of tp_tc_chain_backward, x = images tp_tc32_forward saved); partial is
 * [splits][n_jobs][256][256] with splits = tp_tc_dw_splits(S, n_jobs).  a_slots/b_slots: HOST arrays.
 * Reduce with tp_reduce_partials(partial, splits, n_jobs*65536, ...). */
int tp_tc_dw_gemm(const void* a_images, int a_nslots, const void* b_images, int b_nslots, const int32_t* a_slots,
                  const int32_t* b_slots, int n_jobs, int64_t S, float* partial, int64_t partial_floats, void* stream);

/* Backward of both heads on the images tp_tc_nerf_stl_forward saved, in five launches: the dX chain kernel also accumulates,
 * on the tensor pipe, every thin gradient -- bias gradients, output-layer weight gradients, the xyz / view-direction columns
 * of mlp_rgb[0], per-image sums for the latent terms -- then two finish kernels and the six 256x256 weight-gradient GEMMs write the reference's parameter gradients (autograd of layers/nerf_static_transient_light.py:104-137
 * under the losses of model/nerf_adapt_st_gan.py:747-763) straight into caller tensors.
 * grads: HOST array of 16 DEVICE pointers {rgb dW0 [256,ld_r0], db0, dW1 [256,256], db1, dW2, db2, dW3 [3,256], db3 [3],
 * transient dW0 [256,ld_t0], db0, dW1, db1, dW2, db2, dW3 [5,256], db3 [5]}.  d_lat_* [B,n] or NULL.  B = images,
 * per_image = samples per image (B*per_image >= S).  Requires tp_tc_heads_backward_supported(S, per_image) (a CTA's contiguous
 * tile range may touch at most 4 images); workspace >= tp_tc_heads_backward_workspace(S, B) floats. */
int tp_tc_heads_backward_supported(int64_t S, int64_t per_image);
int64_t tp_tc_heads_backward_workspace(int64_t S, int B);
int tp_tc_heads_backward(const float* dz_rgb, const float* dz_trans, int64_t S, int N, int64_t per_image, int B,
                         const float* center, const float* ray, const float* depth, int L_view,
                         const void* packed_bwd, const void* saved, void* dz_images, const float* W_r0,
                         int64_t ld_r0, const float* W_t0, int64_t ld_t0, const float* lat_light, int n_light,
                         const float* lat_trans, int n_trans, float* const* grads, float* d_lat_light,
                         float* d_lat_trans, float* workspace, int64_t workspace_floats, void* stream);

/* out[r,:] = sum over the N samples of ray r of an image slot (per-ray column sums, fp32 [ceil(S/N),256]). */
int tp_tc_image_ray_sums(const void* images, int slot, int n_slots, int64_t S, int N, float* out, void* stream);

/* out[c] = sum_s x[s,c] for a thin fp32 matrix [S,C<=8]; workspace >= 2*SMs*C floats. */
int tp_thin_colsum(const float* x, int64_t S, int C, float* out, float* workspace, int64_t workspace_floats, void* stream);

/* partial[blk][m][k] = sum_s thin[s][m] * x[s][k] for a thin fp32 operand [S,M], M in {1,3,5}; x = image slot. */
int tp_tc_thin_dw(const float* thin, int M, const void* images, int slot, int n_slots, int64_t S, float* partial,
                  int64_t partial_floats, int* n_blocks_out, void* stream);

/* ---- fused patch gather + ray-wise losses + backward seeds (SURVEY 8 f2) ---------------------------------------- */

/* Graph.compute_loss(train_step='nerf') ray-wise terms and Model.summarize_loss (model/nerf_adapt_st_gan.py:712-763,
 * model/base.py:145-157) in two launches.  image [B,3,H,W]; obj_mask [B,H,W] raw (>0 = object); coords [B,R,2] in [-1,1]
 * (R = h*w patch rays); rgb [B,R,3], uncert [B,R], density [B*R*N,2] = outputs of the render.  terms: bit 0 render
 * (uncertainty-weighted masked MSE), bit 1 uncert (5 + mean log u^2 / 2), bit 2 trans_reg (mean transient density); w_* =
 * 10^loss_weight.  Writes image_sample [B,3,R] (bilinear, align_corners=True), mask_sample [B,R] (nearest,
 * align_corners=False), losses[4] = {render, uncert, trans_reg, all}, and d(all)/d{rgb, uncert, density} (g_density [B*R*N,2]
 * may be NULL; g_rgb = g_uncert = g_density = NULL computes the scalars only and leaves the seeds to tp_patch_loss_backward).
 * Deterministic (fixed-order reductions).  workspace >= tp_patch_loss_workspace() floats. */
int64_t tp_patch_loss_workspace(void);
int tp_patch_loss(const float* image, const float* obj_mask, const float* coords, int B, int R, int H, int W,
                  const float* rgb, const float* uncert, const float* density, int N, float w_render, float w_uncert,
                  float w_trans_reg, int terms, float* image_sample, float* mask_sample, float* losses, float* g_rgb,
                  float* g_uncert, float* g_density, float* workspace, int64_t workspace_floats, void* stream);
/* Backward of tp_patch_loss for arbitrary upstream gradients g_losses[4] (DEVICE memory: no host sync) of {render, uncert,
 * trans_reg, all} -- autograd of model/nerf_adapt_st_gan.py:747-763 whichever way the caller combines the terms (the reference
 * engine backpropagates the `all` that Model.summarize_loss builds, model/base.py:145-157: g = {10^w_r, 10^w_u, 10^w_t, 0}).
 * image_sample, mask_sample and workspace are the forward call's outputs; same B, R, N, weights and terms. */
int tp_patch_loss_backward(const float* g_losses, const float* image_sample, const float* mask_sample, int B, int R,
                           const float* rgb, const float* uncert, int N, float w_render, float w_uncert, float w_trans_reg,
                           int terms, float* g_rgb, float* g_uncert, float* g_density, const float* workspace,
                           int64_t workspace_floats, void* stream);

/* ---- eval-frame epilogue (SURVEY 8 f3) --------------------------------------------------------------------------- */

/* dX chain of any stack of 256-wide ReLU layers on the tensor cores (csrc/mlp_tc_chain.cu; autograd of layers/nerf.py:61-99 for
 * the plain model, whose trunk trains): per 128-sample tile and stage, dz_out = (dz_in W) * [saved activation > 0], every dz
 * tile stored as a bf16 image for tp_tc_dw_gemm.  thin0 [S,cols0] / thin1 [S,cols1] (<= 8 fp32 columns; thin1 may be NULL):
 * narrow gradients that enter the chain through one K = 16 step (the rgb output layer's dz, the raw-density gradient).
 * packed_bwd: n_chunks x 16 KB transposed weight chunks (tp_tc_pack_weights, transpose flag).  stages: HOST int32 [n_stages,6]
 * rows {thin operand (-1 | 0 | 1), its 8 KB chunk, first K = 32 chunk, number of K = 32 chunks (0 | 8, read against the previous
 * stage's output), mask slot, dz slot written}; the first stage reads only a thin operand, every later one reads the previous output.
 * mask_bits [tiles][n_saved][8 planes][128 rows] uint32 = the ReLU bitmasks tp_tc32_forward (precision 1, save) writes behind its
 * tile images (at byte offset tiles * n_save * 65536 of the save buffer); dz_out [tiles][n_out][64 KB]. */
/* Column sums of tile images over all samples (bias gradients): sel DEVICE int32 [n_sel] slots; partial [blocks][n_sel][256]
 * with blocks = tp_tc_images_colsum_blocks(), reduced by tp_reduce_partials(partial, blocks, n_sel * 256, out).  Rows of the last
 * tile beyond S must be zero (the dz images of tp_tc_chain_backward are). */
int tp_tc_images_colsum_blocks(void);
int tp_tc_images_colsum(const void* images, int n_slots, int64_t S, const int32_t* sel, int n_sel, float* partial,
                        int64_t partial_floats, void* stream);
int tp_tc_chain_max_stages(void);
int tp_tc_chain_backward(const float* thin0, int cols0, const float* thin1, int cols1, int64_t S, const void* packed_bwd,
                         int n_chunks, const int32_t* stages, int n_stages, const void* mask_bits, int n_saved, void* dz_out,
                         int n_out, void* stream);
/* The same dX chain at fp32 parity (K2c, csrc/mlp_tc_chain.cu): dz, the thin operands and the weights carried as bf16 hi + lo,
 * three tcgen05.mma passes per K = 16 step (dz_hi W_hi + dz_hi W_lo + dz_lo W_hi, fp32 accumulate).  packed_bwd: n_chunks x 16 KB
 * K = 16 slots [W^T hi 8 KB | W^T lo 8 KB] from tp_tc_pack_weights_split; stage rows as tp_tc_chain_backward's, except that the
 * number of chunks a stage reads against the previous output is 0 | 16 (K = 16 slots) and the thin operand's chunk is one slot.
 * mask_bits: the bitmasks of tp_tc32_forward_split_save (at byte offset tiles * 2 * n_save * 65536 of its save buffer);
 * dz_out [tiles][2 n_out][64 KB]: stage output slot k is written as hi (image 2k) and lo (image 2k + 1). */
int tp_tc_chain_backward_split(const float* thin0, int cols0, const float* thin1, int cols1, int64_t S, const void* packed_bwd,
                               int n_chunks, const int32_t* stages, int n_stages, const void* mask_bits, int n_saved, void* dz_out,
                               int n_out, void* stream);
/* chunk_desc: DEVICE int64 [n_chunks,10] rows as tp_tc_pack_weights' with n_layout 256 and no bias; each row is ONE K = 16 step
 * (cols_valid <= 16): 8 KB bf16(W) then 8 KB bf16(W - bf16(W)), each [2 k8][256 n][8]. */
int tp_tc_pack_weights_split(const int64_t* chunk_desc, int n_chunks, void* packed, void* stream);

/* ---- K7: mesh depth / NOCS / colour rasteriser (SURVEY 8 f4) --------------------------------------------------------
 * tools/mvrenderer.py:33-178 as compute_surfelinfo.py:114-116 calls it (pytorch3d MeshRasterizer, faces_per_pixel 1, blur 0,
 * perspective-correct barycentrics; vertex-attribute shader; softmax_rgb_blend with sigma = gamma, black background).
 * pytorch3d is absent and unpinned by the reference: its published rules are restated -- parity unpinned (DESIGN.md).
 *   verts [V,3] object space; faces [F,3] int32; attr [V,C] per-vertex attributes (C <= 8: vertex colours, or the NOCS
 *   coordinates of mvrenderer.py:695-722), may be NULL when out is NULL; pose [B,12] = [R | t] rows (OpenCV camera: x right,
 *   y down, z forward), K [B,9] pixel intrinsics.
 * Outputs (any may be NULL): out [B,C,H,W]; depth [B,H,W] = view depth of the nearest face, -1 where none (fragments.zbuf);
 * pix_to_face [B,H,W] int32, -1 where none.  Deterministic (64-bit atomicMin on depth | face index). */
int64_t tp_mesh_render_workspace(int B, int V, int H, int W);
int tp_mesh_render(const float* verts, int V, const int32_t* faces, int F, const float* attr, int C, const float* pose,
                   const float* K, int B, int H, int W, float sigma, float* out, float* depth, int32_t* pix_to_face,
                   void* workspace, int64_t workspace_bytes, void* stream);

/* Latent rows of a training batch (model/nerf_adapt_st_gan.py:589-603): out_a[b,:] = table_a[idx[b],:], out_b likewise -- both
 * embedding tables in one launch; idx DEVICE int64 [B].  The backward writes the dense table gradients: d_table[r,:] = sum of
 * g[b,:] over the b with idx[b] == r, in ascending b (deterministic); untouched rows are zero. */
int tp_latent_rows(const float* table_a, int cols_a, const float* table_b, int cols_b, const int64_t* idx, int B,
                   float* out_a, float* out_b, void* stream);
int tp_latent_rows_backward(const float* g_a, int cols_a, int64_t rows_a, const float* g_b, int cols_b, int64_t rows_b,
                            const int64_t* idx, int B, float* d_table_a, float* d_table_b, void* stream);

/* Model.evaluate_full per frame (model/nerf_adapt_st_gan.py:341-362) for B views at once, no host sync: rgb [B,HW,3]
 * (rgb_static of the render) -> rgb_map [B,3,HW]; depth [B,HW] -> depth_map = depth / depth_scale; image [B,3,HW] * mask
 * [B,HW] -> image_masked; mse[b] = mean((rgb_map - image_masked)^2), psnr[b] = -10 log10(mse[b]) stay on the device.
 * workspace >= tp_eval_epilogue_workspace(B) floats. */
int64_t tp_eval_epilogue_workspace(int B);
int tp_eval_epilogue(const float* rgb, const float* depth, const float* image, const float* mask, int B, int64_t HW,
                     float depth_scale, float* rgb_map, float* depth_map, float* image_masked, float* mse, float* psnr,
                     float* workspace, int64_t workspace_floats, void* stream);

/* ---- gradient exchange over NVLink peer memory (SURVEY 8e) ------------------------------------------------------- */

/* The one exchange of the path: mean over the ranks of the flat fp32 gradient bucket (heads + latent embeddings, ~1.7 MB;
 * the reference is single-GPU, options.py:112, so this replaces what DistributedDataParallel's bucket allreduce would do).
 * One kernel over CUDA-IPC peer windows instead of a library allreduce: publish "my gradients of step `epoch` are in place"
 * into every peer's window header (NVLink stores), wait on the local header, read all `world` buffers (peer loads) and add
 * them in rank order -> bit-identical result on every rank.
 * Window layout: [1 KB header | data buffer 0 | data buffer 1], each buffer tp_peer_capacity_bytes(n) long; the caller
 * writes its gradients into buffer (epoch & 1) of its OWN window (offset tp_peer_data_offset) before the call; epochs count
 * 1, 2, 3, ... identically on every rank.
 * The window is the only driver object the library creates (set-up time, host calls): create = cudaMalloc + zero,
 * export/import = the 64-byte CUDA IPC handle a peer process opens, release/destroy undo them.
 * windows: HOST array of `world` device pointers (windows[rank] = the local window, the others imported, same order on
 * every rank; a single process may pass windows of one device to exercise the protocol).  out: local, >= n rounded up to
 * 4 floats, 16-byte aligned.  grid_ctas 0 = default.  A peer that does not arrive within timeout_ms (0 = 10 s) makes
 * the kernel fill `out` with NaN (stale or partial gradients can never pass for a result) and store `epoch` in the window's
 * status word (tp_peer_status: host call, synchronising copy, 0 = healthy). */
int64_t tp_peer_capacity_bytes(int64_t n_floats);
int64_t tp_peer_window_bytes(int64_t n_floats);
int64_t tp_peer_data_offset(int64_t n_floats, int parity);
int tp_peer_window_create(int64_t bytes, void** window_out);
int tp_peer_window_destroy(void* window);
int tp_peer_window_export(const void* window, void* handle64);
int tp_peer_window_import(const void* handle64, void** window_out);
int tp_peer_window_release(void* imported_window);
int tp_peer_allreduce_mean(void* const* windows, int world, int rank, int64_t n_floats, uint32_t epoch, float* out,
                           int grid_ctas, int64_t timeout_ms, void* stream);
int tp_peer_status(const void* window, uint32_t* status_host);

/* The same exchange with a device-held epoch, so that it can be captured in a CUDA graph (a capture freezes the host epoch
 * argument of tp_peer_allreduce_mean and the host-chosen buffer of the pack).  Together the two calls replace "write buffer
 * (epoch & 1), then tp_peer_allreduce_mean(epoch)":
 *   tp_peer_stage copies src[0:n] into data buffer (e+1)&1 of the LOCAL window, e = the window's device epoch (header byte
 *   768, 0 after create), and advances the device epoch to e+1 (16-byte vectors, local HBM only, never waits);
 *   tp_peer_allreduce_mean_dev is tp_peer_allreduce_mean with `epoch` read from the local window's device epoch: publish,
 *   bounded wait, rank-order sum / world -> out, NaN in `out` + the failed epoch in the status word on a timeout.
 * Caller: one tp_peer_stage, then one tp_peer_allreduce_mean_dev, per exchange, on one stream, and the same number of
 * exchanges on every rank (eager calls and graph replays count alike: they advance one counter); a window is driven either
 * by this pair or by tp_peer_allreduce_mean with host epochs, never both.  src: local, 16-byte aligned, >= n floats.
 * n_floats must be the n the window was sized for (tp_peer_window_bytes(n)): it places data buffer 1, and the stage writes
 * there without a bounds check.
 * Arguments as above; TP_ERR_BAD_ARG for null pointers, n < 0 or a rank outside the world, TP_ERR_ALIGN for a window that is
 * not 256-byte aligned or an `src` / `out` that is not 16-byte aligned. */
int tp_peer_stage(void* window, int64_t n_floats, const float* src, void* stream);
int tp_peer_allreduce_mean_dev(void* const* windows, int world, int rank, int64_t n_floats, float* out, int grid_ctas,
                               int64_t timeout_ms, void* stream);

/* Completion barrier over the same windows (no data): rank publishes `epoch` (1, 2, ...) to every peer's header and waits
 * for every peer's.  Stream-ordered after a tp_render_fused_forward launch whose output pointers address the root rank's
 * window, it makes that rank's row block of the frame visible to the root (one-frame multi-GPU render, SURVEY 8e: "row
 * blocks of HW ... gather of 56 B/ray").  A peer that never arrives sets the status word after timeout_ms (default 10 s). */
int tp_peer_barrier(void* const* windows, int world, int rank, uint32_t epoch, int64_t timeout_ms, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* TEXPOSE_B200_H_ */
