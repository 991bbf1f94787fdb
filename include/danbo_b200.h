/* danbo_b200.h -- C ABI of libdanbo_b200.so: the B200 (sm_100a) kernels of DANBO's per-sample body-field hot path.
 *
 * The reference (LemonATsu/DANBO-pytorch) has no FFI layer: its seam is the Python class RayCaster/GraphCaster
 * (core/raycasters.py:205-716).  These entry points are what a binding for that path calls; each one names the
 * reference code it replaces.  Conventions:
 *   - every pointer is a DEVICE pointer (fp32 unless stated) owned by the caller; nothing is allocated here
 *   - `stream` is a cudaStream_t passed as void*; entries only enqueue work and never synchronise
 *   - return 0 on success, < 0 for invalid arguments, > 0 = cudaError_t of a failed launch
 *   - re-entrant, no global mutable state
 *   - rays: row-major (n_rays, ray_stride >= 8) = [o(3), d(3), near, far, ...]      (raycasters.py:302-306)
 *   - poses: ray n uses pose min(n / rays_per_pose, n_poses-1); pose_skts is (n_poses,24,4,4) world->bone
 *   - sample ids: id = ray*S + s; the extra id n_rays*S + ray is the ray's "sample that no bone sees"
 */
#ifndef DANBO_B200_H
#define DANBO_B200_H

#ifdef __cplusplus
extern "C" {
#endif

/* ABI version of this header (bumped on any change of a signature or of a pointer-array contract): 5. */
int danbo_version(void);

/* NF1 + NF2.  get_near_far_in_cylinder (core/utils/ray_utils.py:294-346) followed, when use_box != 0, by
 * GraphCaster.get_near_far / get_ray_box_intersections (core/raycasters.py:648-707, ray_utils.py:383-417):
 * fp64 plane hits, a box counts only with exactly two hits inside +-(bound+1e-4) (bound_hi = fp32(bound+1e-4)).
 * Rays that miss the cylinder take the nanmean of their segment of seg_len rays (the reference's chunk).
 * seg_acc: workspace of 4*n_seg doubles.  p_valid/v_valid (n_rays,24) bytes are optional (may be NULL). */
int danbo_nearfar(const float* rays, int ray_stride, int n_rays, const float* pose_cyl, int cyl_stride,
                  const float* pose_skts, int rays_per_pose, int n_poses, const float* align, const float* axis_scale,
                  int seg_len, int use_box, float bound, float bound_hi, float* near_out, float* far_out,
                  double* seg_acc, int n_seg, unsigned char* p_valid, unsigned char* v_valid, void* stream);

/* consts[11] = { align (24,4,4), axis_scale (24,3), prob_linears.layers.0.lin.weight (24,15,32),
 *               .layers.0.adj_w (24,24), .layers.0.adj (24,24), .layers.0.bias (32), .layers.1.weight (24,32,32),
 *               .layers.1.bias (24,32), .layers.2.weight (24,32), .layers.2.bias (24),
 *               agg_frags or NULL }  (device pointers).
 * consts[10] is read by danbo_field_agg only: NULL selects the fp32 FFMA aggregation-net kernel (the one every
 * published number was measured with); a table filled by danbo_pack_agg_frags selects the split-bf16 mma.sync kernel
 * (csrc/field_mma.cu; logits within 3e-6 of scale; NOT yet run on hardware). */

/* Tuning knob of the tensor-core aggregation net (pair_logits_mma_kernel): resident blocks per SM its register
 * allocation is bounded for (3: 137 registers, 4: 128, 5: 96 with 20 bytes of spill).  Returns the previous value. */
int danbo_pair_logits_set_blocks(int blocks);

/* Bytes of the fragment table, and the packing of prob_linears' layer-0 / layer-1 weights (consts[2], consts[6]) into
 * split-bf16 m16n8k16 B fragments for the tensor-core aggregation net (MixGNN, gnn_backbone.py:225-274,567-629).
 * Re-run after every update of those weights. */
int danbo_agg_frag_bytes(void);
int danbo_pack_agg_frags(const float* const* consts, void* frags, void* stream);

/* SM1 + T1/T2 + bone-visibility mask + compaction.
 * sample_from_lineseg (ray_utils.py:206-253), transform_batch_pts (core/encoders.py:288-303), bone align
 * (encoders.py:442-444), x/|axis_scale| and invalid = any(|x|>1) (core/networks/gnn_backbone.py:802-808).
 * Coarse mode (z_in NULL): z = near(1-t)+far t with t_vals = linspace(0,1,S) (+ jitter t_rand (n,S) or NULL) -> z_out;
 * lindisp != 0 samples linearly in inverse depth instead, z = 1/(1/near (1-t) + 1/far t) (ray_utils.py:226-227).
 * Fine mode: z_in (n,S) given.  mask_out (n,S) gets bit j set when bone j sees the sample; ids of samples with a
 * non-zero mask (and, with append_empty, one extra id per ray) are appended to active_ids at *active_count. */
int danbo_sample_mask(const float* rays, int ray_stride, int n_rays, int S, const float* near, const float* far,
                      const float* t_vals, const float* t_rand, const float* z_in, float* z_out,
                      const float* pose_skts, int rays_per_pose, int n_poses, const float* const* consts,
                      unsigned int* mask_out, int* active_ids, int* active_count, int capacity, int append_empty,
                      int lindisp, void* stream);

/* G1/G2 + A1-A3 + positional encoding for the active entries.
 * FactorizeGNN.sample_from_volume / factorize_grid_sample (gnn_backbone.py:787-828, core/networks/misc.py:331-351),
 * forward_blend -> MixGNN (core/networks/danbo.py:201-216, gnn_backbone.py:567-629), sigmoid blend weights
 * (danbo.py:406-415), blend (danbo.py:299-300), Embedder (core/cutoff_embedder.py:62-73).
 * pose_vol (n_poses,24,240) = graph-net output.  Four launches: bucket the (row, visible bone) pairs by bone (count,
 * scatter), evaluate the aggregation net per pair, then blend + encode per row.  Writes bf16 rows into xtiles
 * ((capacity+127)/128 tiles of 64 KB, swizzled MMA operand image), row_ray[row], the blend logits ("confd") of every
 * visible (sample, bone) into logits (n_rays*S,24) and optionally hbar (rows,16) and x_rows (rows,208 bf16, a
 * row-major copy of the encoded rows for the backward pass).
 * work: int workspace of 64 + pair_capacity entries; pair_capacity >= number of visible pairs + 24*32 (worst case
 * 24 * rows + 24*32).  If there are more visible pairs than that, work[48] is set to 1 and EVERY row of the call is
 * written as NaN (never a silently wrong value); the caller re-runs with a larger workspace.
 * agg_mode 0: sigmoid blend weights (danbo.py:406-415, every shipped config).  agg_mode 1: agg_type = softmax with
 * mask_vol_prob (danbo.py:388-404); its max runs over all 24 logits, so every bone of an active row is evaluated
 * (pair_capacity >= 24 * rows + 24*32) and logits holds all 24 entries of those rows. */
int danbo_field_agg(const float* rays, int ray_stride, int n_rays, int S, const float* z, const unsigned int* mask,
                    const int* active_ids, const int* active_count, int capacity, const float* pose_skts,
                    const float* pose_vol, int rays_per_pose, int n_poses, const float* const* consts, void* xtiles,
                    int* row_ray, float* logits, float* hbar_out, void* x_rows, int* work, int pair_capacity,
                    int num_sms, int agg_mode, void* stream);

/* Whether danbo_pack_mlp_weights also computes the empty-sample constants behind the heads (default 1).  A training
 * iteration repacks every step and never reads them (danbo_mlp_empty_rows is an eval-path call): switch them off for
 * those packs.  Returns the previous setting. */
int danbo_mlp_set_pack_empty(int enable);

/* Output of the field for a sample NO bone sees (blended feature 0 -> MLP input PE(0), danbo.py:299-302 + nerf.py:176-209):
 * the density trunk and the feature part of the view layer are constants of the weights (danbo_pack_mlp_weights leaves
 * them behind the heads), so per ray only rgb = W_rgb . relu(c + ray_bias) + b_rgb remains.  raw_tail (n_rays,4) =
 * [rgb, sigma0]: the compositing kernels read it for every sample whose visibility mask is 0.  heads = the buffer
 * danbo_pack_mlp_weights filled; ray_bias = danbo_ray_bias's output. */
int danbo_mlp_empty_rows(const float* ray_bias, int n_rays, const float* heads, float* raw_tail, int num_sms, void* stream);

/* V1 folded into the view layer: out (n_rays,128) = W_v[:,256:411] . [PE(rays_d) ; frame code] + b_v
 * (core/networks/nerf.py:252-279, core/networks/embedding.py:86-108).  codes is (n_codes+1,128) with the mean code in
 * the last row (used for cam_idx < 0); wv_ray comes from danbo_pack_mlp_weights; table = (n_codes+1,128) floats of
 * workspace (receives the per-code part, which is shared by all rays of a camera). */
int danbo_ray_bias(const float* rays, int ray_stride, int n_rays, const int* cam_idx, const float* codes, int n_codes,
                   const float* wv_ray, float* table, float* out, void* stream);

/* Sizes of the packed-weight buffers below. */
int danbo_mlp_workspace_bytes(long long* wstream_bytes, long long* heads_bytes, long long* raybias_bytes);

/* fp32 nn.Linear weights -> bf16 tiled + swizzled stage stream (written twice: 84 x 16 KB in single-CTA order, then the
 * same tiles regrouped per CTA of a pair so that one bulk copy stages two half-stages), fp32 head vector and the
 * transposed per-ray slice of views_linears.0.  Re-run after every optimizer step.  w_pts / b_pts are HOST arrays of 8 device pointers. */
int danbo_pack_mlp_weights(const float* const* w_pts, const float* const* b_pts, const float* w_alpha,
                           const float* b_alpha, const float* w_feat, const float* b_feat, const float* w_view,
                           const float* b_view, const float* w_rgb, const float* b_rgb, void* wstream, float* heads,
                           float* wv_ray, void* stream);

/* M1: the 8x256 density MLP + feature/view/rgb heads (core/networks/nerf.py:164-209) as one persistent tcgen05
 * kernel over 128-row tiles.  Row r of the tiles is written to out[row_sample[r]] (float4 rgb,sigma; or one float
 * sigma when density_only, nerf.py:136-154).  *n_rows_dev rows are valid (device scalar, e.g. the active counter). */
int danbo_mlp_forward(const void* xtiles, const void* wstream, const float* heads, const float* ray_bias,
                      const int* row_sample, const int* row_ray, const int* n_rows_dev, int max_rows, float* out,
                      int out_capacity, int density_only, int num_sms, void* stream);

/* Profiling aid: the same launch as danbo_mlp_forward; CTA 0 also writes a clock64 timeline of its first 4 tiles to
 * trace[4][2 roles: MMA issuer, epilogue][20 (layer, half)][begin, end] (320 long long) followed by
 * [4][20][tmem loads landed, stores issued] of one epilogue warp (160 long long): 480 in total. */
int danbo_mlp_forward_trace(const void* xtiles, const void* wstream, const float* heads, const float* ray_bias,
                            const int* row_sample, const int* row_ray, const int* n_rows_dev, int max_rows, float* out,
                            int out_capacity, int density_only, int num_sms, long long* trace, void* stream);

/* Selects the kernel variant behind danbo_mlp_forward*: 1 (default) = CTA pairs (clusters of 2, tcgen05 cta_group::2,
 * each CTA stages half of every weight stage), 0 = one CTA per 128-row tile.  Same results bit for bit (the MMA
 * accumulation order does not change).  Returns the previous setting. */
int danbo_mlp_set_cta_pair(int enable);

/* C1 + R1: raw2outputs (nerf.py:281-347) on the coarse samples, then isample_from_lineseg / sample_pdf
 * (ray_utils.py:159-203,257-291) and the sorted merge order.  raw is (n_rays*S + n_rays,4); samples whose mask is 0
 * read the ray's empty entry.  noise (n,S) already scaled, or NULL.  u_vals = linspace(0,1,S_f) (eval) or u_rand
 * (n,S_f) (train).  order (n,S+S_f) int32 = sorted_idxs.  smooth_weights 1: the single_net importance weights
 * (is_only: 0.5 (max(w_k-1, w_k) + max(w_k, w_k+1)) + 0.01); 0: the interior weights themselves (separate fine network,
 * raycasters.py:348).  S_f = 0 composites only.  weights may be NULL: the (n,S) weight row is then not written. */
int danbo_composite_resample(const float* rays, int ray_stride, int n_rays, int S, int S_f, const float* raw,
                             const unsigned int* mask, const float* z, const float* noise, float inv_B,
                             const float* u_vals, const float* u_rand, float* weights, float* alpha, float* rgb0,
                             float* disp0, float* acc0, float* z_samples, float* z_all, int* order, int* inds,
                             int smooth_weights, void* stream);

/* R2 + C1: merge coarse and fine raw by `order` (core/raycasters.py:484-514,745-761) and composite the merged ray.
 * Optional training outputs: merged raw, confd and part_invalid (raycasters.py:710-716). */
int danbo_merge_composite(const float* rays, int ray_stride, int n_rays, int S_c, int S_f, const float* raw0,
                          const unsigned int* mask0, const float* raw1, const unsigned int* mask1, const float* z_all,
                          const int* order, const float* noise, float inv_B, float* weights, float* alpha, float* rgb,
                          float* disp, float* acc, float* raw_merged, const float* confd0, const float* confd1,
                          float* confd_merged, float* invalid_merged, void* stream);

/* Eval-mode R2 + C1 with the body-part map: the composite of danbo_merge_composite (rgb, disp, acc, weights, alpha and
 * raw_merged bit-identical to it) plus part_map (n,24) = sum_m w_m p_m over the merged samples, with p_m the
 * aggregation weights get_agg(confd_m, 1 - visible_m) of the sample (agg_mode 0 sigmoid, 1 masked softmax, as in
 * danbo_field_agg) and 0 for a sample no bone sees.  confd0 / confd1: danbo_field_agg's logits of the two passes;
 * weights, confd0, confd1 and part_map are required. */
int danbo_merge_composite_parts(const float* rays, int ray_stride, int n_rays, int S_c, int S_f, const float* raw0,
                                const unsigned int* mask0, const float* raw1, const unsigned int* mask1,
                                const float* z_all, const int* order, const float* noise, float inv_B, float* weights,
                                float* alpha, float* rgb, float* disp, float* acc, float* raw_merged,
                                const float* confd0, const float* confd1, int agg_mode, float* part_map, void* stream);

/* ---- backward (train mode; autograd of the same rows as reached from core/trainer.py:563-576) -------------------- */

/* Train-mode M1 forward: danbo_mlp_forward plus the bf16 activations the backward needs: act_save [9][save_cap][256]
 * (pts_linears.0..7 after relu, feature_linear), g_save [save_cap][128] (relu(views_linears.0)). */
int danbo_mlp_forward_save(const void* xtiles, const void* wstream, const float* heads, const float* ray_bias,
                           const int* row_sample, const int* row_ray, const int* n_rows_dev, int max_rows, float* out,
                           int out_capacity, int num_sms, void* act_save, void* g_save, int save_cap, void* stream);

/* Backward of C1 on the coarse samples (nerf.py:297-347): d raw (n*S + n, 4) += from d rgb0 (n,3), d acc0 (n). */
int danbo_composite_bwd(const float* rays, int ray_stride, int n_rays, int S, const float* raw, const unsigned int* mask,
                        const float* z, const float* noise, float inv_B, const float* g_rgb, const float* g_acc,
                        float* d_raw, void* stream);

/* Backward of R2 + C1 on the merged samples; also routes d confd (n,S_t,24) to the per-pass logit buffers. */
int danbo_merge_composite_bwd(const float* rays, int ray_stride, int n_rays, int S_c, int S_f, const float* raw0,
                              const unsigned int* mask0, const float* raw1, const unsigned int* mask1,
                              const float* z_all, const int* order, const float* noise, float inv_B, const float* g_rgb,
                              const float* g_acc, const float* g_confd, float* d_raw0, float* d_raw1, float* d_logit0,
                              float* d_logit1, void* stream);

/* M1 backward building blocks (fp32).  rows_dev = device scalar row count.
 * head_bwd : d raw -> delta of views_linears.0 (rows,128), d a7 (rows,256) and the rgb/alpha head + ray-bias grads;
 *            delta9, d_a7 and d_ray_bias may each be NULL (not formed); the four head gradients are all given or all
 *            NULL (not formed: pose-only backward); nothing asked for launches nothing
 * gemm_dgrad: D[rows x N] = A[rows x K] . B[K x N] (+ D) (* [mask > 0]);  gemm_wgrad: dW[M x N] += A^T . B;
 * colsum: db[N] += sum_rows A. */
int danbo_mlp_head_bwd(const float* d_raw, const int* row_sample, const int* row_ray, const int* rows_dev, int max_rows,
                       const void* g_save, const void* a7_save, const float* w_rgb, const float* w_alpha, float* delta9,
                       float* d_a7, float* d_w_rgb, float* d_b_rgb, float* d_w_alpha, float* d_b_alpha,
                       float* d_ray_bias, int num_sms, void* stream);
int danbo_gemm_dgrad(const void* A, int a_is_bf16, int lda, const float* B, int ldb, float* D, int ldd,
                     const int* rows_dev, int max_rows, int N, int K, int accumulate, const void* mask, int ldmask,
                     void* stream);
int danbo_gemm_wgrad(const float* A, int lda, const void* B, int b_is_bf16, int ldb, float* dW, int ldw,
                     const int* rows_dev, int max_rows, int M, int N, void* stream);
int danbo_colsum(const float* A, int lda, float* db, const int* rows_dev, int max_rows, int N, void* stream);

/* Tensor-core (tcgen05) M1 backward.  danbo_mlp_bwd_workspace: sizes for a row capacity; danbo_pack_mlp_dgrad: transposed
 * bf16 weight tiles (once per iteration); danbo_mlp_dgrad: fused data-gradient chain (deltas of every layer saved as
 * bf16 planes [10][cap][256]: 0 = views_linears.0, 1 = d feature, 2..9 = pts_linears.7..0; dX (cap,208) fp32; with
 * delta_t != NULL the planes are also written row-transposed (the deltaT workspace: operand images of the K = rows GEMMs),
 * and danbo_mlp_wgrad is told so with delta_t_ready = 1 and skips that transpose pass; delta_save = NULL, with delta_t
 * NULL too, selects the variant that writes dX only, for a backward that forms no weight gradient);
 * danbo_mlp_wgrad: dW = delta^T . act (K = rows) for dw[10] = { views_linears.0.weight, feature_linear.weight,
 * pts_linears.7, .6, .5, .4, .3, .2, .1, .0 } and db[9] = { feature_linear.bias, pts_linears.7..0 bias }, accumulated. */
int danbo_mlp_bwd_workspace(int cap, long long* wstream_bytes, long long* delta_bytes, long long* deltaT_bytes,
                            long long* actT_bytes, long long* partial_bytes, int* n_splits);
int danbo_pack_mlp_dgrad(const float* const* w_pts, const float* w_feat, const float* w_view, void* wstream, void* stream);
int danbo_mlp_dgrad(const void* wstream_t, const float* w_rgb, const float* w_alpha, const float* d_raw,
                    const int* row_sample, const int* rows_dev, int max_rows, const void* act_save, const void* g_save,
                    int cap, void* delta_save, void* delta_t, float* dX, int num_sms, void* stream);
int danbo_mlp_wgrad(const void* act_save, const void* x_rows, const void* delta_save, int cap, const int* rows_dev,
                    int max_rows, void* deltaT, int delta_t_ready, void* actT, float* partial, float* const* dw,
                    float* const* db, void* stream);

/* V1 backward: d ray_bias (n,128) -> grads of views_linears.0.weight[:,256:411] (written into the (128,411) layout),
 * its bias and the frame codes (core/networks/nerf.py:252-279, embedding.py:86-108). */
int danbo_ray_bias_bwd(const float* rays, int ray_stride, int n_rays, const int* cam_idx, const float* codes, int n_codes,
                       const float* w_view, const float* d_ray_bias, float* d_w_view, float* d_b_view, float* d_codes,
                       void* stream);

/* V1 backward to the root rotation under root-local view directions (perfcap configs: ray_tr_type=root_local,
 * view_type=relray; pose refinement, --opt_pose): autograd of RootLocalEncoder (core/encoders.py:570-578) and
 * VecNormEncoder (:774-795), i.e. of dn = normalize(skts[pose, 0, :3, :3] . rays_d) and its 4-octave encoding, which
 * danbo_ray_bias multiplies by W_v[:, 256:283], with respect to skts.  Ray n belongs to pose min(n / rays_per_pose,
 * n_poses - 1).  w_view (128,411) fp32 and d_ray_bias (n_rays,128) fp32 row-major (16-byte aligned).  d_skts
 * (n_poses,24,4,4) fp32 is added to (zero it first); only rows 0-2, columns 0-2 of joint 0 receive anything. */
int danbo_view_root_bwd(const float* rays, int ray_stride, int n_rays, const float* pose_skts, int rays_per_pose,
                        int n_poses, const float* w_view, const float* d_ray_bias, float* d_skts, void* stream);

/* G1/G2 + A1-A3 + PE backward (danbo.py:261-302, gnn_backbone.py:787-828, misc.py:331-351): d X (rows,208) and the
 * extra logit gradient -> grads[10] = { w0, adj_w, b0, w1, b1, w2, b2 of prob_linears, d vol (n_poses,24,240),
 * d axis_scale (24,3), d skts (n_poses,24,4,4) or NULL } (fp32, accumulated).  d skts is the gradient with respect to
 * the world-to-bone matrices (what the pose layer, core/pose_opt.py:264-339, receives under --opt_pose; rows 0-2 only,
 * the homogeneous row gets none); NULL when the poses are constants.  grads[0..6] and grads[8] all NULL (all or none)
 * select the pose-only variant: no aggregation-net or axis-scale gradient, d vol and d skts as before.  work = the
 * workspace the forward danbo_field_agg filled; agg_mode as in that call. */
int danbo_field_agg_bwd(const float* rays, int ray_stride, int n_rays, int S, const float* z, const unsigned int* mask,
                        const int* active_ids, const int* active_count, int capacity, const float* pose_skts,
                        const float* pose_vol, int rays_per_pose, int n_poses, const float* const* consts,
                        const float* logits, const float* hbar, const float* dX, const float* g_logit_ext, float* d_hbar,
                        float* d_logit, const int* work, int pair_capacity, float* const* grads, int num_sms,
                        int agg_mode, void* stream);

/* The gradient of the field with respect to the sample positions p = o + z d (surface normals: seed d raw with
 * (0,0,0,1) on every row and the rows' own gradients come out of one pass).  Arguments as danbo_field_agg_bwd, with
 * three accumulators (fp32, added to) in place of grads: d_pts (n_rays*S, 3), required; d_vol (n_poses,24,240) and
 * d_skts (n_poses,24,4,4), each optional (NULL: not formed).  No aggregation-net or axis-scale gradient.  Unlike
 * danbo_field_agg_bwd, the derivative of the feature window exp(-2 sum x^6) is included (the true gradient; training
 * detaches the window), in d_pts and d_skts alike.  2 launches. */
int danbo_field_agg_bwd_pts(const float* rays, int ray_stride, int n_rays, int S, const float* z, const unsigned int* mask,
                            const int* active_ids, const int* active_count, int capacity, const float* pose_skts,
                            const float* pose_vol, int rays_per_pose, int n_poses, const float* const* consts,
                            const float* logits, const float* hbar, const float* dX, const float* g_logit_ext,
                            float* d_hbar, float* d_logit, const int* work, int pair_capacity, float* d_pts,
                            float* d_vol, float* d_skts, int num_sms, int agg_mode, void* stream);

/* GN1 + GN2: the per-pose skeleton graph net, pose_bones (n_poses,24,3) axis-angle -> vol_out (n_poses,24,240) bone
 * feature lines (encode_graph_inputs core/encoders.py:460-473,859-877; BodyGNN.forward on FactorizeGNN
 * core/networks/gnn_backbone.py:683-704,225-274; ParallelLinear core/networks/misc.py:174-183; incl. the doubled layer-0
 * output, SURVEY F3).  params[12] = graph_net.layers.{0.lin.weight (24,66,128), 0.adj_w (24,24), 0.adj (24,24), 0.bias
 * (128), 1.lin.weight (24,128,128), 1.adj_w, 1.adj, 1.bias, 2.weight (24,128,128), 2.bias (24,128), 3.weight (24,128,240),
 * 3.bias (24,240)}.  saved[6] = { graph inputs (n_poses,24,66), lin0, n1, lin1, n2, n3 (each n_poses,24,128) }: written by
 * the forward call, read by the backward call.  4 launches each way. */
int danbo_graph_net_fwd(const float* pose_bones, int n_poses, const float* const* params, float* const* saved,
                        float* vol_out, void* stream);

/* grads[10] = d { 0.lin.weight, 0.adj_w, 0.bias, 1.lin.weight, 1.adj_w, 1.bias, 2.weight, 2.bias, 3.weight, 3.bias } (fp32,
 * added to); d_vol (n_poses,24,240); work = 2 * n_poses*24*128 floats.  grads = NULL: the pose-only variant (3 launches,
 * the transposed products only), which leaves in work what danbo_graph_net_bwd_pose reads. */
int danbo_graph_net_bwd(int n_poses, const float* const* params, float* const* saved, const float* d_vol,
                        float* const* grads, float* work, void* stream);

/* d pose from the graph net (encode_graph_inputs core/encoders.py:460-473, AxisAngtoRot6DEncoder :859-877, Embedder
 * core/cutoff_embedder.py:62-73, mask_root gnn_backbone.py:669-670): after danbo_graph_net_bwd, with the same params,
 * saved and work, d_pose_bones (n_poses,24,3) = d loss / d pose_bones through the layer-0 input (written; the root's row
 * is zero).  pose_bones is the axis-angle the forward call read. */
int danbo_graph_net_bwd_pose(const float* pose_bones, int n_poses, const float* const* params, float* const* saved,
                             const float* work, float* d_pose_bones, void* stream);

/* Pose layer (PoseOptLayer.calculate_kinematic core/pose_opt.py:210-224,264-339; axis_angle_to_matrix
 * core/utils/skeleton_utils.py:411-418) for n_poses poses, pose g being frame idx[g * idx_stride] (int64).  Parameters:
 * pelvis (F,3) and bones (F,24,3) axis-angle, or with the multi-view split root_bones (F,3), bones (U,23,3) and kp_map
 * (F, int64; both NULL otherwise).  rest_pose (n_rest,24,3); with n_rest > 1 frame f uses row rest_idx[f] (int64).
 * Writes kps (n_poses,24,3), the gathered axis-angle bones_out (n_poses,24,3) and skts (n_poses,24,4,4) = the rigid
 * inverse of the local-to-world matrices.  stats (or NULL) = { kp_loss, MPJPC } (Trainer._compute_kp_loss
 * core/trainer.py:446-505 without the temporal term: coef * mean over poses and joints 1..23 of
 * sum_c max((anchor_bones - bones)^2 - tol, 0), and the mean |anchor_kps - kps| / ext_scale), anchors (F,24,3). */
int danbo_pose_fwd(const float* pelvis, const float* bones, const float* root_bones, const long long* kp_map,
                   const float* rest_pose, int n_rest, const long long* rest_idx, const long long* idx, int idx_stride,
                   int n_poses, const float* anchor_kps, const float* anchor_bones, float tol, float coef,
                   float ext_scale, float* kps, float* bones_out, float* skts, float* stats, void* stream);

/* Backward of danbo_pose_fwd (same layer arguments): d_skts (n_poses,24,4,4; the homogeneous row is ignored), d_bones
 * (n_poses,24,3) or NULL, d_kps (n_poses,24,3) or NULL, and, when d_reg (a device scalar, d loss / d kp_loss) is not
 * NULL, the regulariser's gradient with anchor_bones, tol and coef.  ADDS (atomics) into g_pelvis (F,3) and g_bones
 * (F,24,3), or g_root_bones (F,3) and g_bones (U,23,3) with the multi-view split. */
int danbo_pose_bwd(const float* pelvis, const float* bones, const float* root_bones, const long long* kp_map,
                   const float* rest_pose, int n_rest, const long long* rest_idx, const long long* idx, int idx_stride,
                   int n_poses, const float* d_skts, const float* d_bones, const float* d_kps,
                   const float* anchor_bones, const float* d_reg, float tol, float coef, float* g_pelvis,
                   float* g_bones, float* g_root_bones, void* stream);

/* 2D keypoint reprojection term of the pose layer's joints.  kps (n_poses,24,3) as danbo_pose_fwd wrote them (world
 * frame), kp2d (n_poses,24,3) = detections (pixel u, pixel v, confidence c >= 0) in SMPL joint order, proj
 * (n_poses,3,4) one projection matrix per pose.  Per joint (u, v) = (P0 X, P1 X) / w with X = [kps, 1], w = P2 X, and
 * the Geman-McClure penalty rho(r) = sigma^2 r^2 / (sigma^2 + r^2) on each coordinate of r = (u - u^, v - v^):
 * stats[0] = coef / (n_poses * 24) * sum c (rho(r_u) + rho(r_v)), stats[1] = the mean |r| over the joints with c > 0
 * in front of the camera (0 when there is none).  Writes d_kps (n_poses,24,3) = d stats[0] / d kps.  A joint with
 * w <= 1e-6 (at or behind the camera) contributes 0 to both stats and to d_kps.  sigma > 0.  One launch. */
int danbo_pose_kp2d(const float* kps, const float* kp2d, const float* proj, int n_poses, float sigma, float coef,
                    float* d_kps, float* stats, void* stream);

/* L*: the trainer's losses on the outputs of the path, value and gradients in one launch (core/trainer.py:396-422
 * _compute_nerf_loss with loss_fn L1 (loss_kind 0) or MSE (1) on rgb + (1 - acc) bg for the fine and, if rgb0 != NULL,
 * the coarse maps; :507-536 _compute_soft_softmax_loss when confd != NULL; :538-553 _compute_volume_scale_loss when
 * axis_scale != NULL).  target (n,3); bgs (n,3) or NULL (then bg_scalar); confd / part_invalid (n,S_t,24); T_i / alpha
 * (n,S_t).  terms[4] (device doubles, overwritten) = { rgb, rgb coarse, soft-softmax, volume-scale } with their
 * coefficients applied; their sum is the trainer's total loss.  g_* receive d total / d input (written), except
 * g_axis_scale (24,3), which is added to. */
int danbo_train_loss(const float* rgb_map, const float* acc_map, const float* rgb0, const float* acc0,
                     const float* target, const float* bgs, float bg_scalar, int use_background, int n_rays,
                     int loss_kind, float rgb_coef, float coarse_weight, const float* confd, const float* part_invalid,
                     const float* T_i, const float* alpha, int S_t, float soft_coef, const float* axis_scale,
                     const float* init_scale, float vol_coef, double* terms, float* g_rgb_map, float* g_acc_map,
                     float* g_rgb0, float* g_acc0, float* g_confd, float* g_axis_scale, void* stream);

/* Adam (torch.optim.Adam formulas, raycasters.py:71-78: betas (0.9, 0.999), no weight decay) over one flat fp32 arena
 * holding every parameter; grads / exp_avg / exp_avg_sq are arenas of the same layout; all 16-byte aligned.  lr_dev
 * and step_dev are device floats (step already incremented) so that a captured graph reads their current values. */
int danbo_adam_step(float* params, const float* grads, float* exp_avg, float* exp_avg_sq, long long n,
                    const float* lr_dev, float beta1, float beta2, float eps, const float* step_dev, int num_sms,
                    void* stream);

/* ---- AN1: A-NeRF field (nerf_type = nerf, BASELINE config #4) -------------------------------------------------
 * Replaces core/networks/nerf.py:164-279 (encode_pts / encode_views / inference with W = 448, view_W = 224),
 * core/cutoff_embedder.py:151-214 and core/encoders.py:305-317,639-651,774-795.  Every sample goes through the field
 * (the cutoff never makes an encoding exactly zero), rows are dense: row = ray * S + sample. */

/* Buffer sizes: packed weight stream, fp32 head vector, frame-code slice of the view layer, per-CTA activation scratch. */
int danbo_anerf_workspace_bytes(int num_sms, long long* wstream_bytes, long long* heads_bytes, long long* code_bytes,
                                long long* scratch_bytes);

/* fp32 nn.Linear weights (pts_linears.0-7 (448,432|448|880), alpha, feature (448,448), views_linears.0 (224,1224), rgb
 * (3,224)) -> bf16 stage stream in consumption order per CTA of a pair, head vector, transposed code slice + b_view. */
int danbo_anerf_pack_weights(const float* const* w_pts, const float* const* b_pts, const float* w_alpha,
                             const float* b_alpha, const float* w_feat, const float* b_feat, const float* w_view,
                             const float* b_view, const float* w_rgb, const float* b_rgb, void* wstream, float* heads,
                             float* w_code, void* stream);

/* Per ray: unit ray direction in each of the 24 bone frames with its 4-octave encoding (n,648) fp32 [row 9][72], and
 * the frame-code contribution of the view layer (n,224) = W_v[:,1096:1224] . code + b_v.  codes as danbo_ray_bias. */
int danbo_anerf_ray_encode(const float* rays, int ray_stride, int n_rays, const float* pose_skts, int rays_per_pose,
                           int n_poses, const int* cam_idx, const float* codes, int n_codes, const float* w_code,
                           float* ray_enc, float* code_bias, void* stream);

/* Per sample (row = ray * S + s, z (n_rays,S)): density input [cutoff PE of the 24 bone distances (360) ; unit vectors
 * (72)] -> xd, view input [direction encoding x cutoff weight (648)] -> xv; bf16 operand tile images of
 * ceil(n_rows/128) tiles x 7 (xd) / 11 (xv) chunks of 16 KB.  align = (24,4,4) bone-align transforms, tau = 20 at init. */
int danbo_anerf_embed(const float* rays, int ray_stride, int S, const float* z, int n_rows, const float* pose_skts,
                      int rays_per_pose, int n_poses, const float* align, const float* ray_enc, float tau, void* xd,
                      void* xv, void* stream);

/* The 8 x 448 MLP + heads on n_rows rows: out (rows,4) = [rgb, sigma].  One persistent launch over CTA pairs.
 * trace: NULL, or 320 long long receiving a clock64 timeline of CTA 0 ([2 tiles][issuer, epilogue][layer, pass][begin,
 * end], then [2 tiles][layer, pass][4 stamps inside one epilogue warp]; profiling aid). */
int danbo_anerf_mlp(const void* xd, const void* xv, const void* wstream, const float* heads, const float* code_bias,
                    void* scratch, int n_rows, int S, float* out, int out_capacity, int num_sms, long long* trace,
                    void* stream);

/* Train-mode variant of danbo_anerf_mlp: every layer's bf16 activation tile image is kept in `save`
 * (danbo_anerf_save_bytes bytes: [tile][9 = pts_linears.0-7 outputs, feature_linear output][7 chunks of 16 KB],
 * operand layout) for the backward pass (autograd of core/networks/nerf.py:164-209 as reached from trainer.py:573). */
int danbo_anerf_save_bytes(int n_rows, long long* bytes);
int danbo_anerf_mlp_save(const void* xd, const void* xv, const void* wstream, const float* heads, const float* code_bias,
                         void* scratch, int n_rows, int S, float* out, int out_capacity, int num_sms, void* save,
                         void* stream);

/* Operand tile images ([tile][chunk][128 rows x 64 k] bf16, 128-byte swizzle; tile_stride bytes between tiles) ->
 * row-major bf16 out (n_rows, n_chunks * 64): how the A-NeRF backward reads xd / xv / saved activations. */
int danbo_anerf_untile(const void* img, long long tile_stride, int n_rows, int n_chunks, void* out, void* stream);

/* Backward of danbo_anerf_embed and of the direction part of danbo_anerf_ray_encode to the poses (pose refinement,
 * --opt_pose): autograd of core/encoders.py:288-303,305-317,442-444,639-651,774-795 and core/cutoff_embedder.py:151-214
 * (encode_pts / encode_views, core/networks/nerf.py:222-279) with respect to skts.  Rows are dense (row = ray * S + s);
 * z, pose_skts, align, ray_enc and tau are what the forward calls of the pass read.  d_xd (n_rays*S,432) and d_xv
 * (n_rays*S,648) fp32, row-major: d loss / d the density and view inputs.  d_skts (n_poses,24,4,4) fp32 is added to
 * (zero it first); rows 0-2 only, the homogeneous row gets nothing.  Near/far and the sample depths are constants. */
int danbo_anerf_embed_bwd(const float* rays, int ray_stride, int n_rays, int S, const float* z, const float* pose_skts,
                          int rays_per_pose, int n_poses, const float* align, const float* ray_enc, float tau,
                          const float* d_xd, const float* d_xv, float* d_skts, void* stream);

#ifdef __cplusplus
}
#endif
#endif
