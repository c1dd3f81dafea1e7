/* interdiff_b200.h -- C ABI of libinterdiff_b200.so (sm_100a).
 *
 * Drop-in boundary for the InterDiff sampling hot path (SURVEY.md section 8b).  The reference
 * reaches this path through Python module APIs, not an FFI; each entry point below names the
 * reference interface it replaces (paths relative to /root/reference/interdiff).  The Python
 * veneer in interdiff_b200/ binds these with ctypes (see INTEGRATION.md for the stub a
 * maintainer of the reference would add).
 *
 * Conventions: plain pointers and sizes only (no torch types); every function returns 0 on
 * success and a non-zero status otherwise, with a message in idb_last_error(); nothing throws
 * or aborts across the boundary.  `stream` is a cudaStream_t passed as void* (NULL = default
 * stream); all work is enqueued on it and no call synchronises unless documented.  Tensor
 * arguments are DEVICE pointers to contiguous float32 unless marked `host_or_dev` (those are
 * copied with cudaMemcpyDefault).  One handle per device; a handle is not re-entrant.
 */
#ifndef INTERDIFF_B200_H
#define INTERDIFF_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct idb_handle idb_handle;

int idb_version(void);
int idb_create(idb_handle** out);                 /* on the current CUDA device */
int idb_destroy(idb_handle* h);
const char* idb_last_error(const idb_handle* h);
long long idb_launch_count(const idb_handle* h);  /* kernels launched so far through h */
int idb_set_gemm_backend(idb_handle* h, int backend); /* 0 = fp32 SIMT (debug/bisect), 1 = tcgen05 split-fp16 (default) */
/* Programmatic dependent launch between the kernels of a sampling step (default 1). Results are identical
   either way; 0 serialises the kernels (for bisecting / profiling). */
int idb_set_dependent_launch(idb_handle* h, int on);
/* Feed-forward block of a decoder layer as one cluster kernel (tensor backend, d_model 256, d_ff 1024): 2 (default) = incl.
   the layer's final LayerNorm in its reduction epilogue, 1 = feed-forward only, 0 = the two separate GEMMs (bisecting);
   3 = a layer's attention half in the same kernel (option, not faster).  10 / 11: self- and cross-attention of the standard
   layers as two launches / one launch (default 11; identical results). */
int idb_set_fused_mlp(idb_handle* h, int on);
/* Cluster-pruned nearest-neighbour search when the target is the loaded body mesh (default 1; results are identical
   to the brute-force scan, index ties included); 0 = always brute force. */
int idb_set_nn_pruning(idb_handle* h, int on);

/* ---- denoiser: MDM.forward / MDM._decode --------------------------------------------------
 * replaces model/diffusion_smpl.py:239-246,226-237 (variant 0) and
 * model/diffusion_skeleton.py:250-257,231-248 (variant 1), incl. TimestepEmbedder
 * (model/layers.py:42-43), PositionalEncoding (:24-26), the 8-layer TransformerDecoder
 * (:258-264; torch.nn.TransformerDecoderLayer for layers without `queries`,
 * TransformerDecoderLayerQaN model/sublayers.py:311-375 otherwise). */
typedef struct {
    int variant;          /* 0 = SMPL (144 ch), 1 = skeleton (106 ch) */
    int d_model;          /* 256 */
    int n_heads;          /* 4 */
    int d_ff;             /* 1024 (SMPL ckpt) / 256 (skeleton ckpt) */
    int n_layers;         /* 8 */
    int n_queries;        /* 10 */
    int c_body;           /* 135 / 63 : channels fed to bodyEmbedding */
    int c_obj;            /* 9 / 36   : channels fed to objEmbedding */
    int c_extra;          /* 0 / 7    : trailing channels not embedded (skeleton 7-D pose) */
    int n_points;         /* skeleton: object keypoints (12); SMPL: 0 */
    int qan_mask;         /* bit i set => layer i is a QaN layer (0x7e for the shipped models) */
    float rotary_offsets[3]; /* q_pos - k_pos for key slots (t-1, t, t+1): {1,0,-1} ('absolute'
                                local-attention <=1.5) or {2,1,0} ('bucketed' >=1.6) */
} idb_denoiser_config;

int idb_denoiser_init(idb_handle* h, const idb_denoiser_config* cfg);
/* Load one tensor by its reference state_dict name without the "model." prefix, e.g.
 * "decoder.layers.3.queries"; data host_or_dev float32.  Unknown names are ignored (returns 0)
 * so a whole checkpoint can be streamed in (strict loading is done by the Python veneer). */
int idb_denoiser_load(idb_handle* h, const char* name, const float* data, const int64_t* shape, int ndim);
int idb_denoiser_commit(idb_handle* h);           /* checks completeness, packs / folds weights */
/* Bind a batch: cond = MDM._get_embeddings()[0], (Tm,B,D) seq-first as the reference passes it
 * in model_kwargs['y']['cond']; zero_pose_obj (B,P,3) for variant 1 else NULL.  Precomputes the
 * step-invariant cross-attention K/V of `cond` for every layer. */
int idb_denoiser_bind(idb_handle* h, int B, int T, int Tm, const float* cond, const float* zero_pose_obj, void* stream);
/* x (B,1,C,T), timesteps (B) int64 device, out (B,1,C,T)  == MDM.forward(x, timesteps, y) */
int idb_denoiser_forward(idb_handle* h, const float* x, const int64_t* timesteps, float* out, void* stream);

/* Conditioning encoder = the part of MDM._get_embeddings after the point-cloud encoder (reference
 * model/diffusion_smpl.py:217-221; encoder layers :20-70, model/sublayers.py:37-203):
 *   cond = encoder(PositionalEmbedding(bodyEmbedding(past[:, :135]) + objEmbedding(past[:, 135:]) + pc_embedding))
 * Needs the "encoder.layers.*" tensors to have been loaded (idb_denoiser_load) before idb_denoiser_commit.
 *   past         (B,1,C,Tp)  the first past_len frames of the motion tensor, channels [body | object]
 *   pc_embedding (B,256)     pcEmbedding(...).view(1,B,-1)[0]   (PointNet++ itself is the remaining half of SURVEY 8f rank 1)
 *   cond_out     (Tp,B,256)  sequence-first like the reference; feed it to idb_denoiser_bind */
int idb_encode_condition(idb_handle* h, int B, int Tp, const float* past, const float* pc_embedding, float* cond_out, void* stream);

/* Conditioning encoder of the skeleton model (variant 1) = MDM._get_embeddings after the `gt` concatenation (reference
 * model/diffusion_skeleton.py:194-215):
 *   cond = encoder(PositionalEmbedding(bodyEmbedding(body_past) + objEmbedding(obj_past) + shapeEmbedding(zero_pose_obj)))
 * Needs the "encoder.layers.*" (d_ff 256) and "shapeEmbedding.*" tensors loaded before idb_denoiser_commit.
 *   past          (B,1,C,Tp)        the first past_len frames of the sample tensor, C = 3 n_joints + 3 n_points + 7 (the 7 pose
 *                                   channels are not embedded, as in the reference)
 *   zero_pose_obj (B,n_points,3)    canonical object keypoints (model_kwargs['zero_pose_obj'])
 *   cond_out      (Tp,B,256)        sequence-first like the reference; feed it to idb_denoiser_bind */
int idb_encode_condition_skeleton(idb_handle* h, int B, int Tp, const float* past, const float* zero_pose_obj, float* cond_out,
                                  void* stream);

/* PointNet++ (MSG) point-cloud encoder = MDM.pcEmbedding, PointNet2Encoder(c_in=1, c_out=256, num_keypoints=1)
 * (reference model/layers.py:111-175, called at model/diffusion_smpl.py:210-211); the furthest-point-sampling /
 * ball-query / grouping operators of the un-vendored pointnet2_ops 3.0.0 are rebuilt for sm_100a.
 * Needs the "pcEmbedding.*" tensors (incl. the BatchNorm running statistics) loaded before idb_denoiser_commit.
 *   obj_points   (B,P,3)   object point cloud in the canonical frame (P = 2048 in the reference; 512..4096)
 *   pc_embedding (B,256)   = pcEmbedding(cat([p, |p|]).unsqueeze(0)).view(1,B,-1)[0]  -> idb_encode_condition */
int idb_pointcloud_embed(idb_handle* h, int B, int P, const float* obj_points, float* pc_embedding, void* stream);

/* ---- diffusion: SpacedDiffusion / GaussianDiffusion sampling ------------------------------
 * replaces diffusion/gaussian_diffusion.py:160-197 (tables), 277-388 (p_mean_variance, START_X,
 * FIXED_SMALL, inpainting blend :307-311), 253-275, 496-548 (p_sample), 598-736 (p_sample_loop),
 * diffusion/respace.py:64-129 (timestep_map).  betas: the (re-spaced) float64 schedule on the
 * host; timestep_map[n] the model timestep of step index i. */
int idb_diffusion_init(idb_handle* h, const double* betas, const int64_t* timestep_map, int n);
/* One p_sample at step index i: x_t -> x_{t-1}.  gt/mask (uint8, 1 = keep gt) may be NULL (no
 * inpainting); noise is the eps drawn for this step; x0_out may be NULL. */
int idb_p_sample(idb_handle* h, int i, const float* x_t, const float* noise, const float* gt,
                 const uint8_t* mask, float* x_out, float* x0_out, void* stream);
/* The two halves of p_sample around the denoised_fn hook (gaussian_diffusion.py:354-360):
 * predict: x0 = inpaint(model(x_t, t_i));  finish: x_{t-1} = posterior(x0', x_t) + sigma*noise */
int idb_p_sample_predict(idb_handle* h, int i, const float* x_t, const float* gt, const uint8_t* mask,
                         float* x0_out, void* stream);
int idb_p_sample_finish(idb_handle* h, int i, const float* x0, const float* x_t, const float* noise,
                        float* x_out, void* stream);
/* Whole loop: x_T = tape[0], eps of the k-th executed step = tape[k+1] (n+1 entries of the
 * sample shape); steps i = n-1 .. 0.  correction != 0 runs the fused denoised_fn
 * (idb_correction_apply) on the steps the reference's hook is active on (t <= 500, t % 50 == 0), in the reference's order
 * model -> inpaint blend -> hook -> posterior (gaussian_diffusion.py:305-376; no re-inpainting after the hook).
 * use_graph: 0 = plain launches, 1 = one captured CUDA graph per step replayed n times, 2 = the whole loop as ONE graph.
 * gt / mask are copied into handle-owned buffers and the tape is read through a device slot, so captured graphs are
 * reused for any later call of the same (B, T, n, mask present, correction) on fresh tensors. */
int idb_p_sample_loop(idb_handle* h, const float* tape, const float* gt, const uint8_t* mask,
                      int correction, int use_graph, float* x_out, void* stream);

/* ---- SMPL-H linear blend skinning: SMPL_Layer.forward -------------------------------------
 * replaces libsmpl/smplpytorch/pytorch/smpl_layer.py:72-175 (+ rodrigues_layer.py:13-52,
 * tensutils.py:6-53).  Model arrays host_or_dev: v_template (V,3), shapedirs (V,3,NB),
 * posedirs (V,3,(J-1)*9), J_regressor (J,V), weights (V,J), parents (J) int32, faces (Fc,3) int32. */
int idb_body_init(idb_handle* h, int V, int J, int NB, int Fc, const float* v_template, const float* shapedirs,
                  const float* posedirs, const float* J_regressor, const float* weights,
                  const int32_t* parents, const int32_t* faces);
/* pose (F,J*3) axis-angle, betas (F,NB), trans (F,3) -> verts (F,V,3), jtr (F,J,3) (either may be NULL) */
int idb_smplh_lbs(idb_handle* h, int F, const float* pose, const float* betas, const float* trans,
                  float* verts, float* jtr, void* stream);

/* ---- geometry helpers ---------------------------------------------------------------------
 * vertex_normals: data/tools.py:4-39 (faces shared by all frames = body faces of idb_body_init)
 * signed_nn:      tools.py:11-76 point2point_signed, one direction: for every query point the
 *                 first-minimum squared-L2 nearest target (chamfer_distance ext, tools.py:45-47),
 *                 dist = |q - t_nn| * sign(n_nn . (q - t_nn)) when target normals are given. */
int idb_vertex_normals(idb_handle* h, int F, const float* verts, float* normals, void* stream);
int idb_signed_nn(idb_handle* h, int F, int Pq, int Pt, const float* query, const float* target,
                  const float* target_normals, float* signed_dist, int32_t* idx, float* vec, void* stream);
/* rotation conversions used around the loop (pytorch3d.transforms 0.7.2 semantics):
 * rot6d (n,6) -> axis-angle (n,3) == matrix_to_axis_angle(rotation_6d_to_matrix(.)) */
int idb_rot6d_to_axis_angle(idb_handle* h, int n, const float* rot6d, float* aa, void* stream);

/* ---- correction: ObjProjector.sample + denoised_fn ----------------------------------------
 * replaces model/correction_smpl.py:79-138 (eval mode) and eval_smpl_short.py:84-130. */
int idb_projector_init(idb_handle* h, int past_len, int future_len, int n_pre, int n_markers);
int idb_projector_load(idb_handle* h, const char* name, const float* data, const int64_t* shape, int ndim);
int idb_projector_commit(idb_handle* h);
/* marker indices (into the P markers) that get the +0.5 hand bonus in the hypothesis selection
 * (correction_smpl.py:129-130; data/utils.py:252-253), host_or_dev */
int idb_projector_set_hand_markers(idb_handle* h, const int32_t* ids, int n);
/* obj_angles (T,B,6), obj_trans (T,B,3), markers (T,B,P,3), contact (B,P) int32 -> out (T,B,9) */
int idb_projector_sample(idb_handle* h, int T, int B, const float* obj_angles, const float* obj_trans,
                         const float* markers, const int32_t* contact, float* out, void* stream);
/* Bind the per-batch context of the hook: hand_pose (T,B,90), betas (T,B,10), obj_points (B,P,3),
 * marker vertex ids (n_markers) int32, hand marker ids (n_hand) int32 (host_or_dev). */
int idb_correction_bind(idb_handle* h, int B, int T, int past_len, int n_obj_points, const float* hand_pose,
                        const float* betas, const float* obj_points, const int32_t* marker_ids,
                        const int32_t* hand_marker_ids, int n_hand, void* stream);
/* denoised_fn body for an ACTIVE step (the caller applies the t <= 500 && t % 50 == 0 gate):
 * x0 (B,1,144,T) is corrected in place; gt is the inpainted motion; t is the timestep value used
 * in the (t/1000) blend.  Optional debug outputs (may be NULL): condition (B) uint8,
 * contact (B,P) int32, markers (T,B,P,3), o2h_signed (T*B,Pobj). */
int idb_correction_apply(idb_handle* h, float* x0, const float* gt, int t, uint8_t* condition_out,
                         int32_t* contact_out, float* markers_out, float* o2h_out, void* stream);
/* ---- skeleton correction net + hook (model/correction_skeleton.py:8-135, eval_skeleton.py:80-111) ----
 * idb_projector_init_skeleton: n_pre 20, n_joints (21) + 1 nodes, joint stack 9-64-32-64-9; weights through idb_projector_load /
 * idb_projector_commit under the same state_dict names.  idb_projector_sample_skeleton = ObjProjector.sample: quaternions xyzw
 * (T,B,4), translations (T,B,3), joints (T,B,n_joints,3).  idb_skeleton_correction_apply = the body of the skeleton denoised_fn
 * for an active step, in place on x0 (B,1,3 n_joints + 3 n_points + 7,T); with a skeleton projector loaded
 * idb_p_sample_loop(correction = 1) runs it on the reference's schedule (t <= 500, t % 50 == 0). */
int idb_projector_init_skeleton(idb_handle* h, int past_len, int future_len, int n_joints);
int idb_projector_sample_skeleton(idb_handle* h, int T, int B, const float* obj_quat, const float* obj_trans, const float* joints,
                                  float* quat_out, float* trans_out, void* stream);
int idb_skeleton_correction_apply(idb_handle* h, int B, int T, int n_points, float* x0, const float* gt, const float* zero_pose_obj,
                                  int t, void* stream);
/* Parity hook for the in-loop path: device buffers cond_log [capacity][B] uint8, contact_log [capacity][B][n_markers] int32
 * receive the decisions of every correction step enqueued after this call, in order (NULL, NULL, 0 = off). */
int idb_correction_set_log(idb_handle* h, uint8_t* cond_log, int32_t* contact_log, int capacity);

/* Evaluation metrics of a batch of predictions (reference eval_smpl_short.py:24-81 `metrics`), per sample, on the device:
 *   obj_pred / obj_gt (T,B,6) = [axis-angle | translation], body_jtr(_gt) (T,B,J,3), body(_gt) (T,B,Db) with the global
 *   translation in the last 3 channels, verts (T,B,V,3) of the loaded body model, obj_points (B,P,3) canonical object cloud.
 *   out [6][B]: global_mpjpe, local_mpjpe (pelvis aligned), body_translation, obj_translation, obj_rot_error
 *   (min over the quaternion sign of the L1 distance), penetrate (share of posed object points inside the body). */
int idb_metrics(idb_handle* h, int T, int B, int J, int P, int Db, const float* obj_pred, const float* body_jtr, const float* body,
                const float* obj_gt, const float* body_jtr_gt, const float* body_gt, const float* verts, const float* obj_points,
                float* out, void* stream);

/* Evaluation metrics of the skeleton model, per sample, on the device (reference eval_skeleton.py:46-68 calc_metric_single and
 * train_diffusion_skeleton.py:65-87 calc_metric, which average the same terms over the whole batch):
 *   pred / gt (B,1,3 n_joints + 3 n_points + 7,T) in the sample layout, channels [joints | object keypoints | trans(3), quat xyzw(4)]
 *   out [5][B]: means over the future frames t >= past_len of mpjpe_h (L2 over joints), mpjpe_o (L2 over keypoints),
 *   translation_error, rotation_error (min over the quaternion sign of the L1 distance, eval_skeleton.py) and
 *   rotation_error_l2 (the same with the L2 norm, train_diffusion_skeleton.py). */
int idb_skeleton_metrics(idb_handle* h, int B, int T, int past_len, int n_joints, int n_points, const float* pred, const float* gt,
                         float* out, void* stream);

/* Post-processing of a sampled window: `smooth` (eval_smpl_short.py:217-223) in place on x (T, inner) - every future frame is
 * shifted by 2 x[-F-1] - x[-F-2] - x[-F] (old values) - and the element-wise minimum that reduces the metric vectors of the
 * diverse samples of a batch (eval_smpl_short.py:268-296: torch.stack + min). */
int idb_smooth(idb_handle* h, int T, int future_len, long long inner, float* x, void* stream);
int idb_metric_min(idb_handle* h, long long n, float* acc, const float* cur, void* stream);

/* ---- autoregressive rollout: the step between two sampling windows (eval_smpl_long.py:26-84 get_batch, :278 denormalize) ----
 * idb_rollout_next_window: from a finished window in the post-processed form - body (T,B,Db) = [66 axis-angle | hand | 3 trans],
 * obj (T,B,6) = [axis-angle | trans], jtr (T,B,J,3) - builds the NEXT window's inpainting tensor gt_out (B,1,144,T): its first
 * past_len frames are the last past_len frames of the finished window, translations relative to centroid_out (B,3) = the
 * pelvis (joint 0) of the first of those frames, rotations re-derived as axis-angle -> matrix -> first two rows
 * (model/diffusion_smpl.py:207-214); the remaining frames repeat the last past frame (eval_smpl_long.py:78).
 * idb_add_offset: x[(t*B+b)*ld + col0 + 3k + c] += sign * offset[b][c], k < K - `denormalize` (sign +1) of translations,
 * vertices and joints back to world coordinates (upstream calls it without defining it; this is get_batch's inverse). */
int idb_rollout_next_window(idb_handle* h, int T, int B, int J, int Db, int past_len, const float* body, const float* obj,
                            const float* jtr, float* gt_out, float* centroid_out, void* stream);
int idb_add_offset(idb_handle* h, int T, int B, int K, long long ld, int col0, float* x, const float* offset, float sign, void* stream);

/* bisecting hook: 0 = the SMPL-H blend GEMM without TMA-multicast row-tile pairs (identical results; default 1) */
int idb_debug_set_gemm_multicast(idb_handle* h, int on);
/* profiling hook: 8-CTA clusters of the fused decoder-layer kernel that fit on the device at once (-1 on error) */
int idb_debug_max_layer_clusters(idb_handle* h);

/* ---- kernel-level hook (tests / bench roofline leg) -----------------------------------------
 * C[M,N] = epi(A[M,K] . W[N,K]^T) with the handle's GEMM backend; epi bit 0 bias, 1 GELU(erf),
 * 2 residual add, 3 SiLU (the fused epilogues of the nn.Linear calls of the denoiser). */
int idb_debug_gemm(idb_handle* h, const float* A, const float* W, const float* bias, const float* res, float* C,
                   int M, int N, int K, int epi, void* stream);
/* the same launch repeated `iters` times from C (roofline leg: host overhead per launch stays small) */
int idb_debug_gemm_repeat(idb_handle* h, const float* A, const float* W, const float* bias, const float* res, float* C,
                          int M, int N, int K, int epi, int iters, void* stream);

/* test hook: number of round-robin TMEM accumulators of the tcgen05 GEMM (0 = default) */
int idb_debug_set_gemm_accumulators(int n);
/* out[M][256] = [LayerNorm(] gelu(x w1^T + b1) w2^T + b2 + res [)] through the fused feed-forward kernel (fp32 device
   pointers; ln_w / ln_b NULL = no norm); iters > 1: launches 2..iters are timed (idb_debug_last_ms); trace != NULL:
   clock64 timeline [ctas][16] of launch 1 */
int idb_debug_mlp(idb_handle* h, const float* x, const float* w1, const float* b1, const float* w2, const float* b2,
                  const float* res, float* out, int M, int iters, long long* trace, const float* ln_w, const float* ln_b,
                  void* stream);
double idb_debug_last_ms(const idb_handle* h);
/* clock64 phase timeline (16 slots, host pointer) of CTA (0,0) of the last fused QaN + cross-attention kernel */
int idb_debug_attn_trace(long long* out16);
/* chain timeline probe (profiles/chain_probe.py): device buffer of 64 lanes x (2 + 2 * capacity) uint64, lane[0] = 0, lane[1] = capacity; every
   kernel of the sampling step then appends (kind | event | grid | block, %globaltimer) records; NULL switches it off */
int idb_debug_chain_trace(idb_handle* h, unsigned long long* buf);
/* one launch with a per-CTA clock64 timeline (16 slots per CTA) of the tcgen05 kernel's pipeline */
int idb_debug_gemm_trace(idb_handle* h, const float* A, const float* W, float* C, int M, int N, int K, long long* trace, void* stream);

/* debug: fp16 (hi, lo) operand split (x = hi + lo * 2^-11), and a GEMM on such pairs */
int idb_debug_split(idb_handle* h, const float* x, void* hi, void* lo, int rows, int cols, int ld_dst, void* stream);
int idb_debug_gemm_presplit(idb_handle* h, const void* A_hi, const void* A_lo, const void* W_hi, const void* W_lo,
                            const float* bias, float* C, int M, int N, int K, int epi, int iters, long long* trace, void* stream);

#ifdef __cplusplus
}
#endif
#endif
