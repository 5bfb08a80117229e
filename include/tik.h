/* tik.h -- C ABI of libtik.so: the B200 (sm_100a) learned-IK inference hot path.
 *
 * Drop-in boundary for khanhha/temporal_inverse_kinematics (reference paths below are
 * relative to the reference checkout).  The reference has no FFI of its own: its hot path
 * is the PyTorch nn.Module / function API, so every entry point here names the Python
 * symbol it replaces.  The host-side mirror that keeps those Python signatures lives in
 * temporal_inverse_kinematics_b200/ and binds this header with ctypes (see INTEGRATION.md).
 *
 * Conventions
 *   - plain C: raw pointers + sizes, no torch / C++ types.
 *   - every pointer marked `dev` is CUDA device memory owned by the caller (PyTorch owns all
 *     tensors, workspaces included); the library never allocates or frees device memory.
 *   - `stream` is a cudaStream_t passed as void*; calls only enqueue work and return
 *     (no host synchronisation, CUDA-graph capturable once a plan exists).
 *   - return value: 0 = TIK_OK, negative = error; tik_last_error() gives a thread-local message.
 *   - activations inside the network use the "node-major" layout (N, V, T, C): channel
 *     contiguous, then time, then graph node, then clip.  Entry points say where the
 *     reference's own layouts ((N,T,V,C) input, (N,C,T,V) NCHW between modules) are converted.
 */
#ifndef TIK_H_
#define TIK_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define TIK_OK 0
#define TIK_ERR_INVALID (-1)     /* bad argument / unsupported shape */
#define TIK_ERR_CUDA (-2)        /* CUDA runtime or driver error */
#define TIK_ERR_UNSUPPORTED (-3) /* valid in the reference but not built here */
#define TIK_ERR_WORKSPACE (-4)   /* caller-provided workspace too small */

#define TIK_F32 0
#define TIK_BF16 1

#define TIK_MAX_BLOCKS 16
#define TIK_MAX_SLABS 6
#define TIK_MAX_JOINTS 64

int tik_version(void);
const char* tik_last_error(void);
/* 0 if the current CUDA device is compute capability 10.x (the only target), else TIK_ERR_UNSUPPORTED. */
int tik_check_device(void);

/* ------------------------------------------------------------------ rotation conversions
 * All tensors fp32, contiguous, device.  M = number of rotations. */

/* common/geometry.py:330-344 rot6d_to_rotmat (identical to rot6d_to_rotmat_spin :308-327).
 * x6 (M,6) -> R (M,3,3) with columns b1,b2,b3. */
int tik_rot6d_to_rotmat(const float* x6_dev, float* R_dev, int64_t M, void* stream);
/* common/kornia_geometry_conversion.py:125-201 angle_axis_to_rotation_matrix. aa (M,3) -> R (M,3,3). */
int tik_aa_to_rotmat(const float* aa_dev, float* R_dev, int64_t M, void* stream);
/* common/geometry.py:22-65 batch_rodrigues (+quat2mat). aa (M,3) -> R (M,9). */
int tik_batch_rodrigues(const float* aa_dev, float* R9_dev, int64_t M, void* stream);
/* common/geometry.py:68-97 rotation_matrix_to_angle_axis (w,x,y,z path, NaN->0). R (M,3,3) -> aa (M,3).
 * kornia_quirk != 0 reproduces common/kornia_geometry_conversion.py:204-227 instead (SURVEY.md 0.6). */
int tik_rotmat_to_aa(const float* R_dev, float* aa_dev, int64_t M, int kornia_quirk, void* stream);

/* The quaternion helpers the two conversions above are made of, as the reference exposes them (all (w,x,y,z)):
 * common/geometry.py:37-65 quat2mat (normalises, q (M,4) -> R (M,3,3)); :153-233 rotation_matrix_to_quaternion
 * (R (M,3,3) -> q (M,4), four-case selection on the transposed matrix); :100-150 quaternion_to_angle_axis (q -> aa). */
int tik_quat_to_rotmat(const float* q_dev, float* R_dev, int64_t M, void* stream);
int tik_rotmat_to_quat(const float* R_dev, float* q_dev, int64_t M, void* stream);
int tik_quat_to_aa(const float* q_dev, float* aa_dev, int64_t M, void* stream);

/* Per-frame mean of overlapping window predictions (inference.py:56-67), for one window per frame: window w is centred
 * on packed frame w.  preds (frames, T_out, D) -> out (frames, D), fp32.  Sequences as in TikSeqBatch: frame_start_dev
 * (n_seqs+1) device table.  Frame j, local index i in its sequence of F_s frames, averages preds[j - o, o + h] over
 * o = -h..h with 0 <= i - o < F_s, summed in ascending o from 0 and divided by the count (IEEE division).
 * TIK_MEAN_EUCLIDEAN averages the D values; TIK_MEAN_ROTATION (D % 3 == 0) averages the Rodrigues matrices of each
 * axis-angle triple, projects the mean back by Gram-Schmidt of its first two columns and returns axis-angle
 * (tik_batch_rodrigues, tik_rot6d_to_rotmat, tik_rotmat_to_aa).  h = 0 copies preds[:, 0] in both modes.
 * Requires 2h+1 <= T_out.  frames = 0 is a no-op.  CUDA-graph capturable. */
#define TIK_MEAN_EUCLIDEAN 0
#define TIK_MEAN_ROTATION 1
int tik_window_mean(const float* preds_dev, int64_t frames, int T_out, int D, const int64_t* frame_start_dev,
                    int64_t n_seqs, int h_w_size, int mode, float* out_dev, void* stream);

/* ------------------------------------------------------------------ body forward kinematics
 * Replaces the joint output of common/smpl_util.py:22-82 run_smpl_inference -> smplx forward
 * (third-party; restated from the published SMPL chain, see oracle/fk_port.py).
 *   pose_dev     (F, J, 3) axis-angle if pose_is_rotmat == 0 (Rodrigues as common/geometry.py:22-65),
 *                (F, J, 3, 3) local rotation matrices otherwise
 *   rest_host    (J,3) rest joints, HOST memory (copied into kernel arguments)
 *   parents_host (J) parent index, -1 for the root, parents[i] < i, HOST memory
 *   transl_dev   (F,3) or NULL
 *   joints_dev   (F,J,3) out; local_R_dev / global_R_dev (F,J,3,3) out, each may be NULL.
 * J <= TIK_MAX_JOINTS (64): the 22-joint SMPL-X body tree and the 60-joint full skeleton (55 joints + 5 face landmarks
 * as rigid children of the head, data_amass.py:176-218) have thread-per-frame specialisations; any other tree runs on
 * a warp-per-frame kernel (J <= 32: pointer jumping over shuffles; J <= 64: level order through shared memory). */
int tik_fk_body(const float* pose_dev, int pose_is_rotmat, const float* rest_host, const int32_t* parents_host,
                int J, const float* transl_dev, float* joints_dev, float* local_R_dev, float* global_R_dev,
                int64_t F, void* stream);

/* ------------------------------------------------------------------ mesh skinning
 * Replaces the vertex output of common/smpl_util.py:22-82 run_smpl_inference(return_mesh=True) -> smplx.lbs.lbs
 * (third-party; restated from the published SMPL-X formulation, see oracle/lbs_port.py).  The 55 SMPL-X joints and
 * their local / global rotations come from tik_fk_body (want local and global rotations, NO transl); tik_lbs adds the
 * pose blend shapes, skins the vertices and applies transl to vertices and joints, as smplx does.
 * Device arrays of a model, packed once by the caller (temporal_inverse_kinematics_b200/smpl_util.py SmplxBodyModel): */
#define TIK_LBS_MAX_LANDMARKS 8
typedef struct TikLbsModel {
  int32_t V;                 /* vertices */
  int32_t J;                 /* joints: 55 */
  int32_t kmax;              /* columns of the sparse skinning table: most non-zero weights of any vertex */
  int32_t n_landmarks;       /* joints J .. J+n_landmarks-1 are these vertices (smplx VertexJointSelector) */
  int32_t landmark_vid[TIK_LBS_MAX_LANDMARKS];
  const float* v_shaped_dev;     /* (V,3) fp32: v_template + shapedirs . betas */
  const float* rest_joints_dev;  /* (J,3) fp32: J_regressor . v_shaped, the rest joints given to tik_fk_body */
  const void* posedirs_dev;      /* (ceil(3V/128)*128, 512) in the call's dtype, K contiguous: row 3v+c, column
                                    9(j-1)+3a+b = posedirs[v,c,9(j-1)+3a+b] of the model file, zero padded; 16-byte aligned */
  const int32_t* skin_idx_dev;   /* (V,kmax) joint of each non-zero skinning weight (padding: joint 0) */
  const float* skin_w_dev;       /* (V,kmax) that weight (padding: 0) */
} TikLbsModel;
/* bytes of device workspace tik_lbs needs for F frames in `dtype` */
int tik_lbs_workspace_bytes(const TikLbsModel* model, int dtype, int64_t F, int64_t* bytes);
/* joints_dev (F,fk_J,3), local_R_dev / global_R_dev (F,fk_J,3,3): tik_fk_body outputs for the pose, fk_J >= 55 (joints
 * past 54 are ignored); transl_dev (F,3) or NULL.  verts_dev (F,V,3) fp32 out.  joints_out_dev (F,joints_out_J,3) or NULL:
 * posed joints + transl, joints_out_J <= 55 (the first joints_out_J joints) or 55 + n_landmarks (then followed by the
 * landmark vertices).  dtype TIK_F32: 3xTF32 pose blend (1e-4 parity path); TIK_BF16: bf16 operands, fp32 accumulate.
 * Skinning arithmetic is fp32 in both.  workspace_dev 256-byte aligned.  CUDA-graph capturable; F = 0 is a no-op. */
int tik_lbs(const TikLbsModel* model, int dtype, const float* joints_dev, const float* local_R_dev, const float* global_R_dev,
            int fk_J, const float* transl_dev, int64_t F, void* workspace_dev, int64_t workspace_bytes, float* verts_dev,
            float* joints_out_dev, int joints_out_J, void* stream);

/* ------------------------------------------------------------------ body keypoints
 * Replaces the keypoint half of inference.py:70-79 amass_data_to_3d_keypoints and data_amass.py:176-218
 * (run_smpl_inference -> generate_smplx_to_coco_mappings -> gather) without skinning the mesh: one kernel per call,
 * thread per frame, rest skeleton Jt + Jd . betas per frame, FK over the 55 SMPL-X joints, and the landmark points
 * (smplx VertexJointSelector vertices) as pose-blended, linearly skinned vertices.  Points 0..54 are the joints,
 * 55..55+L-1 the landmarks.  Device arrays of a model, packed once by the caller (smpl_util.*.keypoint_pack): */
#define TIK_KP_MAX_BETAS 16
#define TIK_KP_MAX_SELECT 64
typedef struct TikKeypointModel {
  int32_t n_betas;                 /* B in [0, TIK_KP_MAX_BETAS] */
  const float* joint_template_dev; /* (55,3)   J_regressor . v_template */
  const float* joint_dirs_dev;     /* (55,3,B) J_regressor . shapedirs[..., :B]; NULL iff B == 0 */
  int32_t n_landmarks;             /* L in [0, TIK_LBS_MAX_LANDMARKS]: points 55 .. 55+L-1 */
  int32_t kmax;                    /* columns of the landmark skinning table, in [1, 55] when L > 0 */
  const float* lm_template_dev;    /* (L,3) */
  const float* lm_dirs_dev;        /* (L,3,B); NULL iff B == 0 */
  const float* lm_posedirs_dev;    /* (3L,486) row 3l+c, or NULL: no pose blend (rigid landmarks) */
  const int32_t* lm_skin_idx_dev;  /* (L,kmax) joint of each skinning weight (indices outside [0,55) are ignored) */
  const float* lm_skin_w_dev;      /* (L,kmax) that weight (padding: 0) */
} TikKeypointModel;
/* pose_dev (F, pose_J, 3) axis-angle, pose_J in {22, 55, 60} (row pitch; joints >= min(pose_J,55) are identity, 55..59
 * ignored); betas_dev NULL (zero betas), (B) for every frame (betas_per_frame = 0) or (F,B) (betas_per_frame = 1);
 * transl_dev (F,3) or NULL; select_host: n_select in [1, TIK_KP_MAX_SELECT] point indices in [0, 55+L), HOST memory
 * (repeats allowed); out_dev (F, n_select, 3) fp32.  fp32 arithmetic; no workspace; F = 0 is a no-op; CUDA-graph
 * capturable.  Tiles of 64 frames move by bulk copies when every per-frame array is 16-byte aligned. */
int tik_body_keypoints(const TikKeypointModel* m, const float* pose_dev, int pose_J, const float* betas_dev,
                       int betas_per_frame, const float* transl_dev, const int32_t* select_host, int n_select,
                       int64_t F, float* out_dev, void* stream);

/* ------------------------------------------------------------------ keypoint fitting
 * Poses that make tik_body_keypoints hit observed points: per frame f, a few Levenberg-Marquardt steps on
 *   E(theta, tau) = sum_k w_k |kp_k(theta, beta, tau) - y_k|^2 + prior_weight |theta - theta0|^2
 * over theta = the axis-angle rotations of joints 0..21 (joints 22..54 stay identity, as pose_J = 22 gives) and, with
 * fit_transl = 1, the translation tau.  Analytic Jacobian (pose blend of the landmarks included); each iteration solves
 * (H + mu diag(H)) delta = -g with H = J^T W J + prior_weight I, g = J^T W r + prior_weight (theta - theta0) by
 * Cholesky and takes the step iff E drops strictly: mu starts at 1e-3, then mu = max(mu/10, 1e-7) on acceptance and
 * min(mu*10, 1e7) on rejection (a non-positive pivot is a rejection).  n_iter counts solves; E never increases.
 *   m, betas_dev, betas_per_frame, select_host, n_select: as tik_body_keypoints.
 *   target_dev (F, n_select, 3): the points y; weights_dev NULL (all 1), (n_select) (weights_per_frame = 0) or
 *   (F, n_select) (weights_per_frame = 1), non-negative; init_pose_dev (F,22,3): theta0, the start and the prior's
 *   centre; transl_dev (F,3) or NULL (zero): tau's start (fit_transl = 1) or its fixed value (fit_transl = 0);
 *   prior_weight > 0 (keeps the system positive definite); n_iter >= 0.
 *   pose_out_dev (F,22,3); transl_out_dev (F,3) or NULL; cost_dev (F,2) [initial E, final E] or NULL.  A frame whose
 *   initial E is not finite is returned unchanged with final cost NaN.
 * fp32, one warp per frame; frames are independent and a frame's result does not depend on the rest of the call.  No
 * workspace, no host synchronisation, CUDA-graph capturable; F = 0 is a no-op; outputs may not overlap inputs or each
 * other (checked); nothing outside the outputs is written. */
int tik_fit_keypoints(const TikKeypointModel* m, const float* target_dev, const float* weights_dev, int weights_per_frame,
                      const float* init_pose_dev, const float* betas_dev, int betas_per_frame, const float* transl_dev,
                      int fit_transl, const int32_t* select_host, int n_select, float prior_weight, int n_iter, int64_t F,
                      float* pose_out_dev, float* transl_out_dev, float* cost_dev, void* stream);

/* One body shape per sequence and a pose per frame: sequences s = 0..n_seqs-1 packed back to back, sequence s the frames
 * [frame_start[s], frame_start[s+1]), and per sequence Levenberg-Marquardt steps on
 *   E_s = sum_{f in s} [ sum_k w_fk |kp_k(theta_f, beta_s, tau_f) - y_fk|^2 + prior_weight |theta_f - theta0_f|^2 ]
 *         + shape_prior_weight |beta_s|^2
 * over beta_s (the model's B = n_betas >= 1 shape coefficients), theta_f and, with fit_transl = 1, tau_f.  The schedule is
 * tik_fit_keypoints' applied per sequence: mu_s starts at 1e-3, each iteration solves the damped system of all the
 * sequence's unknowns, (H + mu diag(H)) delta = -g, by a Schur complement on the betas (frame blocks in fp32, the B x B
 * system summed and solved in fp64) and takes the step iff E_s drops strictly; a non-positive pivot in any frame block or
 * in the B x B system is a rejection.  n_iter counts solves; E_s never increases.
 *   m, target_dev, weights_dev, weights_per_frame, init_pose_dev, transl_dev, fit_transl, select_host, n_select,
 *   prior_weight, n_iter, F: as tik_fit_keypoints.
 *   frame_start_dev: n_seqs + 1 int64 DEVICE entries (TikSeqBatch): non-decreasing, [0] = 0, [n_seqs] = F, every sequence
 *   at least one frame (n_seqs >= 1 iff F >= 1); indices from a malformed table are clamped into the buffers.
 *   betas_init_dev (n_seqs, B) or NULL (zero): the start of each beta_s; shape_prior_weight > 0 (the prior is centred on
 *   the mean shape, beta = 0).
 *   workspace_dev: 256-byte aligned, workspace_bytes >= tik_fit_keypoints_shape_workspace_bytes (~17 KB per frame).
 *   pose_out_dev (F,22,3); transl_out_dev (F,3) or NULL; betas_out_dev (n_seqs, B); cost_dev (n_seqs, 2) [initial E_s,
 *   final E_s] or NULL.  A sequence whose initial E_s is not finite is returned unchanged with final cost NaN.
 * A sequence's results do not depend on the other sequences of the call or on its position.  No host synchronisation,
 * CUDA-graph capturable; F = 0 is a no-op; outputs may not overlap inputs, the workspace or each other (checked). */
int tik_fit_keypoints_shape_workspace_bytes(const TikKeypointModel* m, int n_select, int fit_transl, int64_t F,
                                            int64_t n_seqs, int64_t* bytes);
int tik_fit_keypoints_shape(const TikKeypointModel* m, const float* target_dev, const float* weights_dev,
                            int weights_per_frame, const float* init_pose_dev, const float* transl_dev, int fit_transl,
                            const int64_t* frame_start_dev, int64_t n_seqs, const float* betas_init_dev,
                            float shape_prior_weight, const int32_t* select_host, int n_select, float prior_weight,
                            int n_iter, int64_t F, void* workspace_dev, int64_t workspace_bytes, float* pose_out_dev,
                            float* transl_out_dev, float* betas_out_dev, float* cost_dev, void* stream);

/* ------------------------------------------------------------------ ST-GCN primitives
 * dtype is TIK_F32 (SIMT fp32, 1e-4 parity path) or TIK_BF16 (tcgen05 tensor cores, fp32 accumulate). */

/* Block-0 graph convolution fused with data_bn, BN and ReLU.
 * Replaces StgGcn18.forward's data_bn + permutes (mmskeleton/models/backbones/st_gcn_aaai18.py:119-125)
 * and the first ConvTemporalGraphical + tcn.0/tcn.1 (gconv_origin.py:56-65, st_gcn_aaai18.py:178-179).
 *   x (N,T,V,Cin) fp32 (the reference's input layout); in_scale/in_shift (V*Cin) folded data_bn;
 *   agg (K,V,V) fp32 = A*importance; w (Cout, K*Cin) fp32 BN-folded; bias (V,Cout) fp32;
 *   out (N,V,T,Cout) dtype, ReLU applied if relu != 0.
 * If res_w_dev != NULL the block's residual branch (1x1 conv stride (s,1) + BN, st_gcn_aaai18.py:198-204)
 * is produced in the same pass: res_out[n,w,t',:] = res_w[w] . x[n, s*t', w, :] with res_w (V,Cout,Cin)
 * fp32 (data_bn scale folded in, constants go to the temporal conv's per-node bias),
 * res_out (N,V,floor((T-1)/s)+1,Cout) dtype. */
int tik_stem_gcn(int dtype, const float* x_dev, const float* in_scale_dev, const float* in_shift_dev,
                 const float* agg_dev, const float* w_dev, const float* bias_dev, void* out_dev,
                 const float* res_w_dev, void* res_out_dev, int res_stride,
                 int64_t N, int T, int V, int Cin, int K, int Cout, int relu, void* stream);

/* Window mode of the stem (SURVEY.md section 8f row 1): the stem reads one resident sequence (frames,V,C); clip n,
 * frame t is sequence frame clamp(n*stride + t + offset, 0, frames-1) -- the edge padding of sample_window
 * (mmskeleton/datasets/data_amass.py:18-42) -- minus the root 0.5*(kp[root_a] + kp[root_b]) of that frame
 * (InferenceDataset, data_amass.py:232-235; root_a < 0: no centring).  A batch of materialised (N,T,V,C) clips is the
 * same read with frames = N*T, offset = 0, stride = T and no root: the library runs every batch that way. */
typedef struct TikWindowing {
  int64_t frames;
  int32_t offset, stride, root_a, root_b;
} TikWindowing;

/* Adjacency aggregation: out[k][(n,w),t,c] = sum_v agg[k][v][w] * x[(n,v),t,c].
 * The einsum 'nkctv,kvw->nctw' of gconv_origin.py:63 moved in front of the 1x1 convolution
 * (SURVEY.md Appendix B).  x (N,V,T,C) dtype -> out (K,N,V,T,C) dtype. */
int tik_aggregate(int dtype, const void* x_dev, const float* agg_dev, void* out_dev,
                  int64_t N, int T, int V, int C, int K, void* stream);

/* Fused graph convolution (tensor cores, bf16, K = 1 partition): aggregation + 1x1 channel GEMM + bias [+ReLU]
 * in one kernel; replaces tik_aggregate + tik_rowgemm for (Cin,Cout) in {(64,64),(64,128),(128,128),(128,256),(256,256)}.
 *   x (N,V,T,Cin) bf16; abd (128,128) bf16 with abd[w*f+t][v*f+t'] = agg[v][w] * (t==t'), f = ceil(T / ceil(T/7)) <= 7
 *   (Cin = 256: f = ceil(T / ceil(T/5)) <= 5), zero elsewhere; w (Cout,Cin) bf16; bias (V,Cout) fp32; out (N,V,T,Cout) bf16. */
int tik_gcn_fused(const void* x_dev, const void* abd_dev, const void* w_dev, const float* bias_dev, void* out_dev,
                  int64_t N, int T, int V, int Cin, int Cout, int relu, void* stream);

typedef struct TikSlab {
  const void* a_dev;  /* source activations, node-major (NV, t_in, c), dtype of the call */
  int32_t c;          /* channels = K-extent contributed by this slab */
  int32_t t_in;       /* frames of the source tensor */
  int32_t t_mul;      /* source frame = t_out * t_mul + t_off; frames outside [0,t_in) read as zero */
  int32_t t_off;
} TikSlab;

#define TIK_ACT_NONE 0
#define TIK_ACT_RELU 1
#define TIK_ACT_LEAKY 2
#define TIK_RES_NONE 0
#define TIK_RES_IDENTITY 1 /* res_dev: node-major (NV,t_out,c_out), dtype of the call */
#define TIK_RES_STEM 2     /* res_dev: raw fp32 input (N,T,V,res_cin); res_w (V,c_out,res_cin) fp32 */
#define TIK_OUT_NODE_MAJOR 0 /* (NV, t_out, c_out) dtype of the call */
#define TIK_OUT_TIME_MAJOR 1 /* (N, t_out, V, c_out) dtype of the call: StgGcn18 output order, st_gcn_aaai18.py:131-133 */
#define TIK_OUT_ROWS_F32 2   /* (NV*t_out, c_out_valid) fp32 */

/* out[row, :] = act( sum_slabs A_s[row_s, :] . W[:, koff_s:koff_s+c_s]^T + bias + residual ).
 * One routine serves the BN-folded 1x1 channel GEMM of ConvTemporalGraphical (gconv_origin.py:59),
 * the (kt x 1) temporal convolution with its residual branch, BN and ReLU
 * (st_gcn_aaai18.py:177-214) as an implicit GEMM, and the two Linear layers of the head
 * (pose_trainer.py:89-92). */
typedef struct TikRowGemm {
  int32_t n_slabs;
  TikSlab slabs[TIK_MAX_SLABS];
  const void* w_dev;     /* (c_out, sum_s c_s) dtype, K contiguous */
  const float* bias_dev; /* (bias_rows, c_out) fp32; bias_rows = V if bias_per_node else 1 */
  int32_t bias_per_node;
  int64_t nv;            /* N*V row groups (for the head: 1) */
  int32_t v;             /* V (for the head: 1) */
  int32_t t_out;         /* output frames per row group (for the head: number of rows) */
  int32_t c_out;         /* rows of W; multiple of 64 for TIK_BF16 */
  int32_t c_out_valid;   /* columns actually stored (<= c_out) */
  int32_t act;
  float slope;
  int32_t res_kind;
  const void* res_dev;
  const float* res_w_dev;
  int32_t res_cin;
  int32_t res_t_mul;     /* TIK_RES_STEM: source frame = t_out * res_t_mul */
  int32_t res_t_in;
  void* out_dev;
  int32_t out_layout;
} TikRowGemm;

int tik_rowgemm(int dtype, const TikRowGemm* desc, void* stream);

/* ------------------------------------------------------------------ whole network
 * Packed (BN/bias/importance-folded) description of PoseRegressor (pose_trainer.py:66-133):
 * StgGcn18 backbone (st_gcn_aaai18.py:32-133) + Linear/LeakyReLU/Linear head. */
typedef struct TikBlock {
  int32_t c_in, c_out, stride, kt, res_kind; /* res_kind: TIK_RES_NONE / IDENTITY / 3 = 1x1 conv folded as a slab / STEM */
  const float* agg_dev;   /* (K,V,V) fp32 */
  const void* w_gcn_dev;  /* (c_out, K*c_in) dtype  [block 0: fp32 always] */
  const float* b_gcn_dev; /* (V, c_out) fp32 */
  const void* w_tcn_dev;  /* (c_out, kt*c_out [+ c_in if res conv]) dtype */
  const float* b_tcn_dev; /* (1 or V, c_out) fp32 */
  const float* w_res_stem_dev; /* (V, c_out, c_in) fp32, block 0 conv residual only */
  int32_t res_as_slab;    /* identity / stem residual folded into w_tcn as a trailing (c_out x c_out) identity block:
                             the plan feeds the residual tensor as one more K-slab (exact in fp32 accumulate) */
} TikBlock;
#define TIK_RES_CONV 3

typedef struct TikNet {
  int32_t V, K, c_in, n_blocks;
  const float* in_scale_dev; /* (V*c_in) */
  const float* in_shift_dev;
  TikBlock blocks[TIK_MAX_BLOCKS];
  int32_t head_hidden, head_out; /* 0 hidden = backbone only */
  const void* w1_dev;  /* (hidden, V*c_last) dtype */
  const float* b1_dev;
  const void* w2_dev;  /* (head_out rounded up to 64 rows for bf16, hidden) dtype */
  const float* b2_dev;
  float leaky_slope;
} TikNet;

/* ------------------------------------------------------------------ weight folding (eval mode)
 * The packing above computed ON THE DEVICE from the reference's raw parameters: BN1 / BN2 / residual-BN scale and shift,
 * convolution biases and A * edge_importance folded into the packed weights (SURVEY.md Appendix B; the algebra of
 * st_gcn_aaai18.py:128-129,177-214 and gconv_origin.py:56-65 in eval mode).  All inputs fp32 device tensors exactly
 * as the reference's state_dict holds them; arithmetic in fp64, rounded once to the output type (identical to the
 * host-side packer engine.PackedNet).  Only enqueues kernels on `stream`. */
typedef struct TikRawBN {     /* an eval-mode BatchNorm: y = (x - mean) / sqrt(var + eps) * weight + bias */
  const float* weight_dev;    /* NULL: 1 */
  const float* bias_dev;      /* NULL: 0 */
  const float* mean_dev;      /* running_mean; NULL together with var_dev: no BatchNorm here (scale 1, shift 0) */
  const float* var_dev;       /* running_var */
  double eps;
} TikRawBN;

typedef struct TikRawBlock {  /* one st_gcn_block of the reference (st_gcn_aaai18.py:136-214) */
  int32_t c_in, c_out, stride, kt;
  int32_t K, V;
  int32_t residual;             /* TIK_RES_NONE / TIK_RES_IDENTITY / TIK_RES_CONV (1x1 conv + BN) */
  const float* A_dev;           /* (K,V,V) backbone buffer A */
  const float* importance_dev;  /* (K,V,V) edge_importance[i], NULL: 1 */
  const float* gcn_w_dev;       /* (K*c_out, c_in)   gcn.conv.weight (1x1) */
  const float* gcn_b_dev;       /* (K*c_out) or NULL gcn.conv.bias */
  TikRawBN bn1;                 /* tcn.0 */
  const float* tcn_w_dev;       /* (c_out, c_out, kt) tcn.2.weight (kt x 1) */
  const float* tcn_b_dev;       /* (c_out) or NULL */
  TikRawBN bn2;                 /* tcn.3 */
  const float* res_w_dev;       /* (c_out, c_in)      residual.0.weight, TIK_RES_CONV only */
  const float* res_b_dev;       /* (c_out) or NULL */
  TikRawBN bn_res;              /* residual.1 */
} TikRawBlock;

typedef struct TikPackBuffers { /* caller-allocated device outputs; sizes from tik_pack_block_bytes */
  float* agg_dev;
  void* w_gcn_dev;
  float* b_gcn_dev;
  void* w_tcn_dev;
  float* b_tcn_dev;
  float* w_res_stem_dev;        /* first block with a conv residual only, else NULL */
} TikPackBuffers;

/* scale / shift (n floats each) of one BatchNorm, e.g. data_bn -> TikNet.in_scale_dev / in_shift_dev (n = V*c_in). */
int tik_pack_bn(const TikRawBN* bn, int64_t n, float* scale_dev, float* shift_dev, void* stream);
/* bytes[6] = sizes of the TikPackBuffers members in declaration order (0 where the member is not produced).
 * first_block != 0: the block that reads the raw input (w_gcn stays fp32, its conv residual is folded with data_bn
 * into w_res_stem / a per-node b_tcn: TIK_RES_STEM). */
int tik_pack_block_bytes(const TikRawBlock* raw, int dtype, int first_block, int64_t* bytes);
/* Folds one block into `buf` and fills `out` (sizes, res_kind, res_as_slab and the pointers of `buf`).
 * data_bn: the backbone's data_bn for the first block (NULL: none), ignored otherwise. */
int tik_pack_block(const TikRawBlock* raw, int dtype, int first_block, const TikRawBN* data_bn,
                   const TikPackBuffers* buf, TikBlock* out, void* stream);

typedef struct TikPlan TikPlan;

/* frames after the strided blocks: T -> floor((T-1)/s)+1 per block (SURVEY.md section 5). */
int tik_stgcn_out_frames(const TikNet* net, int T);
/* bytes of device workspace a plan needs: the backbone runs n_chunk clips at a time (L2-resident layers),
 * the head runs once over up to n_max clips. */
int tik_stgcn_workspace_bytes(const TikNet* net, int dtype, int64_t n_chunk, int64_t n_max, int T, int64_t* bytes);
/* Builds the launch plan (tile shapes, TMA tensor maps over `workspace_dev`).  Host-only work. */
int tik_stgcn_plan_create(const TikNet* net, int dtype, int64_t n_chunk, int64_t n_max, int T, void* workspace_dev,
                          int64_t workspace_bytes, TikPlan** plan);
/* PoseRegressor.forward: x (N,T,V,c_in) fp32 -> poses (N,T',head_out) fp32 (pose_trainer.py:94-133).
 * feat_dev, if not NULL, receives the backbone output (N,T',V*c_last) in the plan dtype
 * (StgGcn18.forward, st_gcn_aaai18.py:113-133).  N may exceed n_chunk and n_max: the backbone
 * processes n_chunk clips at a time and the head n_max clips at a time. */
int tik_stgcn_plan_run(TikPlan* plan, const float* x_dev, int64_t N, float* poses_dev, void* feat_dev,
                       void* stream);
/* Same network over sliding windows of ONE sequence: seq_dev (frames,V,c_in) fp32 replaces the (N,T,V,c_in) batch,
 * n_windows windows of the plan's T frames each (see TikWindowing).  Replaces InferenceDataset + DataLoader +
 * model(...) of inference.py:37-52 without materialising the windows. */
int tik_stgcn_plan_run_windows(TikPlan* plan, const float* seq_dev, const TikWindowing* win, int64_t n_windows,
                               float* poses_dev, void* feat_dev, void* stream);
/* Ragged batch of sequences for the window mode: sequences s = 0..n_seqs-1 packed back to back in one
 * (win->frames, V, c_in) buffer.  Sequence s holds packed frames [frame_start[s], frame_start[s+1]) and windows
 * [window_start[s], window_start[s+1]); window n of sequence s, frame t, reads packed frame
 * frame_start[s] + clamp(n*stride + t + offset, 0, F_s - 1), so the edge padding never reaches a neighbouring sequence.
 * Both tables are DEVICE arrays of n_seqs+1 entries, non-decreasing, [0] = 0; frame_start[n_seqs] = win->frames,
 * window_start[n_seqs] = n_windows.  The library cannot check them without a synchronisation: it clamps the sequence
 * and frame indices it derives from them to the packed buffer, so a malformed table gives wrong values but no read
 * outside it.  Windows come out in sequence order.  inference.sequence_tables builds the tables for the one-window-
 * per-frame rule of forward_windows. */
typedef struct TikSeqBatch {
  int64_t n_seqs;                   /* >= 1 */
  const int64_t* frame_start_dev;   /* (n_seqs+1) */
  const int64_t* window_start_dev;  /* (n_seqs+1) */
} TikSeqBatch;
/* tik_stgcn_plan_run_windows over a ragged batch: poses (n_windows, T', head_out).  Chunks may split sequences. */
int tik_stgcn_plan_run_seq_windows(TikPlan* plan, const float* seq_dev, const TikWindowing* win, const TikSeqBatch* seqs,
                                   int64_t n_windows, float* poses_dev, void* feat_dev, void* stream);
/* Measurement aid (synchronises the stream): one run with CUDA events around every kernel.
 * ms_by_kind[3] / launches_by_kind[3] = {stem, aggregate, implicit-GEMM}; flops_gemm = algorithmic
 * 2*rows*K*c_out summed over the implicit-GEMM launches. */
int tik_stgcn_plan_profile(TikPlan* plan, const float* x_dev, int64_t N, float* poses_dev, void* stream,
                           double* ms_by_kind, int64_t* launches_by_kind, double* flops_gemm);
/* kernels one tik_stgcn_plan_run over N clips launches (for bench.py's gpu_launches). */
int64_t tik_stgcn_plan_launches(const TikPlan* plan, int64_t N);
void tik_stgcn_plan_destroy(TikPlan* plan);

/* ------------------------------------------------------------------ latency plan (BASELINE.json configs[4])
 * The same PoseRegressor.forward for a handful of clips (N * T' <= 32 head rows; e.g. one 64-frame window) as ONE
 * persistent cooperative kernel: every layer is a phase, the 148 resident CTAs meet at a grid-wide barrier between
 * phases, activations stay in L2.  Replaces the 19-25 dependent launches of the throughput plan, which are launch-bound
 * at batch 1 (inference.py:43-52 with DataLoader(batch_size=1); streaming windows).  fp32 arithmetic on the TIK_F32
 * packing of the network (same algebra as the 1e-4 parity path), K = 1 adjacency partition only. */
typedef struct TikLatencyPlan TikLatencyPlan;
int tik_stgcn_latency_workspace_bytes(const TikNet* net, int64_t n_max, int T, int64_t* bytes);
/* Host-only work (+ one small cudaMemcpy of the phase table into the workspace, 256-byte aligned). */
int tik_stgcn_latency_create(const TikNet* net, int64_t n_max, int T, void* workspace_dev, int64_t workspace_bytes,
                             TikLatencyPlan** plan);
/* x (N,T,V,c_in) fp32 -> poses (N,T',head_out) fp32, N <= n_max.  One cooperative launch on `stream`. */
int tik_stgcn_latency_run(TikLatencyPlan* plan, const float* x_dev, int64_t N, float* poses_dev, void* stream);
/* Same over sliding windows of one resident sequence (see TikWindowing / tik_stgcn_plan_run_windows). */
int tik_stgcn_latency_run_windows(TikLatencyPlan* plan, const float* seq_dev, const TikWindowing* win, int64_t n_windows,
                                  float* poses_dev, void* stream);
/* Same over a ragged batch of sequences (see TikSeqBatch), n_windows <= n_max. */
int tik_stgcn_latency_run_seq_windows(TikLatencyPlan* plan, const float* seq_dev, const TikWindowing* win,
                                      const TikSeqBatch* seqs, int64_t n_windows, float* poses_dev, void* stream);
/* number of phases (= grid barriers + 1) of the plan */
int tik_stgcn_latency_phases(const TikLatencyPlan* plan);
void tik_stgcn_latency_destroy(TikLatencyPlan* plan);
/* Probe hook: device buffer of [CTAs = SM count (x TIK_LAT_CTAS_PER_SM)][2 * phases] uint64 receiving %globaltimer (ns)
 * at the start and at the end of every phase's work in every CTA (NULL switches it off).  tools/latency_phases.py. */
int tik_debug_latency_times(TikLatencyPlan* plan, void* dev_buf);

#ifdef __cplusplus
}
#endif
#endif /* TIK_H_ */
