/*
 * dposer_b200 -- C ABI of the B200-native DPoser hot path (libdposer_b200.so).
 *
 * The reference (moonbow721/DPoser) has no FFI layer: its boundary is a set of Python
 * callables (SURVEY.md 8b).  Each entry point below names the reference callable whose
 * arithmetic it replaces (paths relative to the reference checkout); INTEGRATION.md shows
 * the ctypes stub a reference maintainer would add at that call site.
 *
 * Conventions
 *   - extern "C", plain pointers and sizes only; no torch / C++ types cross the boundary.
 *   - every function returns 0 on success or a negative DPB_E* code; dpb_last_error()
 *     returns a thread-local message for the last failure on the calling thread.
 *   - "host" pointers are read during the call; "device" pointers are caller-owned device
 *     buffers (e.g. torch tensors) on the handle's device; nothing is allocated in hot calls:
 *     scratch comes from the caller through (ws, ws_bytes), sized by the *_workspace_bytes query.
 *   - all work is enqueued asynchronously on `stream` (a cudaStream_t passed as void*;
 *     torch.cuda.current_stream().cuda_stream); no entry point synchronises the host.
 *   - model tensors in a handle are immutable after creation and a handle may be used from any host thread;
 *     a score handle also owns the tensor-core engine's per-SM activation scratch, so calls on ONE score
 *     handle must be ordered (same stream, or serialised by events) -- use one handle per concurrent stream.
 *   - there is no CPU fallback: on a machine without a B200-class GPU every compute entry
 *     point fails with DPB_ECUDA.
 */
#ifndef DPOSER_B200_H_
#define DPOSER_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DPB_VERSION 100 /* 0.1.0 */

#define DPB_OK 0
#define DPB_EINVAL (-1)       /* bad argument (maps to ValueError / AssertionError in the Python mirror) */
#define DPB_ECUDA (-2)        /* CUDA runtime / driver failure, or no sm_100 device */
#define DPB_ENOMEM (-3)       /* workspace too small or allocation failure */
#define DPB_EUNSUPPORTED (-4) /* feature not available (maps to NotImplementedError) */

/* network geometry (configs/subvp/amass_scorefc_continuous.py:36-45 + defaults).  A score handle is created for the
 * axis-angle width DPB_POSE_DIM or the rot6d width DPB_POSE_DIM_ROT6D (dpb_score_create_dim). */
#define DPB_POSE_DIM 63
#define DPB_POSE_DIM_ROT6D 126
#define DPB_HIDDEN 1024
#define DPB_EMBED 512
#define DPB_NUM_DENSE 5 /* pre_dense, b1_dense1, b1_dense2, b2_dense1, b2_dense2 */

/* precision / engine selector (flags bits 0..3) */
#define DPB_ENGINE_MASK 0xF
#define DPB_ENGINE_AUTO 0  /* tcgen05 path when t is batch-uniform and B >= 64, else fp32 */
#define DPB_ENGINE_FP32 1  /* fp32 FFMA kernels, fp32 accumulate (exact path, <=2e-5 rel.) */
#define DPB_ENGINE_TC 2    /* tcgen05 tensor cores: fp16 operands (bf16 hi/lo split for the
                              63-wide input layer), fp32 TMEM accumulators (<=1e-3 rel.) */

typedef struct dpb_score dpb_score_t;
typedef struct dpb_lbs dpb_lbs_t;

int dpb_version(void);
const char* dpb_last_error(void);
/* fills sm_count / cc_major / cc_minor of `device`; DPB_ECUDA when there is no usable GPU */
int dpb_device_info(int device, int* sm_count, int* cc_major, int* cc_minor);

/* ------------------------------------------------------------------------------------------
 * Score network  (replaces ScoreModelFC.forward, lib/algorithms/advanced/model.py:141-196,
 * and the score_fn wrapper, lib/algorithms/advanced/utils.py:141-163)
 * ---------------------------------------------------------------------------------------- */
typedef struct {
  /* all HOST fp32 pointers, nn.Linear layout [out, in] row-major; state_dict key in comments */
  const float* pre_w;        /* pre_dense.weight        [1024, D]  (D = the handle's pose width, 63 or 126) */
  const float* pre_b;        /* pre_dense.bias          [1024]       */
  const float* pre_t_w;      /* pre_dense_t.weight      [1024, 512]  */
  const float* pre_t_b;      /* pre_dense_t.bias        [1024]       */
  const float* pre_gn_w;     /* pre_gnorm.weight        [1024]       */
  const float* pre_gn_b;     /* pre_gnorm.bias          [1024]       */
  const float* temb_w;       /* shared_time_embed.0.weight [512,512] */
  const float* temb_b;       /* shared_time_embed.0.bias   [512]     */
  const float* blk_w[4];     /* b1_dense1, b1_dense2, b2_dense1, b2_dense2 .weight [1024,1024] */
  const float* blk_b[4];     /* ... .bias [1024] */
  const float* blk_t_w[4];   /* b{1,2}_dense{1,2}_t.weight [1024,512] */
  const float* blk_t_b[4];   /* ... .bias [1024] */
  const float* blk_gn_w[4];  /* b{1,2}_gnorm{1,2}.weight [1024] */
  const float* blk_gn_b[4];  /* ... .bias [1024] */
  const float* post_w;       /* post_dense.weight [D,1024] */
  const float* post_b;       /* post_dense.bias   [D] */
  const float* emb_freqs;    /* [256] exp(-k ln(1e4)/255) evaluated by the host in fp32 (model.py:41-43) */
} dpb_score_weights;

/* pose_dim = 63 (axis-angle, ScoreModelFC(config, 21, 3)) or 126 (rot6d, ScoreModelFC(config, 21, 6)); any other
 * value: DPB_EUNSUPPORTED.  Every entry point that takes the handle reads D = pose_dim from it; "[B,D]" below means
 * that width. */
int dpb_score_create_dim(dpb_score_t** h, const dpb_score_weights* w, int pose_dim, int device);
/* D of the handle (63 or 126), or DPB_EINVAL for a null handle */
int dpb_score_pose_dim(dpb_score_t* h);
int dpb_score_destroy(dpb_score_t* h);

/* Time path, hoisted (model.py:161-167,174,181 with utils.py:152): for each of n labels
 * (= t*999, fp32, DEVICE) computes temb = SiLU(W_s [sin|cos](label f_k) + b_s) and the five
 * projections W_lt temb + b_lt + b_l.  table is DEVICE fp32 [n, 5, 1024]. */
int dpb_score_time_table(dpb_score_t* h, const float* labels, int n, float* table, void* stream);

size_t dpb_score_workspace_bytes(dpb_score_t* h, int64_t B, int flags);

/* out[B,D] = post_dense(...)(x) * scale.
 *   x         DEVICE fp32 [B,D]
 *   table     DEVICE fp32 [n,5,1024] from dpb_score_time_table
 *   t_index   DEVICE int32 [B] row -> table entry, or NULL (every row uses entry 0)
 *   row_scale DEVICE fp32 [B] or NULL (then `scale` is used for every row).  The caller folds
 *             1/sigmas[floor(label)] (model.py:159,192-194) and -1/std(t) (utils.py:162) here.
 */
int dpb_score_forward(dpb_score_t* h, const float* x, const float* table, const int32_t* t_index,
                      const float* row_scale, float scale, float* out, int64_t B, int flags,
                      void* ws, size_t ws_bytes, void* stream);

/* Forward-mode derivative of dpb_score_forward: out [B,D] as dpb_score_forward, jv [B,D] = (d out / d x) v for a
 * direction v [B,D], with the same row_scale / scale applied to both (t_index NULL: split-fp16 tcgen05 GEMMs; per-row
 * t_index: the fp32 SGEMM path).  Replaces the autograd
 * call of the Hutchinson-Skilling trace estimator in lib/algorithms/advanced/likelihood.py:26-37: the scalar
 * eps . (J eps) it needs is what the reference computes as eps . (J^T eps).  ws: dpb_score_jvp_workspace_bytes. */
size_t dpb_score_jvp_workspace_bytes(dpb_score_t* h, int64_t B);
int dpb_score_jvp(dpb_score_t* h, const float* x, const float* v, const float* table, const int32_t* t_index,
                  const float* row_scale, float scale, float* out, float* jv, int64_t B, void* ws, size_t ws_bytes,
                  void* stream);

/* ------------------------------------------------------------------------------------------
 * Fused PC sampler  (replaces pc_sampler's hot loop, lib/algorithms/advanced/sampling.py:456-461,
 * EulerMaruyamaPredictor.update_fn :182-188, imputation :413-422, RSDE.sde sde_lib.py:98-106)
 * ---------------------------------------------------------------------------------------- */
#define DPB_COEF_STRIDE 8
/* coef[i] = {a, b, c, alpha, std, 0, 0, 0}:  x_mean = a*x + b*raw ;  x = x_mean + c*z ;
 * imputation x = x*(1-m) + (alpha*obs + std*z')*m.  `raw` is the post_dense output BEFORE the
 * sigma division; the host builds a,b,c with the reference's own fp32 torch expressions. */
typedef struct {
  int n_steps;             /* steps executed by this call */
  const float* coef;       /* DEVICE fp32 [n_steps, DPB_COEF_STRIDE] */
  const float* time_table; /* DEVICE fp32 [n_steps, 5, 1024] */
} dpb_step_tables;

#define DPB_SAMPLER_IMPUTE (1 << 4)      /* args.task == 'completion' */
#define DPB_SAMPLER_NOISE_GIVEN (1 << 5) /* consume caller-supplied Gaussian draws (parity mode) */

/*   x_io      DEVICE fp32 [B,D] in: x_T (or z), out: x after the last step
 *   obs,mask  DEVICE fp32 [B,D] (only with DPB_SAMPLER_IMPUTE)
 *   noise     DEVICE fp32: with NOISE_GIVEN, [n_steps, K, B, D] where K=1 (predictor draw) or
 *             K=3 with IMPUTE (draw after corrector, predictor draw, draw after predictor --
 *             the reference's order, sampling.py:459-460).  Otherwise NULL: Philox4x32-10
 *             keyed by (seed, row, step+step_offset, column); see dpb_normal_fill_dim for the layout.
 *   traj      DEVICE fp32 [n_steps,B,D] or NULL;  x_mean DEVICE fp32 [B,D] or NULL.
 */
int dpb_sampler_run(dpb_score_t* h, float* x_io, const dpb_step_tables* tbl, const float* obs,
                    const float* mask, const float* noise, uint64_t seed, uint64_t step_offset,
                    float* traj, float* x_mean, int64_t B, int flags, void* ws, size_t ws_bytes,
                    void* stream);

/* Langevin corrector pieces (sampling.py:282-302) on rows of pose_dim (63 or 126) columns: batch sums of row norms,
 * then the update.
 * sums DEVICE fp32[2] must be zeroed by the caller; norms: sums[0]+=sum_b||grad_b||, sums[1]+=sum_b||noise_b||.
 * update: step = (snr*(sums[1]/Bglobal)/(sums[0]/Bglobal))^2 * 2*alpha ; x_mean = x + step*grad ;
 *         x = x_mean + sqrt(2 step)*noise. */
int dpb_langevin_norms_dim(const float* grad, const float* noise, float* sums, int64_t B, int pose_dim, void* stream);
int dpb_langevin_update_dim(float* x_io, float* x_mean, const float* grad, const float* noise, const float* sums,
                            float snr, float alpha, int64_t B, int pose_dim, void* stream);
/* Predictor-corrector sampling with the Langevin corrector, all n_steps from ONE call (replaces the loop body
 * sampling.py:456-461 with LangevinCorrector.update_fn :282-302 and the predictor of dpb_sampler_run):
 *   score_scale HOST [n]: -1 / (sigma * std) of each step (score = raw * score_scale); lang_alpha HOST [n]: the alpha of
 *   sampling.py:287-291; noise (DPB_SAMPLER_NOISE_GIVEN): DEVICE [n, K+1, B, D], the Langevin draw first, then the K
 *   planes of dpb_sampler_run; otherwise Philox slot 4 serves the corrector.  Batch norms are over the B rows given.
 *   With the tcgen05 engine and at most one 128-row tile per SM (B <= 18 944) all steps run in ONE persistent kernel;
 *   columns 5 and 6 of tbl->coef (DEVICE, spare) are then overwritten with score_scale / lang_alpha. */
size_t dpb_sampler_pc_workspace_bytes(dpb_score_t* h, int64_t B);
int dpb_sampler_run_pc(dpb_score_t* h, float* x_io, const dpb_step_tables* tbl, const float* score_scale,
                       const float* lang_alpha, float snr, const float* obs, const float* mask, const float* noise,
                       uint64_t seed, uint64_t step_offset, float* traj, float* x_mean, int64_t B, int flags, void* ws,
                       size_t ws_bytes, void* stream);
/* fills out [B, pose_dim] with N(0,1) draws of the library's Philox stream.  Draw (row, column c) of (step, slot) is
 * Box-Muller output c % 4 of the Philox4x32-10 block with key = seed and counter = (row lo, row hi, step,
 * slot * DP/4 + c/4), DP = 64 for pose_dim 63 and 128 for 126: every (slot, column) of a row has its own counter.
 * Slots: 0 imputation before the score, 1 predictor, 2 imputation after the predictor, 3 prior-loss z, 4 Langevin. */
int dpb_normal_fill_dim(float* out, int64_t B, uint64_t seed, uint64_t step, int slot, int pose_dim, void* stream);

/* ------------------------------------------------------------------------------------------
 * DPoser prior loss  (replaces DPoserComp.loss run/completion.py:131-149,
 * MotionDenoise.DPoser_loss run/motion_denoising.py:125-143, DPoser.DPoser_loss run/smplify.py:94-107)
 * ---------------------------------------------------------------------------------------- */
/* x_t = alpha*x0 + std*z ; raw = net(x_t) ; x0_hat = (x_t + std^2 * (-raw*inv_sigma_std))/alpha ;
 * loss = sum_all( w (x0-x0_hat)^2 ) / divisor, w = 0.5 or 0.5*sqrt(1+alpha/std) ;
 * grad = 2 w (x0-x0_hat)/divisor  (x0_hat is detached in the reference).
 *   table      DEVICE fp32 [1,5,1024] time table of this t
 *   x0         DEVICE fp32 [B,D]
 *   z          DEVICE fp32 [B,D] Gaussian draw or NULL (Philox with seed/step)
 *   loss_out   DEVICE fp32 [1] (overwritten), grad_out DEVICE fp32 [B,D] or NULL
 *   row_loss   DEVICE fp32 [B] or NULL: per-row sums of w (x0-x0_hat)^2 (for per-problem normalisation)
 */
int dpb_prior_loss(dpb_score_t* h, const float* x0, const float* table, float alpha, float std,
                   float inv_sigma_std, int weighted, float divisor, const float* z, uint64_t seed,
                   uint64_t step, float* loss_out, float* grad_out, float* row_loss, int64_t B,
                   int flags, void* ws, size_t ws_bytes, void* stream);

/* ------------------------------------------------------------------------------------------
 * Linear blend skinning (replaces smplx==0.1.28 lbs()/SMPL.forward/SMPLX.forward as called from
 * lib/body_model/body_model.py:75-88 and lib/body_model/smpl.py:67-78)
 * ---------------------------------------------------------------------------------------- */
typedef struct {
  int V, J, S;                 /* vertices, joints, shape(+expression) components; P = (J-1)*9 */
  const float* v_template;     /* HOST [V,3]    */
  const float* shapedirs;      /* HOST [V,3,S]  */
  const float* posedirs;       /* HOST [P,3V]   */
  const float* J_regressor;    /* HOST [J,V]    */
  const float* lbs_weights;    /* HOST [V,J]    */
  const int32_t* parents;      /* HOST [J], parents[0] = -1, parents[i] < i */
  int n_extra;                 /* extra vertex joints (VertexJointSelector) */
  const int32_t* extra_vids;   /* HOST [n_extra] */
  int n_lmk;                   /* barycentric landmarks (SMPL-X static face landmarks) */
  const int32_t* lmk_faces;    /* HOST [n_lmk,3] vertex ids of each landmark's face */
  const float* lmk_bary;       /* HOST [n_lmk,3] */
} dpb_body_tensors;

#define DPB_LBS_ENGINE_FP32 1 /* fp32 FFMA pose-blend (exact) */
#define DPB_LBS_ENGINE_TC 2   /* tcgen05 pose-blend, fp16 hi/lo-split operands, fp32 accumulate */

#define DPB_LBS_CONST_TAIL (1 << 4) /* dpb_lbs_forward flag: full_pose[:, n_var*3:] equals the declared constant tail */
#define DPB_LBS_NO_SAVE (1 << 5)    /* dpb_lbs_forward flag: forward only -- `ws` will NOT be handed to dpb_lbs_backward,
                                       so the per-pose fp32 transforms / features need not be stored */

int dpb_lbs_create(dpb_lbs_t** h, const dpb_body_tensors* m, int device);
/* Declare that joints n_var..J-1 always carry the same rotation (SMPL-X through lib/body_model/body_model.py with
 * pose_hand / pose_jaw / pose_eye omitted: zeros; through lib/body_model/smpl.py: the model's constant mean hand pose,
 * jaw and eyes zero).  Their pose-blend features (R - I) are then constants: the library folds
 * posedirs[tail]^T . feat(tail) into the template and the blend's K shrinks from S + 9(J-1) to S + 9(n_var-1)
 * (SMPL-X: 506 -> 209).  tail_pose HOST [(J - n_var)*3] axis-angle.  Afterwards dpb_lbs_forward calls that pass
 * DPB_LBS_CONST_TAIL promise full_pose[:, n_var*3:] == tail_pose in every row (the kinematic chain still reads
 * full_pose); calls without the flag are unaffected. */
int dpb_lbs_set_const_tail(dpb_lbs_t* h, int n_var, const float* tail_pose);
int dpb_lbs_destroy(dpb_lbs_t* h);
int dpb_lbs_num_joints_out(dpb_lbs_t* h); /* J + n_extra + n_lmk */
size_t dpb_lbs_workspace_bytes(dpb_lbs_t* h, int64_t B, int flags);

/*   betas DEVICE [B,S], full_pose DEVICE [B,J*3] axis-angle (global_orient first), transl DEVICE [B,3] or NULL
 *   verts DEVICE [B,V,3] or NULL (joints-only: skins only the vertices the extra joints need)
 *   joints DEVICE [B, J+n_extra+n_lmk, 3]
 *   ws keeps the per-pose skinning transforms / rotations needed by dpb_lbs_backward when the same
 *   workspace is handed to it afterwards. */
int dpb_lbs_forward(dpb_lbs_t* h, const float* betas, const float* full_pose, const float* transl,
                    float* verts, float* joints, int64_t B, int flags, void* ws, size_t ws_bytes,
                    void* stream);

/* Vector-Jacobian product of dpb_lbs_forward w.r.t. full_pose, betas, transl.
 *   g_verts DEVICE [B,V,3] or NULL, g_joints DEVICE [B,J+n_extra+n_lmk,3] or NULL
 *   g_pose DEVICE [B,J*3], g_betas DEVICE [B,S], g_transl DEVICE [B,3] (each may be NULL)
 *   scratch DEVICE (optional, dpb_lbs_backward_scratch_bytes(h, B) bytes): with it and g_verts the vertex pass is
 *   split into tensor-core blend recompute + skinning adjoint (dL/dA on tcgen05) + transposed blend on tcgen05;
 *   without it a single slower kernel runs */
size_t dpb_lbs_backward_scratch_bytes(dpb_lbs_t* h, int64_t B);
/* scratch for the joints-only case (g_verts == NULL): the vertices the extra joints / landmarks read take the same
 * tensor-core pass as a small body model of their own; 0 when unavailable (a single slower kernel runs without it) */
size_t dpb_lbs_backward_scratch_bytes_joints(dpb_lbs_t* h, int64_t B);
int dpb_lbs_backward(dpb_lbs_t* h, const float* betas, const float* full_pose, const float* g_verts,
                     const float* g_joints, float* g_pose, float* g_betas, float* g_transl, int64_t B,
                     int flags, void* ws, size_t ws_bytes, void* scratch, size_t scratch_bytes, void* stream);

/* ------------------------------------------------------------------------------------------
 * SMPLify body-fitting loss (replaces body_fitting_loss lib/body_model/fitting_losses.py:59-103 and the
 * helpers it calls: perspective_projection :6-38, gmof :41-47, angle_prior :50-56), forward and cotangents
 * in one pass.  All pointers DEVICE fp32.
 *   joints [B,K,3] (camera translation already applied, as in the reference), joints_2d [B,K,2], conf [B,K],
 *   center [B,2], body_pose [B,pose_dim] or NULL (no angle prior), betas [B,n_betas] or NULL (no shape prior)
 *   focal_b [B] per-image focal lengths or NULL (then the scalar `focal` is used for every image; the reference
 *   assigns K[:,0,0] = focal_length, fitting_losses.py:24-26, so both a float and a [B] tensor are valid there)
 *   loss [B] = sum_k conf^2 GMoF(proj - kp) + w_angle^2 sum exp(+-pose[..])^2 + w_shape^2 sum betas^2
 *   reproj [B,K] or NULL (the per-joint reprojection term, output='reprojection')
 *   g_joints [B,K,3], g_pose [B,pose_dim], g_betas [B,n_betas]: d loss[b] / d input, each may be NULL
 * ---------------------------------------------------------------------------------------- */
int dpb_fit_loss(const float* joints, const float* joints_2d, const float* conf, const float* center,
                 const float* body_pose, int pose_dim, const float* betas, int n_betas, int n_joints,
                 const float* focal_b, float focal, float sigma, float w_angle, float w_shape, float* loss,
                 float* reproj, float* g_joints, float* g_pose, float* g_betas, int64_t B, void* stream);

/* ------------------------------------------------------------------------------------------
 * Fitting-loop steps on the device: everything an Adam step of the reference's task loops does besides the LBS
 * and the prior (run/motion_denoising.py:226-268, run/smplify.py:208-260, run/completion.py:178-203), so that no
 * framework op runs inside a step and a whole step can be captured in one CUDA graph.  All pointers DEVICE fp32.
 * ---------------------------------------------------------------------------------------- */
/* Motion-denoising terms for rows = n_seq * seq_len frames (each sequence an independent problem):
 *   temporal  w_temp * mean_{t < seq_len-1, v} ||verts[t,v] - verts[t+1,v]||   (motion_denoising.py:256-257; rows of
 *             different sequences are never differenced)
 *   data      w_data * mean_{t, j < n_data} ||joints[t,j] - target[t,j]||, dropped for a sequence whose term is not
 *             > 0 (the reference's NaN guard `if data_term > 0`, :262, as a per-sequence device predicate)
 * Writes the cotangents g_verts [rows,V,3] and g_joints [rows,n_out,3] (zero beyond n_data) of the weighted sum.
 * seq_terms [n_seq,2] (optional, reporting): unweighted temporal and data term of each sequence. */
int dpb_motion_loss(const float* verts, const float* joints, const float* target, int64_t rows, int seq_len, int V,
                    int n_out, int n_data, float w_temp, float w_data, float* g_verts, float* g_joints,
                    float* seq_terms, void* stream);
/* camera_fitting_loss (lib/body_model/fitting_losses.py:106-136): loss [B] = reprojection of the four torso joints
 * (OpenPose slots when all four are confident, else the GT slots) + depth_weight^2 (t_z - t_z,est)^2, with the
 * cotangents g_joints [B,K,3] and g_cam_t [B,3] (either may be NULL).  focal_b [B] or NULL as in dpb_fit_loss. */
int dpb_camera_fit_loss(const float* joints, const float* joints_2d, const float* conf, const float* center,
                        const float* cam_t, const float* cam_t_est, const float* focal_b, float focal,
                        float depth_weight, int n_joints, float* loss, float* g_joints, float* g_cam_t, int64_t B,
                        void* stream);
/* torch.optim.Adam step `step` (1-based; amsgrad off, no weight decay) on a strided [rows, cols] parameter view with
 * state m, v [rows*cols]:  grad = s1 g1 + s2 col_scale2[c] g2 + s3 g3  (g2, col_scale2, g3 may be NULL). */
int dpb_adam_step(float* param, int64_t ld_p, float* m, float* v, const float* g1, int64_t ld1, float s1,
                  const float* g2, int64_t ld2, float s2, const float* col_scale2, const float* g3, int64_t ld3,
                  float s3, int64_t rows, int cols, float lr, float beta1, float beta2, float eps, int step,
                  void* stream);
/* grad = d/dx mean((x*mask - obs*mask)^2) = 2 mask^2 (x - obs) / n   (the data term of run/completion.py:197) */
int dpb_masked_mse_grad(const float* x, const float* obs, const float* mask, float* grad, int64_t n, void* stream);
/* Posenormalizer z-score (lib/dataset/AMASS.py:187-259): out = (x - mean) / std per column, or x * std + mean (inverse),
 * on strided views (row strides ldx, ldo).  squash > 0 first maps x -> tanh(squash * x): benchmarks with random-init
 * score weights use it to bring the sampler's output into a plausible angle range before the body model. */
int dpb_affine_cols(const float* x, int64_t ldx, const float* mean, const float* std, float* out, int64_t ldo,
                    int64_t rows, int cols, int inverse, float squash, void* stream);
/* The input of a rot6d (126-D) prior from axis-angle poses: Posenormalizer.offline_normalize(poses, from_axis=True)
 * (run/smplify.py:109-115, with axis_angle_to_rot6d of lib/utils/transforms.py:237-255), on strided views.  For joint j
 * of row r, a = x[r*ldx + 3j .. 3j+2] and R = I + (sin t / t)[a]x + ((1 - cos t) / t^2)[a]x^2 (t = |a|):
 *   out[r*ldo + 6j + k] = (rot6d_k - mean[6j+k]) / std[6j+k],   rot6d = (R00, R01, R10, R11, R20, R21).
 * mean / std [6 n_joints] express every rule of the normaliser: z-score; min-max as mean = (lo + hi) / 2,
 * std = (hi - lo) / 2; no normalisation as 0 / 1.  The map is smooth through t = 0 (series below t = 1.2, see
 * fitstep.cu); a non-finite coordinate gives NaN in that joint's 6 outputs only. */
int dpb_axis_to_rot6d_cols(const float* x, int64_t ldx, const float* mean, const float* std, float* out, int64_t ldo,
                           int64_t rows, int n_joints, void* stream);
/* Its vector-Jacobian product: g_x[r*ldgx + 3j + i] = sum_k (g[r*ldg + 6j+k] / std[6j+k]) d rot6d_k / d a_i, recomputed
 * from x (nothing is saved by the forward); NaN in a joint's 3 entries when its input is non-finite. */
int dpb_axis_to_rot6d_cols_vjp(const float* x, int64_t ldx, const float* std, const float* g, int64_t ldg, float* g_x,
                               int64_t ldgx, int64_t rows, int n_joints, void* stream);
/* The other way, the body pose of a rot6d (126-D) network's normalised output:
 * Posenormalizer.offline_denormalize(x, to_axis=True) (lib/utils/transforms.py:197-234), on strided views.  For joint j
 * of row r, u = x[r*ldx + 6j .. 6j+5] * std[6j..] + mean[6j..] and
 *   out[r*ldo + 3j .. 3j+2] = rot6d_to_axis_angle(u):
 * Gram-Schmidt of the columns a1 = (u0, u2, u4), a2 = (u1, u3, u5) into R = [b1 b2 b3], Shepperd's quaternion (pivot:
 * the largest of trace / R00 / R11 / R22), then 2 atan2(|v|, w) v / |v| (2 v for |v| < 1e-12); the angle is in [0, pi].
 * mean / std [6 n_joints] as in dpb_axis_to_rot6d_cols.  Degenerate joints -- |a1| or |a2 - (b1.a2) b1| below 1e-12
 * (F.normalize's clamp) -- non-finite inputs and non-finite results give 0 in the joint's 3 outputs. */
int dpb_rot6d_to_axis_cols(const float* x, int64_t ldx, const float* mean, const float* std, float* out, int64_t ldo,
                           int64_t rows, int n_joints, void* stream);
/* Its vector-Jacobian product: g_x[r*ldgx + 6j + k] = sum_i g[r*ldg + 3j+i] d out_i / d x_k, recomputed from x (nothing
 * is saved by the forward); 0 in a joint's 6 entries wherever the forward gives 0 by the rule above, or the result is
 * not finite. */
int dpb_rot6d_to_axis_cols_vjp(const float* x, int64_t ldx, const float* mean, const float* std, const float* g,
                               int64_t ldg, float* g_x, int64_t ldgx, int64_t rows, int n_joints, void* stream);
/* out[r,c] = w0 x[r-1,c] + w1 x[r,c] + w2 x[r+1,c] inside each sequence of seq_len rows, zero-padded at its ends
 * (gaussian_smoothing(window_size=3), lib/utils/misc.py:84-95, per sequence as in run/motion_denoising.py:281-285);
 * keep_ends != 0 copies the first and last row of every sequence instead.  out must not alias x. */
int dpb_seq_smooth3(const float* x, float* out, int64_t rows, int seq_len, int cols, float w0, float w1, float w2,
                    int keep_ends, void* stream);
/* joints[:, joint_map] (lib/body_model/smpl.py:70) and its adjoint (g_in is overwritten; repeated map entries add) */
int dpb_joint_map_gather(const float* joints, int n_in, const int32_t* map, int n_map, float* out, int64_t B,
                         void* stream);
int dpb_joint_map_scatter(const float* g_out, int n_map, const int32_t* map, int n_in, float* g_in, int64_t B,
                          void* stream);

/* ------------------------------------------------------------------------------------------
 * Probability-flow ODE on the device (replaces scipy.integrate.solve_ivp(method='RK45') as driven by
 * lib/algorithms/advanced/likelihood.py:93-101 and sampling.py:520-524): Dormand-Prince stages and error norm on DEVICE
 * vectors, fp64 state, fp32 stage derivatives k [7, n]; the host keeps scipy's step-size controller and reads one scalar
 * per attempted step.
 * ---------------------------------------------------------------------------------------- */
/* stage 1..5: y + h sum_j a[stage][j] k_j;  stage 6: the 5th-order solution y + h sum_j b_j k_j.
 * y_out DEVICE fp64 [n] and / or x_out DEVICE fp32 [nx] (the first nx entries, the network's input), either may be NULL */
int dpb_rk45_stage(const double* y, const float* k, int64_t n, double h, int stage, double* y_out, float* x_out,
                   int64_t nx, void* stream);
/* ((double*)scratch)[0] = sum_i (h sum_j e_j k_j[i] / (atol + rtol max(|y_i|, |y_new_i|)))^2, fixed summation order */
size_t dpb_rk45_scratch_bytes(void);
int dpb_rk45_error(const double* y, const double* y_new, const float* k, int64_t n, double h, double rtol, double atol,
                   void* scratch, void* stream);
/* k_out[b,c] = fx x - 0.5 g2 score (drift of the reverse ODE, sde_lib.py:98-106 with probability_flow) and, with jv / eps,
 * k_out[B*D + b] = fx sum_c eps^2 - 0.5 g2 sum_c jv eps (Hutchinson divergence, likelihood.py:26-37); x, score, jv, eps
 * [B,D] with D = pose_dim (63 or 126; any other value: DPB_EUNSUPPORTED, checked before the arguments) */
int dpb_pf_ode_rhs_dim(const float* x, const float* score, const float* jv, const float* eps, float fx, float g2,
                       float* k_out, int64_t B, int pose_dim, void* stream);

/* ------------------------------------------------------------------------------------------
 * Training step of the score network (replaces loss_fn + loss.backward() + optimize_fn + ema.update of
 * lib/algorithms/advanced/losses.py:31-57,61-137,187-275 with model.py:141-196 in train mode and
 * lib/algorithms/ema.py:35-50).  Every contraction of the forward and backward pass is a split-fp16 tcgen05 GEMM.
 * ---------------------------------------------------------------------------------------- */
typedef struct dpb_train dpb_train_t;
/* the fields of dpb_score_weights, but DEVICE fp32 pointers: parameters (read) or their gradients (written).
 * emb_freqs (parameters only) = DEVICE [256]. */
typedef dpb_score_weights dpb_train_tensors;

/* scratch for steps of exactly `batch` rows (activations, cotangents, fp16 operand copies) of a network of width
 * pose_dim = 63 (axis-angle) or 126 (rot6d); any other value: DPB_EUNSUPPORTED, before any device is touched.  "[B,D]"
 * below means that width. */
int dpb_train_create_dim(dpb_train_t** h, int64_t batch, int pose_dim, int device);
int dpb_train_destroy(dpb_train_t* h);
/* loss = mean_b row_w[b] sum_k (res_c[b] res[b,k] + z_c[b] z[b,k])^2 on perturbed = mean_c x + std_c z, where res is the
 * network's post_dense output at the per-row label (losses.py:108-131; the sigma / std divisions and the reduce_mean /
 * likelihood-weighting factors are folded into the row scalars by the host).
 *   params    DEVICE parameter pointers;  grads  DEVICE gradient pointers (every one overwritten) or NULL = loss only
 *   batch     DEVICE fp32 [B,D] clean (normalised) poses
 *   rows      DEVICE fp32 [6,B]: label (= 999 t), mean_c, std_c, res_c, z_c, row_w
 *   z_given   DEVICE fp32 [B,D] Gaussian draws (parity mode) or NULL: Philox4x32-10 keyed by (seed, row, column quad)
 *   mask_given DEVICE uint8 [5,B,1024] dropout keep-masks in layer order (parity mode) or NULL: Philox
 *   drop_p    dropout probability (0 = eval mode)
 *   loss      DEVICE fp32 [1];  loss_rows DEVICE fp32 [B] or NULL */
int dpb_train_loss_grad(dpb_train_t* h, const dpb_train_tensors* params, const dpb_train_tensors* grads,
                        const float* batch, const float* rows, const float* z_given, const uint8_t* mask_given,
                        float drop_p, uint64_t seed, float* loss, float* loss_rows, void* stream);
/* The two halves of dpb_train_loss_grad on their own, for losses that chain several network evaluations under the
 * optimiser (the auxiliary loss: multi_step_denoise of losses.py:91-106 feeding the body model, :244-258).  One handle holds
 * the activations of ONE evaluation: forward stores them, backward consumes them (same mask / drop_p / seed).
 *   x DEVICE [B,D] network input, labels DEVICE [B] (= 999 t), res DEVICE [B,D] post_dense output (before the sigma division)
 *   g_res DEVICE [B,D] cotangent of res; accumulate != 0 adds to the gradients instead of overwriting them;
 *   g_x DEVICE [B,D] cotangent of x, or NULL */
int dpb_train_forward(dpb_train_t* h, const dpb_train_tensors* params, const float* x, const float* labels,
                      const uint8_t* mask_given, float drop_p, uint64_t seed, float* res, void* stream);
int dpb_train_backward(dpb_train_t* h, const dpb_train_tensors* params, const dpb_train_tensors* grads, const float* g_res,
                       const uint8_t* mask_given, float drop_p, uint64_t seed, int accumulate, float* g_x, void* stream);
/* out[b,c] = a[b] x[b,c] + b[b] y[b,c] (y may be NULL): the affine steps of the DDIM chain and their adjoints */
int dpb_rows_axpby(const float* a, const float* x, const float* b, const float* y, float* out, int cols, int64_t B,
                   void* stream);
/* loss[0] = scale sum_b w[b] sum_i (p[b,i] - q[b,i])^2, grad_q = -2 scale w[b] (p - q) (optional): the weighted v2v / j2j
 * terms of losses.py:253-254; row_scratch DEVICE fp32 [B] */
int dpb_weighted_sqdiff(const float* p, const float* q, const float* w, int64_t B, int64_t n, float scale, float* loss,
                        float* grad_q, float* row_scratch, void* stream);
/* C[M,N] = A[M,K] B[N,K]^T (+ bias[n]) on the split-fp16 tcgen05 GEMM the training step is built from (DEVICE fp32,
 * row-major, ~1e-6 relative); utility / unit-test entry, the operands are converted on every call */
size_t dpb_gemm_nt_workspace_bytes(int M, int N, int K);
int dpb_gemm_nt(const float* A, const float* B, const float* bias, float* C, int M, int N, int K, void* ws,
                size_t ws_bytes, void* stream);
/* scratch for the two calls below (DEVICE, any contents) */
size_t dpb_train_adam_scratch_bytes(void);
/* ((double*)scratch)[0] = sum of squares of a flat gradient buffer, added in a fixed order */
int dpb_train_grad_norm(const float* g, int64_t n, void* scratch, void* stream);
/* torch.optim.Adam's update on flat buffers (losses.py:31-41), preceded by torch.nn.utils.clip_grad_norm_ when
 * grad_clip >= 0 (losses.py:53-54): the clip coefficient is evaluated on the device, no host synchronisation.
 * `lr` already contains the warm-up factor (losses.py:50-52); step >= 1 is Adam's own step count. */
int dpb_train_adam(float* p, const float* g, float* m, float* v, int64_t n, float lr, float beta1, float beta2,
                   float eps, float weight_decay, int64_t step, float grad_clip, const float* hyper_dev, void* scratch,
                   void* stream);
/* hyper_dev (optional, for CUDA-graph replay): DEVICE fp32 [2] = { lr / (1 - beta1^step), 1 / sqrt(1 - beta2^step) }
 * read by the kernel instead of the values derived from lr / step on the host */
/* shadow -= one_minus_decay * (shadow - p)   (ExponentialMovingAverage.update, ema.py:35-50) */
int dpb_ema_update(float* shadow, const float* p, int64_t n, float one_minus_decay, const float* omd_dev, void* stream);
/* omd_dev (optional): DEVICE fp32 [1] read instead of one_minus_decay.  dpb_train_set_seed_pointer: the Philox seed of
 * dpb_train_loss_grad is read from DEVICE memory from now on (NULL switches back to the argument) -- with both, a
 * captured CUDA graph of one training step can be replayed with fresh draws and schedule values. */
int dpb_train_set_seed_pointer(dpb_train_t* h, const uint64_t* seed_dev);

/* ------------------------------------------------------------------------------------------
 * Metrics (replaces average_pairwise_distance lib/utils/metric.py:8-37 and the per-sample
 * reductions of Evaler.eval_bodys lib/dataset/AMASS.py:275-298)
 * ---------------------------------------------------------------------------------------- */
/* row_sums[i - row0] = sum over j in [0,B), j != i of mean_k ||joints[i,k]-joints[j,k]||  for i in [row0,row0+nrows).
 * row_sums DEVICE fp32[nrows] (overwritten; no atomics, deterministic).  APD = sum(row_sums over all rows) / (B(B-1));
 * the caller adds the rows in double precision. */
int dpb_apd_partial(const float* joints, int64_t B, int n_joints, int64_t row0, int64_t nrows,
                    float* row_sums, void* stream);
/* out[b] = 1000 * mean_{k in idx} ||a[b,idx[k]] - c[b,idx[k]]||  (idx DEVICE int32[n_idx] or NULL = all) */
int dpb_mean_point_error(const float* a, const float* c, int64_t B, int n_points, const int32_t* idx,
                         int n_idx, float* out, void* stream);

/* Procrustes-aligned point error, PA-MPJPE / PA-MPVPE (replaces compute_similarity_transform / reconstruction_error
 * of lib/utils/transforms.py, numpy on the CPU, one sample at a time).  Per row: the similarity transform (scale s,
 * proper rotation R, translation t) minimising sum_k ||s R s1[k] + t - s2[k]||^2 over the points idx selects (all
 * when idx is NULL), fitted in fp64, and err = mean over those points of ||s R s1[k] + t - s2[k]|| (the full rule:
 * dposer_b200/metric.py).  Deterministic; no host synchronisation (graph-capturable).
 *   s1, s2   DEVICE fp32 [B, n_points, 3] (prediction, target);
 *   idx      DEVICE int32 [n_idx] or NULL; entries are not range-checked here;
 *   err      DEVICE fp32 [B], in the input's units; NaN for a row whose selected points hold a non-finite
 *            coordinate, or whose selected predicted points all coincide (n_idx == 1 included);
 *   aligned  DEVICE fp32 [B, n_points, 3] or NULL: s R s1[k] + t for every point;
 *   params   DEVICE fp32 [B, 13] or NULL: s, R (row-major), t.  NaN rows are NaN throughout. */
int dpb_procrustes(const float* s1, const float* s2, int64_t B, int n_points, const int32_t* idx, int n_idx,
                   float* err, float* aligned, float* params, void* stream);

/* Self-intersection metric (replaces self_intersections_percentage lib/utils/metric.py:41-89, pymeshlab on the CPU).
 * A pair of distinct faces intersects according to s, the number of vertex ids they share: s = 0 the closed triangles
 * have a common point; s = 1 the edge opposite the shared vertex, moved halfway to it, crosses the other face's open
 * interior (either way round); s = 2 never; s = 3 always; a zero-area face never.  A face is selected when it is in an
 * intersecting pair; SI = 100 * selected / n_faces.  Every decision is the sign of an fp64 expression of the fp32
 * inputs (the full rule: dposer_b200/metric.py).  Deterministic; no host synchronisation (graph-capturable).
 *   create: faces HOST int32 [n_faces,3], every id in [0, n_vertices) (DPB_EINVAL otherwise), uploaded once;
 *           n_faces > 32768: DPB_EUNSUPPORTED.  One handle serves any number of meshes of that topology.
 *   run:    vertices DEVICE fp32 [B, n_vertices, 3] (e.g. dpb_lbs_forward's verts);
 *           counts DEVICE int32 [B]: selected faces of each mesh, -1 when a face references a non-finite vertex;
 *           selection DEVICE uint8 [B, n_faces] (1 = selected, all 0 for a non-finite mesh) or NULL;
 *           ws DEVICE, dpb_selfisect_workspace_bytes(h, B) bytes, any contents. */
typedef struct dpb_selfisect dpb_selfisect_t;
int dpb_selfisect_create(dpb_selfisect_t** h, const int32_t* faces, int n_faces, int n_vertices, int device);
int dpb_selfisect_destroy(dpb_selfisect_t* h);
size_t dpb_selfisect_workspace_bytes(dpb_selfisect_t* h, int64_t B);
int dpb_selfisect_run(dpb_selfisect_t* h, const float* vertices, int64_t B, int32_t* counts, uint8_t* selection,
                      void* ws, size_t ws_bytes, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* DPOSER_B200_H_ */
