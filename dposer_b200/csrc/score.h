// Internal layout of the score-network handle (not part of the C ABI).
#pragma once
#include <cuda.h>

#include "common.cuh"

struct dpb_score {
  int device = 0;
  int sm_count = 0;
  int pose_dim = 63, pose_dp = 64;   // pose width D of this network (63 or 126) and its padded width DP (64 or 128)
  // ---- fp32 parameters on the device (exact engine + time path)
  float* pre_w = nullptr;       // [1024, DP]  (K padded D -> DP with zeros)
  float* blk_w[4] = {};         // [1024, 1024]
  float* post_w = nullptr;      // [DP, 1024]  (N padded D -> DP with zero rows)
  float* post_b = nullptr;      // [DP]
  float* lin_b[5] = {};         // pre_b, blk_b[0..3]            [1024]
  float* t_w[5] = {};           // pre_t_w, blk_t_w[0..3]        [1024, 512]
  float* t_b[5] = {};           // pre_t_b, blk_t_b[0..3]        [1024]
  float* gn_w[5] = {};          // pre_gn_w, blk_gn_w[0..3]      [1024]
  float* gn_b[5] = {};
  float* temb_w = nullptr;      // [512, 512]
  float* temb_b = nullptr;      // [512]
  float* emb_freqs = nullptr;   // [256]
  float* gn_packed = nullptr;   // [5][2][1024] gamma|beta, contiguous (tcgen05 epilogue staging)
  // ---- tensor-core operands
  __half* w16[4] = {};          // fp16 copies of blk_w          [1024, 1024]
  __half* post16 = nullptr;     // fp16 copy of post_w           [DP, 1024]
  __nv_bfloat16* pre_split = nullptr;  // [1024, 3 DP] = [hi | hi | lo] bf16 split of pre_w (K-extension)
  CUtensorMap tm_w[4];          // box {64 (K), 256 (N)} over w16[l]
  CUtensorMap tm_post;          // box {64, DP / 2}
  CUtensorMap tm_pre;           // box {64, 256} over pre_split
  bool tc_ready = false;
  // TC scratch owned by the handle (sized by the grid, not by B): activations + x operand per CTA slot
  __half* act_h = nullptr;      // [slots*128, 1024] residual stream
  __half* act_t = nullptr;      // [slots*128, 1024] block intermediate
  CUtensorMap tm_act_h, tm_act_t;  // box {64, 128}
  float* pc_buf = nullptr;      // predictor-corrector mode: [2 * PC_MAX_STEPS] batch norm sums + one int barrier counter
  int tc_slots = 0;
  float* gn_tc = nullptr;       // [5][2][1024] gamma | beta as staged by the tcgen05 epilogue
  int* tc_flags = nullptr;      // [slots] hand-off flags of the sampler's segment schedule (score_tc.cu: SegIter)
  void* jvp_ops = nullptr;      // fp16 [hi | lo] weight operands of the tensor-core JVP (jvp_tc.cu), built on first use
};

namespace dpb {

// ---- fp32 engine (score_simt.cu)
int simt_time_table(dpb_score* h, const float* labels, int n, float* table, cudaStream_t st);
size_t simt_forward_ws_bytes(int64_t B, int dp = DP);
// raw[B,DP] = post_dense output (columns D.. are padding); buffers carved from ws
int simt_forward_jvp_raw(dpb_score* h, const float* x, const float* v, const float* table, const int32_t* t_index,
                         float* raw, int64_t B, void* ws, size_t ws_bytes, cudaStream_t st);
int simt_forward_raw(dpb_score* h, const float* x, const float* table, const int32_t* t_index, float* raw,
                     int64_t B, void* ws, size_t ws_bytes, cudaStream_t st);

// ---- tcgen05 engine (score_tc.cu)
int tc_prepare(dpb_score* h, const dpb_score_weights* w);   // fp16/bf16 operand copies, tensor maps, scratch
void tc_release(dpb_score* h);

struct TcJob {
  // mode 0: forward  out = raw*scale (row_scale optional)      mode 1: sampler      mode 2: prior loss
  int mode;
  int64_t B;
  const float* x_in;        // forward / prior: x [B,D]
  float* x_io;              // sampler state
  const float* table;       // [n_steps,5,1024]
  const float* coef;        // [n_steps,8] (sampler)
  int n_steps;
  const float* row_scale; float scale; float* out;       // forward
  const float* obs; const float* mask; const float* noise; int noise_k;  // sampler
  uint64_t seed; uint64_t step_offset; float* traj; float* x_mean; int impute;
  // prior loss
  float alpha, std, inv_sigma_std, divisor; int weighted; const float* z; float* loss_out; float* grad_out;
  float* row_loss;
  // predictor-corrector (Langevin) sampling fused into the sampler kernel: coef columns 5 / 6 carry score scale / alpha
  int pc; float snr;
};
int tc_launch(dpb_score* h, const TcJob& job, cudaStream_t st);
bool tc_pc_possible(const dpb_score* h, int64_t B, int n_steps);

}  // namespace dpb
