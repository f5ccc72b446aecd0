// Internal layout of the LBS handle (not part of the C ABI).
#pragma once
#include <cuda.h>
#include <cuda_fp16.h>

#include <vector>

#include "common.cuh"

// A blend basis as the tcgen05 engine reads it: row (c*V_pad + v) = [shape dirs | pose dirs of joints 1..n_var-1 |
// template] as fp16 [hi | lo].  The FULL variant has n_var = J; a CONST-TAIL variant folds the (constant) pose-blend
// contribution of joints n_var..J-1 into the template slot, so K shrinks from S + 9(J-1) + 1 to S + 9(n_var-1) + 1.
struct LbsVariant {
  int n_var = 0;            // joints whose rotation varies per pose
  int p_feat = 0;           // pose features in the blend K: 9 * (n_var - 1)
  int kext = 0;             // [hi | lo] width, multiple of 64
  __half* dirs16 = nullptr; // [3*V_pad, kext]
  CUtensorMap tm_dirs;      // box {64, 128}
};

struct dpb_lbs {
  int device = 0;
  int sm_count = 0;
  int V = 0, J = 0, S = 0, P = 0, n_extra = 0, n_lmk = 0, n_out = 0;
  int max_depth = 0;
  int nnz = 0;                    // ELL width of the skinning weights
  std::vector<int> parents_h;
  // device tensors
  float* v_template = nullptr;    // [V,3]
  float* shapedirs = nullptr;     // [V,3,S]
  float* posedirs = nullptr;      // [P,3V]
  float* j_template = nullptr;    // [J,3]     J_regressor . v_template
  float* j_shapedirs = nullptr;   // [J,3,S]   J_regressor . shapedirs
  float* j_shapedirsT = nullptr;  // [S, 3J]   the same, transposed: lanes walk (joint, coordinate) pairs contiguously
  int32_t* parents = nullptr;     // [J]
  int32_t* depth = nullptr;       // [J]
  int32_t* child_ptr = nullptr;   // [J+1]  CSR of each joint's children (the backward sweep pulls instead of using atomics)
  int32_t* child_idx = nullptr;   // [J-1]
  int32_t* ell_idx = nullptr;     // [nnz,V]
  float* ell_w = nullptr;         // [nnz,V]
  int32_t* extra_vids = nullptr;  // [n_extra]
  int32_t* lmk_faces = nullptr;   // [n_lmk,3]
  float* lmk_bary = nullptr;      // [n_lmk,3]
  // joints-only mode: compact list of the vertices the extra joints / landmarks need
  int n_need = 0;
  int32_t* need_vids = nullptr;   // [n_need] sorted unique vertex ids
  int32_t* extra_pos = nullptr;   // [n_extra] position of extra_vids[i] in need_vids
  int32_t* lmk_pos = nullptr;     // [n_lmk,3]
  int32_t* need_index = nullptr;  // [V] position in need_vids or -1
  // tensor-core pose-blend operands (lbs_tc.cu)
  bool tc_ready = false;
  int kext = 0;                   // extended K (multiple of 64)
  __half* dirs16 = nullptr;       // [3V_pad, kext] K-major fp16 hi/lo-split blend basis
  CUtensorMap tm_dirs;
  int n_cols_pad = 0;
  int jp = 0;                     // joints padded to 32
  __half* wop16 = nullptr;        // [V_pad, 2*jp] fp16 [hi | lo] skinning weights
  CUtensorMap tm_wop;
  LbsVariant tailv;               // const-tail variant (dpb_lbs_set_const_tail), dirs16 == nullptr until declared
  // backward: transposed-blend GEMM operand (lbs_bwd.cu)
  int bw_np = 0, bw_kp = 0;       // (P+S) padded to 64, 3V padded to 16
  float* dirs_pad = nullptr;      // [bw_np, bw_kp] fp32: rows 0..P-1 posedirs, rows P..P+S-1 shapedirs^T, zero padding
  // backward: the same operand for the tcgen05 transposed blend (lbs_bwd_tc.cu)
  bool bt_ready = false;
  int bt_rp = 0, bt_kp = 0;       // 3V padded to 64; feature rows padded to 256 / 512
  __half* basisT16 = nullptr;     // [bt_kp, 2*bt_rp] fp16 [hi | lo]
  CUtensorMap tm_bT;
  // backward: skinning adjoint with dL/dA on tcgen05 (lbs_skin_bwd_tc.cu)
  bool sb_ready = false;
  int sb_vp = 0, sb_smem = 0;     // V padded to 64; dynamic shared memory of the kernel
  __half* wT16 = nullptr;         // [128, 2*sb_vp] fp16 [hi | lo]: rows < J = weights^T, row J = ones
  CUtensorMap tm_wT;
  int32_t* csr_ptr = nullptr;     // [J+1] per-joint vertex lists of the sparse weights (V <= 1024: compact sets)
  int32_t* csr_v = nullptr;
  float* csr_w = nullptr;
  // joints-only mode on the tensor cores: the n_need vertices the extra joints / landmarks read, as a body model of
  // their own (same joints, shape and pose spaces; vertex i = need_vids[i]) -- every vertex kernel runs on it unchanged
  dpb_lbs* sub = nullptr;
};

namespace dpb {
// per-pose workspace layout shared by forward and backward
struct LbsWs {
  float* A;       // [B,J,12]  skinning transforms (rotation | translation)
  float* feat;    // [B,P]     pose feature (R - I), joints 1..J-1
  float* G;       // [B,J,12]  global transforms (kept for backward)
  float* jrest;   // [B,J,3]
  float* compact; // [B,n_need,3] (joints-only mode)
  // backward scratch
  float* gA;      // [B,J,12]   dL/dA
  float* gfeat;   // [B,P]      dL/dfeat
  float* gextra;  // [B,n_need,3] joint grads scattered onto the vertices that produce them
  float* gbeta;   // [B,S+3]    vertex-path part of dL/dbetas | dL/dtransl
  __half* featop; // [B_pad, kext] fp16 [hi | lo] blend operand of the tcgen05 engine (nullptr if unavailable)
  __half* skinop; // [B_pad*12, 2*jp] fp16 [hi | lo] per-pose transform operand of the tcgen05 skinning
};
size_t lbs_ws_bytes(const dpb_lbs* h, int64_t B, bool compact);
bool lbs_carve(const dpb_lbs* h, int64_t B, bool compact, void* ws, size_t ws_bytes, LbsWs* out);
size_t lbs_tc_ws_bytes(const dpb_lbs* h, int64_t B);
int lbs_tc_blend(dpb_lbs* h, const LbsVariant& var, const float* betas, const float* feat, __half* featop, float* verts,
                 int64_t B, cudaStream_t st);
int lbs_tc_skin(dpb_lbs* h, const float* A, const float* transl, __half* skinop, float* verts, int64_t B,
                cudaStream_t st);
bool lbs_tc_skin_fits(const dpb_lbs* h);
int lbs_tc_skin_adjoint(dpb_lbs* h, const float* A, __half* skinop, const float* g_verts, const float* gextra,
                        bool have_extra, const float* scale, __half* gvp16, int64_t B, cudaStream_t st);
inline LbsVariant lbs_full_variant(const dpb_lbs* h) {
  LbsVariant v;
  v.n_var = h->J; v.p_feat = h->P; v.kext = h->kext; v.dirs16 = h->dirs16; v.tm_dirs = h->tm_dirs;
  return v;
}
int lbs_tc_make_tail(dpb_lbs* h, int n_var, const float* tail_pose);
bool lbs_fused2_fits(const dpb_lbs* h, const LbsVariant& v);
int lbs_fused2(dpb_lbs* h, const LbsVariant& v, __half* featop, __half* skinop, float* verts, int64_t B,
               cudaStream_t st);
bool lbs_fused3_fits(const dpb_lbs* h, const LbsVariant& v);
int lbs_fused3(dpb_lbs* h, const LbsVariant& v, __half* featop, __half* skinop, float* verts, int64_t B,
               cudaStream_t st);
int lbs_bwd_tc_prepare(dpb_lbs* h, const dpb_body_tensors* m);
void lbs_bwd_tc_release(dpb_lbs* h);
int lbs_blendT_splits(const dpb_lbs* h, int64_t B);
int lbs_blendT_tc(dpb_lbs* h, const __half* gvp16, const float* scale, float* cpart, float* gfeat, float* gbeta,
                  int64_t B, cudaStream_t st);
int lbs_skin_bwd_tc_prepare(dpb_lbs* h, const dpb_body_tensors* m);
void lbs_skin_bwd_tc_release(dpb_lbs* h);
int lbs_bwd_rowscale(dpb_lbs* h, const float* g_verts, const float* gextra, bool have_extra, float* scale, int64_t B,
                     cudaStream_t st);
int lbs_skin_bwd_tc(dpb_lbs* h, const float* vposed, const float* g_verts, const float* gextra, bool have_extra,
                    float* gA, float* gbt, const float* scale, int64_t B, cudaStream_t st);
int lbs_skin_bwd_small(dpb_lbs* h, const float* vposed, const float* g_verts, float* gA, float* gbt, int64_t B,
                       cudaStream_t st);
int lbs_bwd_prepare(dpb_lbs* h, const dpb_body_tensors* m);
void lbs_bwd_release(dpb_lbs* h);
}  // namespace dpb
