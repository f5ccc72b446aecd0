// Internal declarations of the training-step path (gemm_tc.cu, train.cu).
#pragma once
#include <cuda_fp16.h>

#include "common.cuh"

struct dpb_score;

namespace dpb {

// A K-major fp16 [hi | lo] GEMM operand living inside a larger buffer: element (r, k) of the operand is
// ptr[(r0 + r) * ld + k0 + k] (hi) and ptr[(r0 + r) * ld + k0 + lo + k] (lo); `rows` = rows of the whole buffer.
struct Op16 {
  __half* ptr = nullptr;
  int64_t ld = 0, rows = 0;
  int r0 = 0, k0 = 0, lo = 0;
  Op16 block(int r, int k) const { Op16 o = *this; o.r0 += r; o.k0 += k; return o; }
};

int gemm_tc_init();
// C[M,N] = A[M,K] B[N,K]^T (+ bias1[n] + bias2[n] + add[m,n]); K is rounded up to 64 (operand pads must be zero)
int gemm_tc(const Op16& A, const Op16& B, int M, int N, int K, float* C, int64_t ldc, const float* bias1,
            const float* bias2, const float* add, int64_t ldadd, cudaStream_t st, int bias_rows = 0x7fffffff);
// fp32 [R, C] -> fp16 [hi | lo] in row form (operand rows = R) and / or column form (operand rows = C)
int split16(const float* src, int R, int Cc, int64_t ld, const Op16* row, const Op16* col, cudaStream_t st);

// score-net JVP on the same GEMM (score_simt.cu): raw [2B, DP] = post_dense of the stacked [primal ; tangent] rows
size_t score_jvp_tc_ws_bytes(int64_t B, int dp);
int score_jvp_tc_raw(dpb_score* h, const float* x, const float* v, const float* table, float* raw, int64_t B, void* ws,
                     size_t ws_bytes, cudaStream_t st);
void score_jvp_tc_release(dpb_score* h);

}  // namespace dpb
