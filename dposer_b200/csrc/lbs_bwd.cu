// Linear blend skinning, backward (vector-Jacobian product w.r.t. full_pose, betas, transl).
//
//   scatter kernel   joint cotangents of the extra vertex joints / landmarks -> the vertices that produce them
//   vertex kernel    recomputes v_posed (same blend as the forward), then for every (pose, vertex):
//                      dL/dA[j] += w (g (x) [v_posed;1]),  g_vposed = T_R^T g,  dL/dtransl += g
//                    and the transposed blend  dL/dfeat = posedirs . g_vposed,  dL/dbeta = shapedirs^T g_vposed
//                    as an in-CTA [poses x 384] x [384 x (P+S)] product (warp per k, coalesced rows)
//   pose kernel      warp per pose: dL/dA -> dL/dG, reverse sweep of the kinematic tree (children push into
//                    their parent), Rodrigues backward, rest-joint cotangents -> dL/dbeta
//
// With full-vertex cotangents, the tensor-core blend available and caller scratch, the vertex kernel is split
// (5x faster on 1920 SMPL-X poses: its in-CTA transposed blend re-read the whole basis for every 8 poses):
//   lbs_tc_blend       recomputes v_posed [B,V,3] on tcgen05 (the forward's kernel)
//   lbs_skin_bwd_kernel  per (pose, vertex): dL/dA, dL/dtransl, g_vposed -> [B, 3V padded]
//   bwd_gemm_kernel    dL/d[feat | beta] = g_vposed [B,3V] . [posedirs ; shapedirs^T]^T  (fp32 SGEMM, 64x64 tiles)
//
// This is the adjoint of lbs.cu (smplx 0.1.28 lbs(); reference call sites lib/body_model/body_model.py:75-88,
// run/motion_denoising.py:255-268, run/smplify.py:243-258 where autograd differentiates the smplx ops).
#include "lbs.h"

namespace dpb {

constexpr int BW_TP = 8;
constexpr int BW_TV = 128;

__global__ void lbs_scatter_joint_grads(const float* __restrict__ g_joints, int n_out, int J, int n_extra, int n_lmk,
                                        const int32_t* __restrict__ extra_pos, const int32_t* __restrict__ lmk_pos,
                                        const float* __restrict__ lmk_bary, int n_need, float* __restrict__ gextra,
                                        int64_t B) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int per = n_extra + n_lmk * 3;
  if (i >= B * per) return;
  const int64_t b = i / per;
  const int k = (int)(i % per);
  int q, src;
  float w = 1.f;
  if (k < n_extra) {
    q = extra_pos[k];
    src = J + k;
  } else {
    const int l = (k - n_extra) / 3, f = (k - n_extra) % 3;
    q = lmk_pos[l * 3 + f];
    w = lmk_bary[l * 3 + f];
    src = J + n_extra + l;
  }
  const float* g = g_joints + ((size_t)b * n_out + src) * 3;
  float* o = gextra + ((size_t)b * n_need + q) * 3;
  atomicAdd(o + 0, w * g[0]);
  atomicAdd(o + 1, w * g[1]);
  atomicAdd(o + 2, w * g[2]);
}

__global__ void __launch_bounds__(BW_TV) lbs_vertex_bwd_kernel(
    const float* __restrict__ betas, const float* __restrict__ feat, const float* __restrict__ A,
    const float* __restrict__ v_template, const float* __restrict__ shapedirs, const float* __restrict__ posedirs,
    const int32_t* __restrict__ ell_idx, const float* __restrict__ ell_w, const int32_t* __restrict__ vlist,
    const int32_t* __restrict__ need_index, int n_verts, int n_need, int V, int J, int S, int P, int nnz,
    const float* __restrict__ g_verts, const float* __restrict__ gextra, float* __restrict__ gA,
    float* __restrict__ gfeat, float* __restrict__ gbt, int64_t B) {
  extern __shared__ float smem[];
  float* feat_s = smem;                              // [P][TP]
  float* beta_s = feat_s + (size_t)P * BW_TP;        // [S][TP]
  float* A_s = beta_s + (size_t)S * BW_TP;           // [TP][J][12]
  float* gA_s = A_s + (size_t)BW_TP * J * 12;        // [TP][J][12]
  float* gvp_s = gA_s + (size_t)BW_TP * J * 12;      // [TP][3*TV]
  float* gtr_s = gvp_s + (size_t)BW_TP * 3 * BW_TV;  // [TP][3]
  const int64_t b0 = (int64_t)blockIdx.y * BW_TP;
  const int np = (int)min((int64_t)BW_TP, B - b0);
  for (int i = threadIdx.x; i < P * BW_TP; i += BW_TV) {
    int k = i / BW_TP, p = i % BW_TP;
    feat_s[i] = p < np ? feat[(b0 + p) * P + k] : 0.f;
  }
  for (int i = threadIdx.x; i < S * BW_TP; i += BW_TV) {
    int k = i / BW_TP, p = i % BW_TP;
    beta_s[i] = p < np ? betas[(b0 + p) * S + k] : 0.f;
  }
  for (int i = threadIdx.x; i < BW_TP * J * 12; i += BW_TV) {
    A_s[i] = i < np * J * 12 ? A[b0 * J * 12 + i] : 0.f;
    gA_s[i] = 0.f;
  }
  for (int i = threadIdx.x; i < BW_TP * 3 * BW_TV; i += BW_TV) gvp_s[i] = 0.f;
  if (threadIdx.x < BW_TP * 3) gtr_s[threadIdx.x] = 0.f;
  __syncthreads();
  const int v0 = blockIdx.x * BW_TV;
  const int vi = v0 + threadIdx.x;
  if (vi < n_verts) {
    const int v = vlist ? vlist[vi] : vi;
    float acc[BW_TP][3];
#pragma unroll
    for (int p = 0; p < BW_TP; ++p) {
      acc[p][0] = v_template[v * 3 + 0];
      acc[p][1] = v_template[v * 3 + 1];
      acc[p][2] = v_template[v * 3 + 2];
    }
    for (int k = 0; k < S; ++k) {
      float s0 = shapedirs[(v * 3 + 0) * S + k], s1 = shapedirs[(v * 3 + 1) * S + k], s2 = shapedirs[(v * 3 + 2) * S + k];
#pragma unroll
      for (int p = 0; p < BW_TP; ++p) {
        float bv = beta_s[k * BW_TP + p];
        acc[p][0] = fmaf(s0, bv, acc[p][0]);
        acc[p][1] = fmaf(s1, bv, acc[p][1]);
        acc[p][2] = fmaf(s2, bv, acc[p][2]);
      }
    }
    const float* pd = posedirs + (size_t)v * 3;
    const size_t pstride = (size_t)V * 3;
    for (int k = 0; k < P; ++k) {
      float d0 = pd[k * pstride + 0], d1 = pd[k * pstride + 1], d2 = pd[k * pstride + 2];
#pragma unroll
      for (int p = 0; p < BW_TP; ++p) {
        float fv = feat_s[k * BW_TP + p];
        acc[p][0] = fmaf(d0, fv, acc[p][0]);
        acc[p][1] = fmaf(d1, fv, acc[p][1]);
        acc[p][2] = fmaf(d2, fv, acc[p][2]);
      }
    }
    const int q = vlist ? vi : (need_index ? need_index[v] : -1);
#pragma unroll
    for (int p = 0; p < BW_TP; ++p) {
      if (p >= np) break;
      float g[3] = {0.f, 0.f, 0.f};
      if (g_verts) {
        const float* gv = g_verts + ((size_t)(b0 + p) * V + v) * 3;
        g[0] = gv[0]; g[1] = gv[1]; g[2] = gv[2];
      }
      if (q >= 0 && gextra) {
        const float* ge = gextra + ((size_t)(b0 + p) * n_need + q) * 3;
        g[0] += ge[0]; g[1] += ge[1]; g[2] += ge[2];
      }
      if (g[0] == 0.f && g[1] == 0.f && g[2] == 0.f) continue;
      float TR[9];
#pragma unroll
      for (int e = 0; e < 9; ++e) TR[e] = 0.f;
      const float x = acc[p][0], y = acc[p][1], z = acc[p][2];
      for (int n = 0; n < nnz; ++n) {
        const float w = ell_w[(size_t)n * V + v];
        if (w == 0.f) continue;
        const int j = ell_idx[(size_t)n * V + v];
        const float* Ap = A_s + ((size_t)p * J + j) * 12;
#pragma unroll
        for (int e = 0; e < 9; ++e) TR[e] = fmaf(w, Ap[e], TR[e]);
        float* gp = gA_s + ((size_t)p * J + j) * 12;
#pragma unroll
        for (int i = 0; i < 3; ++i) {
          const float wg = w * g[i];
          atomicAdd(gp + i * 3 + 0, wg * x);
          atomicAdd(gp + i * 3 + 1, wg * y);
          atomicAdd(gp + i * 3 + 2, wg * z);
          atomicAdd(gp + 9 + i, wg);
        }
      }
      atomicAdd(gtr_s + p * 3 + 0, g[0]);
      atomicAdd(gtr_s + p * 3 + 1, g[1]);
      atomicAdd(gtr_s + p * 3 + 2, g[2]);
      // g_vposed = T_R^T g
      gvp_s[(p * BW_TV + threadIdx.x) * 3 + 0] = TR[0] * g[0] + TR[3] * g[1] + TR[6] * g[2];
      gvp_s[(p * BW_TV + threadIdx.x) * 3 + 1] = TR[1] * g[0] + TR[4] * g[1] + TR[7] * g[2];
      gvp_s[(p * BW_TV + threadIdx.x) * 3 + 2] = TR[2] * g[0] + TR[5] * g[1] + TR[8] * g[2];
    }
  }
  __syncthreads();
  // transposed blend: warp per k over the P pose-blend rows and the S shape-blend rows
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int ncol = min(BW_TV, n_verts - v0) * 3;
  for (int k = warp; k < P + S; k += BW_TV / 32) {
    float part[BW_TP];
#pragma unroll
    for (int p = 0; p < BW_TP; ++p) part[p] = 0.f;
    for (int col = lane; col < ncol; col += 32) {
      const int lv = col / 3, c = col % 3;
      const int v = vlist ? vlist[v0 + lv] : v0 + lv;
      const float d = k < P ? posedirs[(size_t)k * V * 3 + (size_t)v * 3 + c]
                            : shapedirs[((size_t)v * 3 + c) * S + (k - P)];
#pragma unroll
      for (int p = 0; p < BW_TP; ++p) part[p] = fmaf(d, gvp_s[p * 3 * BW_TV + col], part[p]);
    }
#pragma unroll
    for (int p = 0; p < BW_TP; ++p)
      for (int o = 16; o > 0; o >>= 1) part[p] += __shfl_xor_sync(0xffffffffu, part[p], o);
    if (lane < np) {
      float val = 0.f;
#pragma unroll
      for (int p = 0; p < BW_TP; ++p) val = (lane == p) ? part[p] : val;
      if (val != 0.f) {
        if (k < P) atomicAdd(gfeat + (b0 + lane) * P + k, val);
        else atomicAdd(gbt + (b0 + lane) * (S + 3) + (k - P), val);
      }
    }
  }
  for (int i = threadIdx.x; i < np * J * 12; i += BW_TV)
    if (gA_s[i] != 0.f) atomicAdd(gA + b0 * J * 12 + i, gA_s[i]);
  if (threadIdx.x < np * 3) {
    const int p = threadIdx.x / 3, c = threadIdx.x % 3;
    atomicAdd(gbt + (b0 + p) * (S + 3) + S + c, gtr_s[threadIdx.x]);
  }
}

// ---- split path: skinning adjoint only (v_posed given), g_vposed to global memory for the GEMM
__global__ void __launch_bounds__(BW_TV) lbs_skin_bwd_kernel(
    const float* __restrict__ A, const float* __restrict__ vposed, const int32_t* __restrict__ ell_idx,
    const float* __restrict__ ell_w, const int32_t* __restrict__ need_index, int n_need, int V, int J, int S, int nnz,
    const float* __restrict__ g_verts, const float* __restrict__ gextra, float* __restrict__ gA,
    float* __restrict__ gvp, int Kp, __half* __restrict__ gvp16, int Rp, float* __restrict__ gbt, int64_t B) {
  extern __shared__ float smem[];
  float* A_s = smem;                                 // [TP][J][12]
  float* gA_s = A_s + (size_t)BW_TP * J * 12;        // [TP][J][12]
  float* gtr_s = gA_s + (size_t)BW_TP * J * 12;      // [TP][3]
  const int64_t b0 = (int64_t)blockIdx.y * BW_TP;
  const int np = (int)min((int64_t)BW_TP, B - b0);
  for (int i = threadIdx.x; i < BW_TP * J * 12; i += BW_TV) {
    A_s[i] = i < np * J * 12 ? A[b0 * J * 12 + i] : 0.f;
    gA_s[i] = 0.f;
  }
  if (threadIdx.x < BW_TP * 3) gtr_s[threadIdx.x] = 0.f;
  __syncthreads();
  // lane = (vertex, pose): the 8 poses of a vertex sit in adjacent lanes, so the shared-memory atomics of a warp go
  // to 8 different [pose] slices (different banks) instead of 32 lanes hammering one joint's 12 floats
  static_assert(BW_TP == 8 && BW_TV % 16 == 0, "lane mapping: 8 poses x 16 vertices per pass");
  const int p = threadIdx.x & 7;
  for (int it = 0; it < BW_TV / 16; ++it) {
    const int v = blockIdx.x * BW_TV + it * 16 + (threadIdx.x >> 3);
    if (v >= V || p >= np) continue;
    const float* gv = g_verts + ((size_t)(b0 + p) * V + v) * 3;
    float g[3] = {gv[0], gv[1], gv[2]};
    const int q = need_index ? need_index[v] : -1;
    if (q >= 0 && gextra) {
      const float* ge = gextra + ((size_t)(b0 + p) * n_need + q) * 3;
      g[0] += ge[0]; g[1] += ge[1]; g[2] += ge[2];
    }
    if (g[0] == 0.f && g[1] == 0.f && g[2] == 0.f) continue;   // gvp was zeroed
    const float* xp = vposed + ((size_t)(b0 + p) * V + v) * 3;
    const float x = xp[0], y = xp[1], z = xp[2];
    float TR[9];
#pragma unroll
    for (int e = 0; e < 9; ++e) TR[e] = 0.f;
    for (int n = 0; n < nnz; ++n) {
      const float w = ell_w[(size_t)n * V + v];
      if (w == 0.f) continue;
      const int j = ell_idx[(size_t)n * V + v];
      const float* Ap = A_s + ((size_t)p * J + j) * 12;
#pragma unroll
      for (int e = 0; e < 9; ++e) TR[e] = fmaf(w, Ap[e], TR[e]);
      float* gp = gA_s + ((size_t)p * J + j) * 12;
#pragma unroll
      for (int i = 0; i < 3; ++i) {
        const float wg = w * g[i];
        atomicAdd(gp + i * 3 + 0, wg * x);
        atomicAdd(gp + i * 3 + 1, wg * y);
        atomicAdd(gp + i * 3 + 2, wg * z);
        atomicAdd(gp + 9 + i, wg);
      }
    }
    atomicAdd(gtr_s + p * 3 + 0, g[0]);
    atomicAdd(gtr_s + p * 3 + 1, g[1]);
    atomicAdd(gtr_s + p * 3 + 2, g[2]);
    const float o0 = TR[0] * g[0] + TR[3] * g[1] + TR[6] * g[2];   // g_vposed = T_R^T g
    const float o1 = TR[1] * g[0] + TR[4] * g[1] + TR[7] * g[2];
    const float o2 = TR[2] * g[0] + TR[5] * g[1] + TR[8] * g[2];
    if (gvp16) {   // operand of the tcgen05 transposed blend: fp16 [hi | lo] halves of a [B, 2*Rp] row
      __half* oh = gvp16 + (size_t)(b0 + p) * 2 * Rp + (size_t)v * 3;
      const __half h0 = __float2half_rn(o0), h1 = __float2half_rn(o1), h2 = __float2half_rn(o2);
      oh[0] = h0; oh[1] = h1; oh[2] = h2;
      oh[Rp + 0] = __float2half_rn(o0 - __half2float(h0));
      oh[Rp + 1] = __float2half_rn(o1 - __half2float(h1));
      oh[Rp + 2] = __float2half_rn(o2 - __half2float(h2));
    } else {
      float* o = gvp + (size_t)(b0 + p) * Kp + (size_t)v * 3;
      o[0] = o0; o[1] = o1; o[2] = o2;
    }
  }
  __syncthreads();
  for (int i = threadIdx.x; i < np * J * 12; i += BW_TV)
    if (gA_s[i] != 0.f) atomicAdd(gA + b0 * J * 12 + i, gA_s[i]);
  if (threadIdx.x < np * 3) {
    const int p = threadIdx.x / 3, c = threadIdx.x % 3;
    atomicAdd(gbt + (b0 + p) * (S + 3) + S + c, gtr_s[threadIdx.x]);
  }
}

// C [M, N] = X [M, K] . W [N, K]^T in fp32 (N % 64 == 0, K % 16 == 0, rows of X and W 16-byte aligned).
// 64x64 tile, 16-deep K slices, 256 threads with 4x4 micro-tiles -- the same scheme as the exact score engine.
__global__ void __launch_bounds__(256) bwd_gemm_kernel(const float* __restrict__ X, const float* __restrict__ W,
                                                       float* __restrict__ C, int64_t M, int N, int K) {
  __shared__ float Xs[16][64 + 4];
  __shared__ float Ws[16][64 + 4];
  const int tid = threadIdx.x;
  const int64_t m0 = (int64_t)blockIdx.y * 64;
  const int n0 = blockIdx.x * 64;
  const int tx = tid & 15, ty = tid >> 4;
  const int lr = tid >> 2, lk = (tid & 3) * 4;
  float acc[4][4] = {};
  const bool row_ok = m0 + lr < M;
  const float* xrow = X + (size_t)(row_ok ? m0 + lr : 0) * K + lk;
  const float* wrow = W + (size_t)(n0 + lr) * K + lk;
  float4 a = row_ok ? *reinterpret_cast<const float4*>(xrow) : make_float4(0.f, 0.f, 0.f, 0.f);
  float4 w = *reinterpret_cast<const float4*>(wrow);
  for (int k0 = 0; k0 < K; k0 += 16) {
    Xs[lk + 0][lr] = a.x; Xs[lk + 1][lr] = a.y; Xs[lk + 2][lr] = a.z; Xs[lk + 3][lr] = a.w;
    Ws[lk + 0][lr] = w.x; Ws[lk + 1][lr] = w.y; Ws[lk + 2][lr] = w.z; Ws[lk + 3][lr] = w.w;
    __syncthreads();
    if (k0 + 16 < K) {   // next slice in flight during the math
      if (row_ok) a = *reinterpret_cast<const float4*>(xrow + k0 + 16);
      w = *reinterpret_cast<const float4*>(wrow + k0 + 16);
    }
#pragma unroll
    for (int kk = 0; kk < 16; ++kk) {
      const float4 av = *reinterpret_cast<const float4*>(&Xs[kk][ty * 4]);
      const float4 wv = *reinterpret_cast<const float4*>(&Ws[kk][tx * 4]);
      const float ar[4] = {av.x, av.y, av.z, av.w}, wr[4] = {wv.x, wv.y, wv.z, wv.w};
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(ar[i], wr[j], acc[i][j]);
    }
    __syncthreads();
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int64_t m = m0 + ty * 4 + i;
    if (m < M) *reinterpret_cast<float4*>(C + m * N + n0 + tx * 4) = make_float4(acc[i][0], acc[i][1], acc[i][2], acc[i][3]);
  }
}

// gfeat[b, k] += C[b, k] (k < P);  gbeta[b, s] += C[b, P + s] (s < S)
__global__ void bwd_unpack_kernel(const float* __restrict__ C, int Np, int P, int S, float* __restrict__ gfeat,
                                  float* __restrict__ gbt, int64_t B) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= B * (P + S)) return;
  const int64_t b = i / (P + S);
  const int k = (int)(i % (P + S));
  const float v = C[b * Np + k];
  if (k < P) gfeat[b * P + k] += v;
  else gbt[b * (S + 3) + (k - P)] += v;
}

// d(loss)/d(axis-angle) from d(loss)/d(R) for R = I + sin(a) K + (1-cos(a)) K^2, a = ||r + 1e-8||, K = skew(r/a)
__device__ __forceinline__ void rodrigues_bwd(const float* __restrict__ r, const float* __restrict__ gR, float* gr) {
  const float ex = r[0] + 1e-8f, ey = r[1] + 1e-8f, ez = r[2] + 1e-8f;
  const float a = sqrtf(ex * ex + ey * ey + ez * ez);
  const float x = r[0] / a, y = r[1] / a, z = r[2] / a;
  float s, c;
  sincosf(a, &s, &c);
  const float oc = 1.0f - c;
  const float K[9] = {0.f, -z, y, z, 0.f, -x, -y, x, 0.f};
  const float K2[9] = {-(z * z) - y * y, x * y, x * z, x * y, -(z * z) - x * x, y * z, x * z, y * z, -(y * y) - x * x};
  float ga = 0.f;
#pragma unroll
  for (int e = 0; e < 9; ++e) ga += gR[e] * (c * K[e] + s * K2[e]);
  // gK = s gR + (1-c)(gR K^T + K^T gR)
  float gK[9];
#pragma unroll
  for (int i = 0; i < 3; ++i)
#pragma unroll
    for (int j = 0; j < 3; ++j) {
      float t = 0.f;
#pragma unroll
      for (int k = 0; k < 3; ++k) t += gR[i * 3 + k] * K[j * 3 + k] + K[k * 3 + i] * gR[k * 3 + j];
      gK[i * 3 + j] = s * gR[i * 3 + j] + oc * t;
    }
  const float gd[3] = {gK[7] - gK[5], gK[2] - gK[6], gK[3] - gK[1]};
  const float dot = gd[0] * r[0] + gd[1] * r[1] + gd[2] * r[2];
  const float ia = 1.0f / a, ia3 = ia * ia * ia;
  gr[0] = gd[0] * ia - dot * ex * ia3 + ga * ex * ia;
  gr[1] = gd[1] * ia - dot * ey * ia3 + ga * ey * ia;
  gr[2] = gd[2] * ia - dot * ez * ia3 + ga * ez * ia;
}

__device__ __forceinline__ void rodrigues_fwd(const float* __restrict__ p, float* R) {
  float bx = p[0] + 1e-8f, by = p[1] + 1e-8f, bz = p[2] + 1e-8f;
  float angle = sqrtf(bx * bx + by * by + bz * bz);
  float x = p[0] / angle, y = p[1] / angle, z = p[2] / angle;
  float s, c;
  sincosf(angle, &s, &c);
  float oc = 1.0f - c;
  R[0] = 1.0f + oc * (-(z * z) - y * y); R[1] = s * (-z) + oc * (x * y); R[2] = s * y + oc * (x * z);
  R[3] = s * z + oc * (x * y); R[4] = 1.0f + oc * (-(z * z) - x * x); R[5] = s * (-x) + oc * (y * z);
  R[6] = s * (-y) + oc * (x * z); R[7] = s * x + oc * (y * z); R[8] = 1.0f + oc * (-(y * y) - x * x);
}

// one warp per pose, 4 poses per CTA; smem per warp: gG [J][12] + gJ [J][3]
__global__ void __launch_bounds__(128) lbs_pose_bwd_kernel(
    const float* __restrict__ pose, const float* __restrict__ G, const float* __restrict__ jrest,
    const float* __restrict__ gA, const float* __restrict__ gfeat, const float* __restrict__ gbt,
    const float* __restrict__ g_joints, const float* __restrict__ j_shapedirsT, const int32_t* __restrict__ parents,
    const int32_t* __restrict__ depth, const int32_t* __restrict__ child_ptr, const int32_t* __restrict__ child_idx, int J,
    int S, int max_depth, int n_out, float* __restrict__ g_pose, float* __restrict__ g_betas, float* __restrict__ g_transl,
    int64_t B) {
  extern __shared__ float smem[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int64_t b = (int64_t)blockIdx.x * 4 + warp;
  if (b >= B) return;
  float* gG = smem + (size_t)warp * J * 30;
  float* gJ = gG + (size_t)J * 12;
  float* ctb = gJ + (size_t)J * 3;                     // [J,15] what joint j hands to its parent (gG part, gJ part)
  const int P = (J - 1) * 9;
  float gt[3] = {0.f, 0.f, 0.f};
  // The kernel is issue-bound (ncu: 8.8 k warp instructions per pose at 12 of 32 lanes active, a third of them in the
  // compare-and-swap loops that fp32 shared-memory atomics compile to: ATOMS.CAST.SPIN).  So: no atomics -- children
  // publish their contribution, parents pull it through a child list; the tree tables stay in registers; the sweep skips
  // (level, lane-slot) pairs that hold no joint.
  int dep[2] = {-1, -1}, par[2] = {0, 0}, c0[2] = {0, 0}, c1[2] = {0, 0};
#pragma unroll
  for (int s = 0; s < 2; ++s) {
    const int j = lane + 32 * s;
    if (j < J) { dep[s] = depth[j]; par[s] = parents[j]; c0[s] = child_ptr[j]; c1[s] = child_ptr[j + 1]; }
  }
  for (int j = lane; j < J; j += 32) {
    const float* a = gA + (b * J + j) * 12;
    const float* g = G + (b * J + j) * 12;
    const float* jr = jrest + (b * J + j) * 3;
    float gj[3] = {0.f, 0.f, 0.f};
    if (g_joints) {
      const float* q = g_joints + ((size_t)b * n_out + j) * 3;
      gj[0] = q[0]; gj[1] = q[1]; gj[2] = q[2];
      gt[0] += gj[0]; gt[1] += gj[1]; gt[2] += gj[2];
    }
    // A_R = G_R, A_t = G_t - G_R jrest
#pragma unroll
    for (int i = 0; i < 3; ++i) {
#pragma unroll
      for (int k = 0; k < 3; ++k) gG[j * 12 + i * 3 + k] = a[i * 3 + k] - a[9 + i] * jr[k];
      gG[j * 12 + 9 + i] = a[9 + i] + gj[i];
    }
#pragma unroll
    for (int k = 0; k < 3; ++k) gJ[j * 3 + k] = -(g[0 * 3 + k] * a[9] + g[1 * 3 + k] * a[10] + g[2 * 3 + k] * a[11]);
  }
  __syncwarp();
  // reverse sweep: level d publishes, level d - 1 pulls
  for (int d = max_depth; d >= 1; --d) {
#pragma unroll
    for (int s = 0; s < 2; ++s) {
      const int j = lane + 32 * s;
      const bool mine = dep[s] == d;
      if (!__any_sync(0xffffffffu, mine)) continue;      // warp-uniform: no joint of this slot sits at this level
      if (!mine) continue;
      const int p = par[s];
      float R[9];
      rodrigues_fwd(pose + (b * J + j) * 3, R);
      const float* gp = G + (b * J + p) * 12;
      float rel[3], gg[12];
#pragma unroll
      for (int k = 0; k < 3; ++k) rel[k] = jrest[(b * J + j) * 3 + k] - jrest[(b * J + p) * 3 + k];
#pragma unroll
      for (int e = 0; e < 12; ++e) gg[e] = gG[j * 12 + e];
      // for the parent: gG_R,p += gG_R,j R_j^T + gG_t,j (x) rel ; gG_t,p += gG_t,j
#pragma unroll
      for (int i = 0; i < 3; ++i) {
#pragma unroll
        for (int k = 0; k < 3; ++k)
          ctb[j * 15 + i * 3 + k] = gg[i * 3 + 0] * R[k * 3 + 0] + gg[i * 3 + 1] * R[k * 3 + 1] + gg[i * 3 + 2] * R[k * 3 + 2] +
                                    gg[9 + i] * rel[k];
        ctb[j * 15 + 9 + i] = gg[9 + i];
      }
      // own local transform: g_R_j = G_R,p^T gG_R,j (kept in place), g_rel = G_R,p^T gG_t,j
      float gl[12];
#pragma unroll
      for (int i = 0; i < 3; ++i) {
#pragma unroll
        for (int k = 0; k < 3; ++k)
          gl[i * 3 + k] = gp[0 * 3 + i] * gg[0 * 3 + k] + gp[1 * 3 + i] * gg[1 * 3 + k] + gp[2 * 3 + i] * gg[2 * 3 + k];
        gl[9 + i] = gp[0 * 3 + i] * gg[9] + gp[1 * 3 + i] * gg[10] + gp[2 * 3 + i] * gg[11];
      }
#pragma unroll
      for (int e = 0; e < 12; ++e) gG[j * 12 + e] = gl[e];
#pragma unroll
      for (int k = 0; k < 3; ++k) {
        gJ[j * 3 + k] += gl[9 + k];                       // own slot: nobody else writes it at this level
        ctb[j * 15 + 12 + k] = -gl[9 + k];
      }
    }
    __syncwarp();
#pragma unroll
    for (int s = 0; s < 2; ++s) {
      const int j = lane + 32 * s;
      const bool mine = dep[s] == d - 1 && c1[s] > c0[s];
      if (!__any_sync(0xffffffffu, mine)) continue;
      if (!mine) continue;
      float acc[15];
#pragma unroll
      for (int e = 0; e < 12; ++e) acc[e] = gG[j * 12 + e];
#pragma unroll
      for (int k = 0; k < 3; ++k) acc[12 + k] = gJ[j * 3 + k];
      for (int ci = c0[s]; ci < c1[s]; ++ci) {            // children in index order: a fixed summation order
        const float* cb = ctb + child_idx[ci] * 15;
#pragma unroll
        for (int e = 0; e < 15; ++e) acc[e] += cb[e];
      }
#pragma unroll
      for (int e = 0; e < 12; ++e) gG[j * 12 + e] = acc[e];
#pragma unroll
      for (int k = 0; k < 3; ++k) gJ[j * 3 + k] = acc[12 + k];
    }
    __syncwarp();
  }
  if (lane == 0) {  // root: M_0 = G_0, rel_0 = jrest_0
    gJ[0] += gG[9]; gJ[1] += gG[10]; gJ[2] += gG[11];
  }
  __syncwarp();
  // Rodrigues backward (gG[j][0..8] now holds dL/dR_j of the local rotation)
  for (int j = lane; j < J; j += 32) {
    float gR[9];
#pragma unroll
    for (int e = 0; e < 9; ++e) gR[e] = gG[j * 12 + e] + (j > 0 ? gfeat[b * P + (j - 1) * 9 + e] : 0.f);
    float gr[3];
    rodrigues_bwd(pose + (b * J + j) * 3, gR, gr);
    if (g_pose) {
      g_pose[(b * J + j) * 3 + 0] = gr[0];
      g_pose[(b * J + j) * 3 + 1] = gr[1];
      g_pose[(b * J + j) * 3 + 2] = gr[2];
    }
  }
  if (g_betas) {
    for (int s = 0; s < S; ++s) {
      float part = 0.f;
      for (int q = lane; q < 3 * J; q += 32) part = fmaf(j_shapedirsT[s * 3 * J + q], gJ[q], part);   // contiguous rows
      for (int o = 16; o > 0; o >>= 1) part += __shfl_xor_sync(0xffffffffu, part, o);
      if (lane == 0) g_betas[b * S + s] = part + gbt[b * (S + 3) + s];
    }
  }
  if (g_transl) {
#pragma unroll
    for (int c = 0; c < 3; ++c)
      for (int o = 16; o > 0; o >>= 1) gt[c] += __shfl_xor_sync(0xffffffffu, gt[c], o);
    if (lane == 0) {
#pragma unroll
      for (int c = 0; c < 3; ++c) g_transl[b * 3 + c] = gt[c] + gbt[b * (S + 3) + S + c];
    }
  }
}

int lbs_bwd_prepare(dpb_lbs* h, const dpb_body_tensors* m) {
  const int V = h->V, P = h->P, S = h->S;
  h->bw_np = (P + S + 63) / 64 * 64;
  h->bw_kp = (3 * V + 15) / 16 * 16;
  std::vector<float> pad((size_t)h->bw_np * h->bw_kp, 0.f);
  for (int k = 0; k < P; ++k)
    for (int c = 0; c < 3 * V; ++c) pad[(size_t)k * h->bw_kp + c] = m->posedirs[(size_t)k * 3 * V + c];
  for (int c = 0; c < 3 * V; ++c)
    for (int s = 0; s < S; ++s) pad[(size_t)(P + s) * h->bw_kp + c] = m->shapedirs[(size_t)c * S + s];
  DPB_CUDA_CHECK(cudaMalloc((void**)&h->dirs_pad, pad.size() * sizeof(float)));
  DPB_CUDA_CHECK(cudaMemcpy(h->dirs_pad, pad.data(), pad.size() * sizeof(float), cudaMemcpyHostToDevice));
  return DPB_OK;
}

void lbs_bwd_release(dpb_lbs* h) {
  if (h->dirs_pad) cudaFree(h->dirs_pad);
  h->dirs_pad = nullptr;
}

// vposed | g_vposed (fp32 [B, bw_kp] or fp16 [B, 2*bt_rp]) | GEMM output (fp32 [B, bw_np] or [splits, B, bt_kp])
static size_t bwd_gvp_bytes(const dpb_lbs* h, int64_t B) {
  const size_t a = (size_t)B * h->bw_kp * 4, b = h->bt_ready ? (size_t)B * 2 * h->bt_rp * 2 : 0;
  return align_up(a > b ? a : b, 256);
}
static size_t bwd_scratch_bytes(const dpb_lbs* h, int64_t B) {
  const size_t a = (size_t)B * h->bw_np * 4;
  const size_t b = h->bt_ready ? (size_t)lbs_blendT_splits(h, B) * B * h->bt_kp * 4 : 0;
  return align_up((size_t)B * h->V * 3 * 4, 256) + bwd_gvp_bytes(h, B) + align_up(a > b ? a : b, 256) +
         align_up((size_t)B * 4, 256);
}

}  // namespace dpb

using namespace dpb;

extern "C" size_t dpb_lbs_backward_scratch_bytes(dpb_lbs_t* h, int64_t B) {
  if (!h || B <= 0 || !h->tc_ready || !h->dirs_pad) return 0;
  return bwd_scratch_bytes(h, B);
}

extern "C" size_t dpb_lbs_backward_scratch_bytes_joints(dpb_lbs_t* h, int64_t B) {
  if (!h || B <= 0 || !h->sub || !h->sub->bt_ready || !h->sub->sb_ready) return 0;
  return bwd_scratch_bytes(h->sub, B);
}

namespace dpb {
// vertex pass of the backward on the tensor cores for the vertex set of `hv` (the full model or the compact one):
// v_posed recompute -> skinning adjoint (dL/dA, g_vposed) -> transposed blend (dL/dfeat, dL/dbeta)
static int bwd_vertex_pass_tc(dpb_lbs* hv, bool const_tail, const LbsWs& w, const float* betas, const float* g_verts,
                              const float* gextra, bool have_extra, uint8_t* sp, int64_t B, cudaStream_t st) {
  // v_posed recompute with the basis the forward used: the const-tail one (K = 224 for SMPL-X instead of 512) when declared
  const LbsVariant var = (const_tail && hv->tailv.dirs16) ? hv->tailv : lbs_full_variant(hv);
  float* vposed = reinterpret_cast<float*>(sp);
  __half* gvp16 = reinterpret_cast<__half*>(sp + align_up((size_t)B * hv->V * 3 * 4, 256));
  float* gout = reinterpret_cast<float*>(sp + align_up((size_t)B * hv->V * 3 * 4, 256) + bwd_gvp_bytes(hv, B));
  float* scale = reinterpret_cast<float*>(sp + bwd_scratch_bytes(hv, B) - align_up((size_t)B * 4, 256));
  int rc = lbs_tc_blend(hv, var, betas, w.feat, w.featop, vposed, B, st);
  if (rc != DPB_OK) return rc;
  DPB_CUDA_CHECK(cudaMemsetAsync(gvp16, 0, (size_t)B * 2 * hv->bt_rp * 2, st));
  rc = lbs_bwd_rowscale(hv, g_verts, gextra, have_extra, scale, B, st);
  if (rc == DPB_OK) rc = lbs_tc_skin_adjoint(hv, w.A, w.skinop, g_verts, gextra, have_extra, scale, gvp16, B, st);
  if (rc == DPB_OK) {
    // dL/dA: the GEMM, or for small vertex sets without extra cotangents (the compact set) the per-joint vertex lists
    if (hv->csr_ptr && !have_extra) rc = lbs_skin_bwd_small(hv, vposed, g_verts, w.gA, w.gbeta, B, st);
    else rc = lbs_skin_bwd_tc(hv, vposed, g_verts, gextra, have_extra, w.gA, w.gbeta, scale, B, st);
  }
  if (rc != DPB_OK) return rc;
  return lbs_blendT_tc(hv, gvp16, scale, gout, w.gfeat, w.gbeta, B, st);
}
}  // namespace dpb

extern "C" int dpb_lbs_backward(dpb_lbs_t* h, const float* betas, const float* full_pose, const float* g_verts,
                                const float* g_joints, float* g_pose, float* g_betas, float* g_transl, int64_t B,
                                int flags, void* ws, size_t ws_bytes, void* scratch, size_t scratch_bytes,
                                void* stream) {
  if (!h) return fail(DPB_EINVAL, "dpb_lbs_backward: null handle");
  DeviceGuard guard(h->device);
  DPB_REQUIRE(betas && full_pose, "dpb_lbs_backward: betas and full_pose are required");
  DPB_REQUIRE(g_verts || g_joints, "dpb_lbs_backward: need g_verts and/or g_joints");
  if (B <= 0) return DPB_OK;
  cudaStream_t st = (cudaStream_t)stream;
  LbsWs w;
  if (!lbs_carve(h, B, false, ws, ws_bytes, &w)) return fail(DPB_ENOMEM, "dpb_lbs_backward: workspace too small");
  const int J = h->J, S = h->S, P = h->P;
  DPB_CUDA_CHECK(cudaMemsetAsync(w.gA, 0, (size_t)B * J * 12 * 4, st));
  DPB_CUDA_CHECK(cudaMemsetAsync(w.gfeat, 0, (size_t)B * P * 4, st));
  DPB_CUDA_CHECK(cudaMemsetAsync(w.gbeta, 0, (size_t)B * (S + 3) * 4, st));
  const int per = h->n_extra + h->n_lmk * 3;
  const bool have_extra = g_joints && per > 0 && h->n_need > 0;
  if (have_extra) {
    DPB_CUDA_CHECK(cudaMemsetAsync(w.gextra, 0, (size_t)B * h->n_need * 3 * 4, st));
    int64_t n = B * per;
    lbs_scatter_joint_grads<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(g_joints, h->n_out, J, h->n_extra, h->n_lmk,
                                                                          h->extra_pos, h->lmk_pos, h->lmk_bary,
                                                                          h->n_need, w.gextra, B);
    DPB_CUDA_CHECK(cudaGetLastError());
  }
  const bool full = g_verts != nullptr;
  const int n_verts = full ? h->V : h->n_need;
  const bool split = full && scratch && h->tc_ready && w.featop && h->dirs_pad &&
                     scratch_bytes >= bwd_scratch_bytes(h, B);
  if (split) {
    uint8_t* sp = static_cast<uint8_t*>(scratch);
    float* vposed = reinterpret_cast<float*>(sp);
    float* gvp = reinterpret_cast<float*>(sp + align_up((size_t)B * h->V * 3 * 4, 256));
    float* gout = reinterpret_cast<float*>(sp + align_up((size_t)B * h->V * 3 * 4, 256) + bwd_gvp_bytes(h, B));
    float* scale = reinterpret_cast<float*>(sp + bwd_scratch_bytes(h, B) - align_up((size_t)B * 4, 256));
    // skinning adjoint (dL/dA) and transposed blend on tcgen05 where the model's operands exist, else the round-1
    // kernels (shared-memory atomics + fp32 SGEMM)
    const bool tcT = h->bt_ready && h->sb_ready && w.skinop && lbs_tc_skin_fits(h);
    __half* gvp16 = tcT ? reinterpret_cast<__half*>(gvp) : nullptr;
    // v_posed recompute with the basis the forward used (const-tail: K = 224 instead of 512 for SMPL-X)
    const LbsVariant bvar = ((flags & DPB_LBS_CONST_TAIL) && h->tailv.dirs16) ? h->tailv : lbs_full_variant(h);
    int rc = lbs_tc_blend(h, bvar, betas, w.feat, w.featop, vposed, B, st);
    if (rc != DPB_OK) return rc;
    if (tcT) DPB_CUDA_CHECK(cudaMemsetAsync(gvp16, 0, (size_t)B * 2 * h->bt_rp * 2, st));
    else DPB_CUDA_CHECK(cudaMemsetAsync(gvp, 0, (size_t)B * h->bw_kp * 4, st));
    if (tcT) {
      rc = lbs_bwd_rowscale(h, g_verts, w.gextra, have_extra, scale, B, st);
      if (rc == DPB_OK) rc = lbs_tc_skin_adjoint(h, w.A, w.skinop, g_verts, w.gextra, have_extra, scale, gvp16, B, st);
      if (rc == DPB_OK) rc = lbs_skin_bwd_tc(h, vposed, g_verts, w.gextra, have_extra, w.gA, w.gbeta, scale, B, st);
      if (rc != DPB_OK) return rc;
    } else {
    const size_t smem = ((size_t)2 * BW_TP * J * 12 + BW_TP * 3) * 4;
      DPB_CUDA_CHECK(cudaFuncSetAttribute(lbs_skin_bwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
      dim3 grid((h->V + BW_TV - 1) / BW_TV, (unsigned)((B + BW_TP - 1) / BW_TP));
      DPB_REQUIRE(grid.y <= 65535u, "dpb_lbs_backward: batch too large for one call (max 65535*8 poses)");
      lbs_skin_bwd_kernel<<<grid, BW_TV, smem, st>>>(w.A, vposed, h->ell_idx, h->ell_w,
                                                     have_extra ? h->need_index : nullptr, h->n_need, h->V, J, S, h->nnz,
                                                     g_verts, have_extra ? w.gextra : nullptr, w.gA, gvp, h->bw_kp,
                                                     nullptr, 0, w.gbeta, B);
      DPB_CUDA_CHECK(cudaGetLastError());
    }
    if (tcT) {
      rc = lbs_blendT_tc(h, gvp16, scale, gout, w.gfeat, w.gbeta, B, st);
      if (rc != DPB_OK) return rc;
    } else {
      dim3 ggrid(h->bw_np / 64, (unsigned)((B + 63) / 64));
      bwd_gemm_kernel<<<ggrid, 256, 0, st>>>(gvp, h->dirs_pad, gout, B, h->bw_np, h->bw_kp);
      const int64_t n = B * (P + S);
      bwd_unpack_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(gout, h->bw_np, P, S, w.gfeat, w.gbeta, B);
      DPB_CUDA_CHECK(cudaGetLastError());
    }
  } else if (!full && have_extra && h->sub && h->sub->bt_ready && h->sub->sb_ready && w.featop && w.skinop &&
             lbs_tc_skin_fits(h->sub) && scratch &&
             scratch_bytes >= bwd_scratch_bytes(h->sub, B)) {
    // joints-only mode: the cotangents of the compact vertex set go through the same tensor-core pass
    int rc = bwd_vertex_pass_tc(h->sub, (flags & DPB_LBS_CONST_TAIL) != 0, w, betas, w.gextra, nullptr, false,
                                static_cast<uint8_t*>(scratch), B, st);
    if (rc != DPB_OK) return rc;
  } else if (full || have_extra) {
    size_t smem = ((size_t)P * BW_TP + (size_t)S * BW_TP + 2 * (size_t)BW_TP * J * 12 + (size_t)BW_TP * 3 * BW_TV +
                   BW_TP * 3) * 4;
    DPB_CUDA_CHECK(cudaFuncSetAttribute(lbs_vertex_bwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    dim3 grid((n_verts + BW_TV - 1) / BW_TV, (unsigned)((B + BW_TP - 1) / BW_TP));
    DPB_REQUIRE(grid.y <= 65535u, "dpb_lbs_backward: batch too large for one call (max 65535*8 poses)");
    lbs_vertex_bwd_kernel<<<grid, BW_TV, smem, st>>>(betas, w.feat, w.A, h->v_template, h->shapedirs, h->posedirs,
                                                     h->ell_idx, h->ell_w, full ? nullptr : h->need_vids,
                                                     full ? h->need_index : nullptr, n_verts, h->n_need, h->V, J, S,
                                                     P, h->nnz, g_verts, have_extra ? w.gextra : nullptr, w.gA,
                                                     w.gfeat, w.gbeta, B);
    DPB_CUDA_CHECK(cudaGetLastError());
  }
  DPB_REQUIRE(J <= 64, "dpb_lbs_backward: the pose kernel handles up to 64 joints");
  size_t psmem = (size_t)4 * J * 30 * 4;
  lbs_pose_bwd_kernel<<<(unsigned)((B + 3) / 4), 128, psmem, st>>>(full_pose, w.G, w.jrest, w.gA, w.gfeat, w.gbeta,
                                                                    g_joints, h->j_shapedirsT, h->parents, h->depth, h->child_ptr, h->child_idx,
                                                                    J,
                                                                    S, h->max_depth, h->n_out, g_pose, g_betas,
                                                                    g_transl, B);
  DPB_CUDA_CHECK(cudaGetLastError());
  return DPB_OK;
}
