// Linear blend skinning, forward: pose kernel (Rodrigues + warp-per-chain kinematic tree with
// shuffle-based transform propagation) and the fp32 vertex kernel (shape blend + pose blend +
// sparse skinning, coalesced over vertices).  The tcgen05 pose-blend engine lives in lbs_tc.cu.
//
// Follows smplx==0.1.28 lbs()/SMPL.forward/SMPLX.forward as called by the reference at
// lib/body_model/body_model.py:75-88 and lib/body_model/smpl.py:67-78 (SURVEY.md Appendix A.6).
#include "lbs.h"

#include <algorithm>
#include <cmath>
#include <map>

namespace dpb {

// ------------------------------------------------------------------ pose kernel
// One warp per pose.  Lane l owns joint l (slot 0) and joint l+32 (slot 1, SMPL-X only).
// A transform is 12 floats: r[0..8] row-major rotation, r[9..11] translation.
struct Xf {
  float r[12];
};

__device__ __forceinline__ void rodrigues(const float* __restrict__ p, float* R) {
  // batch_rodrigues: angle = ||r + 1e-8||, dir = r / angle, R = I + sin K + (1-cos) K^2
  float ax = p[0], ay = p[1], az = p[2];
  float bx = ax + 1e-8f, by = ay + 1e-8f, bz = az + 1e-8f;
  float angle = sqrtf(bx * bx + by * by + bz * bz);
  float x = ax / angle, y = ay / angle, z = az / angle;
  float s, c;
  sincosf(angle, &s, &c);
  float oc = 1.0f - c;
  R[0] = 1.0f + oc * (-(z * z) - y * y);
  R[1] = s * (-z) + oc * (x * y);
  R[2] = s * y + oc * (x * z);
  R[3] = s * z + oc * (x * y);
  R[4] = 1.0f + oc * (-(z * z) - x * x);
  R[5] = s * (-x) + oc * (y * z);
  R[6] = s * (-y) + oc * (x * z);
  R[7] = s * x + oc * (y * z);
  R[8] = 1.0f + oc * (-(y * y) - x * x);
}

// G_child = G_parent * M_child   (both [R|t])
__device__ __forceinline__ void compose(const float* __restrict__ P, const float* __restrict__ M, float* O) {
#pragma unroll
  for (int i = 0; i < 3; ++i) {
#pragma unroll
    for (int j = 0; j < 3; ++j)
      O[i * 3 + j] = P[i * 3 + 0] * M[0 * 3 + j] + P[i * 3 + 1] * M[1 * 3 + j] + P[i * 3 + 2] * M[2 * 3 + j];
    O[9 + i] = P[i * 3 + 0] * M[9] + P[i * 3 + 1] * M[10] + P[i * 3 + 2] * M[11] + P[9 + i];
  }
}

template <int SLOTS>
__global__ void __launch_bounds__(128) lbs_pose_kernel(
    const float* __restrict__ betas, const float* __restrict__ pose, const float* __restrict__ transl,
    const float* __restrict__ j_template, const float* __restrict__ j_shapedirsT,
    const int32_t* __restrict__ parents, const int32_t* __restrict__ depth, int J, int S, int max_depth,
    float* __restrict__ A_out, float* __restrict__ G_out, float* __restrict__ feat_out,
    float* __restrict__ jrest_out, float* __restrict__ joints_out, int n_out, int64_t B,
    __half* __restrict__ featop, int Kp, int p_feat, __half* __restrict__ skinop, int Jp) {
  // featop / skinop (optional): the tcgen05 engine's fp16 [hi | lo] operands, written here instead of by two more
  // passes over feat and A (lbs_tc.cu: lbs_featop_kernel / lbs_skinop_kernel define the layout)
  const int lane = threadIdx.x & 31;
  const int64_t b = (int64_t)blockIdx.x * 4 + (threadIdx.x >> 5);
  // The fp16 operand rows are assembled in shared memory (2-byte scattered writes) and leave as 16-byte vectors:
  // written straight to global they were ~60 two-byte stores per lane and the kernel took 0.28 ms per 65 536 poses.
  __shared__ __align__(16) __half stage_f[4][1024];       // [hi | lo] blend operand row (2 * Kp <= 1024)
  __shared__ __align__(16) __half stage_s[4][12 * 128];   // 12 transform rows x [hi | lo] (2 * Jp <= 128)
  // fp32 side outputs (A, G, feat: what the backward reads) leave through a per-warp staging row as well: written from the
  // registers each store instruction touched 32 lanes x 4 bytes at a 48- / 36-byte stride (every sector 9-12 times)
  __shared__ float stage_x[4][64 * 12];
  if (b >= B) return;  // warp-uniform
  float* xs = stage_x[threadIdx.x >> 5];
  auto flush = [&](float* __restrict__ dst, int n) {      // staging row -> global, 128 contiguous bytes per instruction
    __syncwarp();
    for (int i = lane; i < n; i += 32) dst[i] = xs[i];
    __syncwarp();
  };
  const int P = (J - 1) * 9;
  __half* fs = stage_f[threadIdx.x >> 5];
  __half* ss = stage_s[threadIdx.x >> 5];
  auto put_split = [](__half* row, int k, int half_width, float x) {
    const __half hi = __float2half_rn(x);
    row[k] = hi;
    row[half_width + k] = __float2half_rn(x - __half2float(hi));
  };
  if (featop) {   // [beta | feat (p_feat of them: the variant's varying joints) | 1 (template slot) | 0] of this pose;
    __half* frow = fs;                            // the feat part is written with the rotations below
    for (int k = lane; k < Kp; k += 32)
      if (k < S) put_split(frow, k, Kp, betas[b * S + k]);
      else if (k >= S + p_feat) put_split(frow, k, Kp, k == S + p_feat ? 1.0f : 0.f);
  }
  // rest joints J_template + J_shapedirs . beta (== J_regressor . v_shaped): lanes walk the (joint, coordinate) pairs, so
  // every load of the transposed table and the jrest store are contiguous (per joint-lane the table is a 12 S-byte stride:
  // 32 cache lines per load instruction, which was most of this kernel's time)
  for (int q = lane; q < 3 * J; q += 32) {
    float acc = j_template[q];
    for (int k = 0; k < S; ++k) acc = fmaf(j_shapedirsT[k * 3 * J + q], betas[b * S + k], acc);
    xs[q] = acc;
    if (jrest_out) jrest_out[b * J * 3 + q] = acc;
  }
  __syncwarp();
  float M[SLOTS][12], G[SLOTS][12], jr[SLOTS][3];
  int par[SLOTS], dep[SLOTS];
#pragma unroll
  for (int s = 0; s < SLOTS; ++s) {
    const int j = lane + 32 * s;
#pragma unroll
    for (int c = 0; c < 3; ++c) jr[s][c] = j < J ? xs[j * 3 + c] : 0.f;
  }
  __syncwarp();                      // the staging row is reused for the pose features below
#pragma unroll
  for (int s = 0; s < SLOTS; ++s) {
    const int j = lane + 32 * s;
    par[s] = -1;
    dep[s] = -1;
#pragma unroll
    for (int e = 0; e < 12; ++e) M[s][e] = G[s][e] = 0.f;
    if (j < J) {
      par[s] = parents[j];
      dep[s] = depth[j];
      rodrigues(pose + (b * J + j) * 3, M[s]);
      if (j > 0) {
#pragma unroll
        for (int e = 0; e < 9; ++e)
        {
          const float f = M[s][e] - ((e == 0 || e == 4 || e == 8) ? 1.0f : 0.0f);
          if (feat_out) xs[(j - 1) * 9 + e] = f;
          if (featop && (j - 1) * 9 + e < p_feat) put_split(fs, S + (j - 1) * 9 + e, Kp, f);
        }
      }
    }
  }
  if (feat_out) flush(feat_out + b * P, P);
  // relative joint offsets need the parent's rest joint: fetch by shuffle
#pragma unroll
  for (int s = 0; s < SLOTS; ++s) {
    const int p = par[s] < 0 ? 0 : par[s];
    float pj[3];
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      float v = __shfl_sync(0xffffffffu, jr[0][c], p & 31);
      if (SLOTS > 1) {
        float v1 = __shfl_sync(0xffffffffu, jr[SLOTS - 1][c], p & 31);
        v = (p >> 5) ? v1 : v;
      }
      pj[c] = v;
    }
#pragma unroll
    for (int c = 0; c < 3; ++c) M[s][9 + c] = jr[s][c] - (par[s] < 0 ? 0.f : pj[c]);
    if (dep[s] == 0) {
#pragma unroll
      for (int e = 0; e < 12; ++e) G[s][e] = M[s][e];
    }
  }
  // level-by-level propagation: lanes at depth d pull their parent's global transform by shuffle
  for (int d = 1; d <= max_depth; ++d) {
#pragma unroll
    for (int s = 0; s < SLOTS; ++s) {
      const int p = par[s] < 0 ? 0 : par[s];
      float Pg[12];
#pragma unroll
      for (int e = 0; e < 12; ++e) {
        float v = __shfl_sync(0xffffffffu, G[0][e], p & 31);
        if (SLOTS > 1) {
          float v1 = __shfl_sync(0xffffffffu, G[SLOTS - 1][e], p & 31);
          v = (p >> 5) ? v1 : v;
        }
        Pg[e] = v;
      }
      if (dep[s] == d) compose(Pg, M[s], G[s]);
    }
  }
  const float tx = transl ? transl[b * 3 + 0] : 0.f, ty = transl ? transl[b * 3 + 1] : 0.f,
              tz = transl ? transl[b * 3 + 2] : 0.f;
#pragma unroll
  for (int s = 0; s < SLOTS; ++s) {
    const int j = lane + 32 * s;
    if (skinop && j >= J && j < Jp) {   // the spare joint slot J carries the translation (weight 1), the rest is padding
      const float t3[3] = {tx, ty, tz};
#pragma unroll
      for (int e = 0; e < 12; ++e)
        put_split(ss + e * 2 * Jp, j, Jp, (j == J && e >= 9) ? t3[e - 9] : 0.f);
    }
    if (j >= J) continue;
    float Ao[12];
#pragma unroll
    for (int e = 0; e < 9; ++e) Ao[e] = G[s][e];
#pragma unroll
    for (int i = 0; i < 3; ++i)
      Ao[9 + i] = G[s][9 + i] - (G[s][i * 3 + 0] * jr[s][0] + G[s][i * 3 + 1] * jr[s][1] + G[s][i * 3 + 2] * jr[s][2]);
    if (A_out) {   // fp32 copy for the backward pass / the fp32 vertex kernel (skipped on forward-only fused calls)
#pragma unroll
      for (int e = 0; e < 12; ++e) xs[j * 12 + e] = Ao[e];
    }
    if (skinop) {
#pragma unroll
      for (int e = 0; e < 12; ++e) put_split(ss + e * 2 * Jp, j, Jp, Ao[e]);
    }
    float* jo = joints_out + (b * n_out + j) * 3;
    jo[0] = G[s][9] + tx;
    jo[1] = G[s][10] + ty;
    jo[2] = G[s][11] + tz;
  }
  if (A_out) {
    flush(A_out + b * J * 12, J * 12);
#pragma unroll
    for (int s = 0; s < SLOTS; ++s) {
      const int j = lane + 32 * s;
      if (j < J) {
#pragma unroll
        for (int e = 0; e < 12; ++e) xs[j * 12 + e] = G[s][e];
      }
    }
    flush(G_out + b * J * 12, J * 12);
  }
  // shared-memory operand rows -> global, 16 bytes per lane per step
  if (featop || skinop) __syncwarp();
  if (featop) {
    const uint4* src = reinterpret_cast<const uint4*>(fs);
    uint4* dst = reinterpret_cast<uint4*>(featop + (size_t)b * 2 * Kp);
    for (int i = lane; i < Kp / 4; i += 32) dst[i] = src[i];          // 2*Kp halves = Kp/4 vectors
  }
  if (skinop) {
    const uint4* src = reinterpret_cast<const uint4*>(ss);
    uint4* dst = reinterpret_cast<uint4*>(skinop + (size_t)b * 12 * 2 * Jp);
    for (int i = lane; i < 3 * Jp; i += 32) dst[i] = src[i];          // 12 rows x 2*Jp halves = 3*Jp vectors
  }
}

// ------------------------------------------------------------------ fp32 vertex kernel
// CTA = 128 threads (one vertex each) x TP poses.  acc[p][c] accumulates
// v_template + shapedirs.beta + posedirs^T.feat; then sparse skinning and the coalesced store.
constexpr int LBS_TP = 16;
constexpr int LBS_TV = 128;

__global__ void __launch_bounds__(LBS_TV) lbs_vertex_kernel(
    const float* __restrict__ betas, const float* __restrict__ transl, const float* __restrict__ feat,
    const float* __restrict__ A, const float* __restrict__ v_template, const float* __restrict__ shapedirs,
    const float* __restrict__ posedirs, const int32_t* __restrict__ ell_idx, const float* __restrict__ ell_w,
    const int32_t* __restrict__ vlist, int n_verts, int V, int J, int S, int P, int nnz,
    const float* vp_in, float* out, int64_t B) {
  // vp_in != nullptr: the blend (v_posed) was already produced by the tcgen05 engine -- skin it in place
  // (vp_in == out, S = P = 0 passed by the caller); otherwise blend here in fp32.
  extern __shared__ float smem[];
  float* feat_s = smem;                       // [P][TP]  (k-major so 4 poses load as one float4)
  float* beta_s = feat_s + (size_t)P * LBS_TP;  // [S][TP]
  float* A_s = beta_s + (size_t)S * LBS_TP;     // [TP][J][12]
  float* tr_s = A_s + (size_t)LBS_TP * J * 12;  // [TP][3]
  const int64_t b0 = (int64_t)blockIdx.y * LBS_TP;
  const int np = (int)min((int64_t)LBS_TP, B - b0);
  for (int i = threadIdx.x; i < P * LBS_TP; i += LBS_TV) {
    int k = i / LBS_TP, p = i % LBS_TP;
    feat_s[i] = p < np ? feat[(b0 + p) * P + k] : 0.f;
  }
  for (int i = threadIdx.x; i < S * LBS_TP; i += LBS_TV) {
    int k = i / LBS_TP, p = i % LBS_TP;
    beta_s[i] = p < np ? betas[(b0 + p) * S + k] : 0.f;
  }
  for (int i = threadIdx.x; i < np * J * 12; i += LBS_TV) A_s[i] = A[b0 * J * 12 + i];
  for (int i = threadIdx.x; i < LBS_TP * 3; i += LBS_TV) {
    int p = i / 3;
    tr_s[i] = (transl && p < np) ? transl[(b0 + p) * 3 + i % 3] : 0.f;
  }
  __syncthreads();
  const int vi = blockIdx.x * LBS_TV + threadIdx.x;
  if (vi >= n_verts) return;
  const int v = vlist ? vlist[vi] : vi;
  float acc[LBS_TP][3];
  if (vp_in) {
#pragma unroll
    for (int p = 0; p < LBS_TP; ++p) {
      const float* s = vp_in + ((size_t)(b0 + (p < np ? p : 0)) * n_verts + vi) * 3;
      acc[p][0] = s[0]; acc[p][1] = s[1]; acc[p][2] = s[2];
    }
  } else {
#pragma unroll
    for (int p = 0; p < LBS_TP; ++p) {
      acc[p][0] = v_template[v * 3 + 0];
      acc[p][1] = v_template[v * 3 + 1];
      acc[p][2] = v_template[v * 3 + 2];
    }
  }
  // shape blend: v_shaped = v_template + shapedirs . beta
  for (int k = 0; k < S; ++k) {
    float s0 = shapedirs[(v * 3 + 0) * S + k], s1 = shapedirs[(v * 3 + 1) * S + k], s2 = shapedirs[(v * 3 + 2) * S + k];
#pragma unroll
    for (int q = 0; q < LBS_TP / 4; ++q) {
      float4 bb = *reinterpret_cast<const float4*>(&beta_s[k * LBS_TP + q * 4]);
      float bv[4] = {bb.x, bb.y, bb.z, bb.w};
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        acc[q * 4 + i][0] = fmaf(s0, bv[i], acc[q * 4 + i][0]);
        acc[q * 4 + i][1] = fmaf(s1, bv[i], acc[q * 4 + i][1]);
        acc[q * 4 + i][2] = fmaf(s2, bv[i], acc[q * 4 + i][2]);
      }
    }
  }
  // pose blend: += feat . posedirs[:, 3v..3v+2]
  const float* pd = posedirs + (size_t)v * 3;
  const size_t pstride = (size_t)V * 3;
#pragma unroll 2
  for (int k = 0; k < P; ++k) {
    float d0 = pd[k * pstride + 0], d1 = pd[k * pstride + 1], d2 = pd[k * pstride + 2];
#pragma unroll
    for (int q = 0; q < LBS_TP / 4; ++q) {
      float4 ff = *reinterpret_cast<const float4*>(&feat_s[k * LBS_TP + q * 4]);
      float fv[4] = {ff.x, ff.y, ff.z, ff.w};
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        acc[q * 4 + i][0] = fmaf(d0, fv[i], acc[q * 4 + i][0]);
        acc[q * 4 + i][1] = fmaf(d1, fv[i], acc[q * 4 + i][1]);
        acc[q * 4 + i][2] = fmaf(d2, fv[i], acc[q * 4 + i][2]);
      }
    }
  }
  // skinning: T = sum_n w_n A[idx_n];  out = T [v;1] + transl
#pragma unroll
  for (int p = 0; p < LBS_TP; ++p) {
    if (p >= np) break;
    float T[12];
#pragma unroll
    for (int e = 0; e < 12; ++e) T[e] = 0.f;
    for (int n = 0; n < nnz; ++n) {
      float w = ell_w[(size_t)n * V + v];
      int j = ell_idx[(size_t)n * V + v];
      const float4* Ap = reinterpret_cast<const float4*>(A_s + ((size_t)p * J + j) * 12);
      float4 a0 = Ap[0], a1 = Ap[1], a2 = Ap[2];
      T[0] = fmaf(w, a0.x, T[0]); T[1] = fmaf(w, a0.y, T[1]); T[2] = fmaf(w, a0.z, T[2]); T[3] = fmaf(w, a0.w, T[3]);
      T[4] = fmaf(w, a1.x, T[4]); T[5] = fmaf(w, a1.y, T[5]); T[6] = fmaf(w, a1.z, T[6]); T[7] = fmaf(w, a1.w, T[7]);
      T[8] = fmaf(w, a2.x, T[8]); T[9] = fmaf(w, a2.y, T[9]); T[10] = fmaf(w, a2.z, T[10]); T[11] = fmaf(w, a2.w, T[11]);
    }
    float x = acc[p][0], y = acc[p][1], z = acc[p][2];
    float ox = T[0] * x + T[1] * y + T[2] * z + T[9] + tr_s[p * 3 + 0];
    float oy = T[3] * x + T[4] * y + T[5] * z + T[10] + tr_s[p * 3 + 1];
    float oz = T[6] * x + T[7] * y + T[8] * z + T[11] + tr_s[p * 3 + 2];
    float* o = out + ((size_t)(b0 + p) * n_verts + vi) * 3;
    o[0] = ox; o[1] = oy; o[2] = oz;
  }
}

// extra vertex joints + barycentric landmarks (VertexJointSelector / vertices2landmarks)
__global__ void lbs_gather_kernel(const float* __restrict__ verts, int n_verts, const int32_t* __restrict__ extra_idx,
                                  int n_extra, const int32_t* __restrict__ lmk_idx,
                                  const float* __restrict__ lmk_bary, int n_lmk, int J, int n_out,
                                  float* __restrict__ joints, int64_t B) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int per = n_extra + n_lmk;
  if (i >= B * per) return;
  const int64_t b = i / per;
  const int k = (int)(i % per);
  const float* vb = verts + (size_t)b * n_verts * 3;
  float o[3];
  if (k < n_extra) {
    const float* s = vb + (size_t)extra_idx[k] * 3;
    o[0] = s[0]; o[1] = s[1]; o[2] = s[2];
  } else {
    const int l = k - n_extra;
    o[0] = o[1] = o[2] = 0.f;
    for (int f = 0; f < 3; ++f) {
      const float* s = vb + (size_t)lmk_idx[l * 3 + f] * 3;
      float w = lmk_bary[l * 3 + f];
      o[0] = fmaf(w, s[0], o[0]); o[1] = fmaf(w, s[1], o[1]); o[2] = fmaf(w, s[2], o[2]);
    }
  }
  float* jo = joints + ((size_t)b * n_out + J + k) * 3;
  jo[0] = o[0]; jo[1] = o[1]; jo[2] = o[2];
}

// ------------------------------------------------------------------ workspace
size_t lbs_ws_bytes(const dpb_lbs* h, int64_t B, bool compact) {
  size_t n = 0;
  n += align_up((size_t)B * h->J * 12 * 4, 256) * 2;  // A, G
  n += align_up((size_t)B * h->P * 4, 256);
  n += align_up((size_t)B * h->J * 3 * 4, 256);
  n += align_up((size_t)B * h->n_need * 3 * 4, 256) * (compact ? 2 : 1);   // compact verts + gextra
  n += align_up((size_t)B * h->J * 12 * 4, 256) + align_up((size_t)B * h->P * 4, 256) +
       align_up((size_t)B * (h->S + 3) * 4, 256);
  n += lbs_tc_ws_bytes(h, B);
  return n + 2048;
}

bool lbs_carve(const dpb_lbs* h, int64_t B, bool compact, void* ws, size_t ws_bytes, LbsWs* out) {
  WsCarver c(ws, ws_bytes);
  out->A = c.take<float>((size_t)B * h->J * 12);
  out->G = c.take<float>((size_t)B * h->J * 12);
  out->feat = c.take<float>((size_t)B * h->P);
  out->jrest = c.take<float>((size_t)B * h->J * 3);
  out->gA = c.take<float>((size_t)B * h->J * 12);
  out->gfeat = c.take<float>((size_t)B * h->P);
  out->gextra = c.take<float>((size_t)B * h->n_need * 3 + 1);
  out->gbeta = c.take<float>((size_t)B * (h->S + 3));
  out->compact = compact ? c.take<float>((size_t)B * h->n_need * 3) : nullptr;
  out->featop = nullptr;
  out->skinop = nullptr;
  if (h->tc_ready && (!compact || h->sub)) {   // joints-only calls run the compact vertex set on the same operands
    c.off = align_up(c.off, 1024);
    out->featop = reinterpret_cast<__half*>(c.base + c.off);
    const int64_t B_pad = (B + 127) / 128 * 128;
    c.off += align_up((size_t)B_pad * h->kext * sizeof(__half), 1024);
    out->skinop = reinterpret_cast<__half*>(c.base + c.off);
    c.off += align_up((size_t)B_pad * 12 * 2 * h->jp * sizeof(__half), 1024);
  }
  return ws != nullptr && c.ok();
}


}  // namespace dpb

using namespace dpb;

template <class T>
static int upload(T** dst, const T* src, size_t n) {
  DPB_CUDA_CHECK(cudaMalloc((void**)dst, std::max<size_t>(n, 1) * sizeof(T)));
  if (n) DPB_CUDA_CHECK(cudaMemcpy(*dst, src, n * sizeof(T), cudaMemcpyHostToDevice));
  return DPB_OK;
}

namespace dpb { int lbs_tc_prepare(dpb_lbs* h, const dpb_body_tensors* m); void lbs_tc_release(dpb_lbs* h); }

extern "C" int dpb_lbs_create(dpb_lbs_t** out, const dpb_body_tensors* m, int device) {
  if (!out || !m) return fail(DPB_EINVAL, "dpb_lbs_create: null argument");
  DPB_REQUIRE(m->V > 0 && m->J > 0 && m->J <= 64 && m->S >= 0, "dpb_lbs_create: need V>0, 0<J<=64, S>=0");
  DPB_REQUIRE(m->v_template && m->shapedirs && m->posedirs && m->J_regressor && m->lbs_weights && m->parents,
              "dpb_lbs_create: missing body tensor");
  DPB_REQUIRE(m->parents[0] == -1, "dpb_lbs_create: parents[0] must be -1");
  for (int j = 1; j < m->J; ++j)
    DPB_REQUIRE(m->parents[j] >= 0 && m->parents[j] < j, "dpb_lbs_create: parents[i] must satisfy 0 <= parents[i] < i");
  for (int i = 0; i < m->n_extra; ++i)
    DPB_REQUIRE(m->extra_vids[i] >= 0 && m->extra_vids[i] < m->V, "dpb_lbs_create: extra vertex id out of range");
  for (int i = 0; i < m->n_lmk * 3; ++i)
    DPB_REQUIRE(m->lmk_faces[i] >= 0 && m->lmk_faces[i] < m->V, "dpb_lbs_create: landmark vertex id out of range");
  DeviceGuard guard(device);
  dpb_lbs* h = new dpb_lbs();
  h->device = device;
  cudaDeviceProp prop;
  DPB_CUDA_CHECK(cudaGetDeviceProperties(&prop, device));
  h->sm_count = prop.multiProcessorCount;
  const int V = h->V = m->V, J = h->J = m->J, S = h->S = m->S;
  h->P = (J - 1) * 9;
  h->n_extra = m->n_extra;
  h->n_lmk = m->n_lmk;
  h->n_out = J + m->n_extra + m->n_lmk;
  h->parents_h.assign(m->parents, m->parents + J);
  std::vector<int32_t> depth(J, 0);
  for (int j = 1; j < J; ++j) depth[j] = depth[m->parents[j]] + 1;
  h->max_depth = *std::max_element(depth.begin(), depth.end());
  // fold the joint regressor: J_template = Jreg . v_template, J_shapedirs = Jreg . shapedirs (fp64 accumulate)
  std::vector<float> jt((size_t)J * 3), js((size_t)J * 3 * std::max(S, 1));
  for (int j = 0; j < J; ++j)
    for (int c = 0; c < 3; ++c) {
      double a = 0;
      for (int v = 0; v < V; ++v) a += (double)m->J_regressor[(size_t)j * V + v] * m->v_template[(size_t)v * 3 + c];
      jt[j * 3 + c] = (float)a;
      for (int s = 0; s < S; ++s) {
        double q = 0;
        for (int v = 0; v < V; ++v)
          q += (double)m->J_regressor[(size_t)j * V + v] * m->shapedirs[((size_t)v * 3 + c) * S + s];
        js[((size_t)j * 3 + c) * S + s] = (float)q;
      }
    }
  // ELL skinning weights (non-zeros in ascending joint order, like the dense sum)
  int nnz = 1;
  for (int v = 0; v < V; ++v) {
    int c = 0;
    for (int j = 0; j < J; ++j) c += m->lbs_weights[(size_t)v * J + j] != 0.f;
    nnz = std::max(nnz, c);
  }
  h->nnz = nnz;
  std::vector<int32_t> eidx((size_t)nnz * V, 0);
  std::vector<float> ew((size_t)nnz * V, 0.f);
  for (int v = 0; v < V; ++v) {
    int c = 0;
    for (int j = 0; j < J; ++j) {
      float w = m->lbs_weights[(size_t)v * J + j];
      if (w != 0.f) { eidx[(size_t)c * V + v] = j; ew[(size_t)c * V + v] = w; ++c; }
    }
  }
  // compact vertex set for the joints-only mode
  std::vector<int32_t> need;
  for (int i = 0; i < m->n_extra; ++i) need.push_back(m->extra_vids[i]);
  for (int i = 0; i < m->n_lmk * 3; ++i) need.push_back(m->lmk_faces[i]);
  std::sort(need.begin(), need.end());
  need.erase(std::unique(need.begin(), need.end()), need.end());
  std::map<int32_t, int32_t> pos;
  for (size_t i = 0; i < need.size(); ++i) pos[need[i]] = (int32_t)i;
  std::vector<int32_t> nidx(V, -1);
  for (size_t i = 0; i < need.size(); ++i) nidx[need[i]] = (int32_t)i;
  std::vector<int32_t> epos(std::max(m->n_extra, 1)), lpos(std::max(m->n_lmk * 3, 1));
  for (int i = 0; i < m->n_extra; ++i) epos[i] = pos[m->extra_vids[i]];
  for (int i = 0; i < m->n_lmk * 3; ++i) lpos[i] = pos[m->lmk_faces[i]];
  h->n_need = (int)need.size();

  int rc = DPB_OK;
#define UP(dst, src, n) if (rc == DPB_OK) rc = upload(&h->dst, src, (size_t)(n))
  UP(v_template, m->v_template, V * 3);
  UP(shapedirs, m->shapedirs, (size_t)V * 3 * S);
  UP(posedirs, m->posedirs, (size_t)h->P * V * 3);
  UP(j_template, jt.data(), J * 3);
  UP(j_shapedirs, js.data(), (size_t)J * 3 * S);
  std::vector<float> jsT((size_t)S * 3 * J);
  for (int q = 0; q < 3 * J; ++q)
    for (int k = 0; k < S; ++k) jsT[(size_t)k * 3 * J + q] = js[(size_t)q * S + k];
  UP(j_shapedirsT, jsT.data(), (size_t)S * 3 * J);
  UP(parents, m->parents, J);
  UP(depth, depth.data(), J);
  std::vector<int32_t> cptr(J + 1, 0), cidx(J > 1 ? J - 1 : 1, 0);
  for (int j = 1; j < J; ++j) cptr[m->parents[j] + 1]++;
  for (int j = 0; j < J; ++j) cptr[j + 1] += cptr[j];
  {
    std::vector<int32_t> fill(cptr.begin(), cptr.end() - 1);
    for (int j = 1; j < J; ++j) cidx[fill[m->parents[j]]++] = j;
  }
  UP(child_ptr, cptr.data(), J + 1);
  UP(child_idx, cidx.data(), J > 1 ? J - 1 : 1);
  UP(ell_idx, eidx.data(), (size_t)nnz * V);
  UP(ell_w, ew.data(), (size_t)nnz * V);
  UP(extra_vids, m->extra_vids, m->n_extra);
  UP(lmk_faces, m->lmk_faces, m->n_lmk * 3);
  UP(lmk_bary, m->lmk_bary, m->n_lmk * 3);
  UP(need_vids, need.data(), need.size());
  UP(extra_pos, epos.data(), m->n_extra);
  UP(lmk_pos, lpos.data(), m->n_lmk * 3);
  UP(need_index, nidx.data(), V);
#undef UP
  if (rc == DPB_OK) rc = lbs_tc_prepare(h, m);
  if (rc == DPB_OK) rc = lbs_bwd_prepare(h, m);
  if (rc == DPB_OK && h->tc_ready) rc = lbs_bwd_tc_prepare(h, m);
  if (rc == DPB_OK && h->bt_ready) rc = lbs_skin_bwd_tc_prepare(h, m);
  if (rc == DPB_OK && h->tc_ready && h->n_need > 0) {
    // the compact vertex set as a small body model (no extra joints / landmarks of its own: no recursion)
    const int Vn = h->n_need, P = h->P;
    std::vector<float> vt((size_t)Vn * 3), sd((size_t)Vn * 3 * std::max(S, 1)), pd((size_t)P * Vn * 3),
        lw((size_t)Vn * J), jr((size_t)J * Vn, 0.f);
    for (int i = 0; i < Vn; ++i) {
      const int v = need[i];
      for (int c = 0; c < 3; ++c) {
        vt[(size_t)i * 3 + c] = m->v_template[(size_t)v * 3 + c];
        for (int k = 0; k < S; ++k) sd[((size_t)i * 3 + c) * S + k] = m->shapedirs[((size_t)v * 3 + c) * S + k];
        for (int k = 0; k < P; ++k) pd[(size_t)k * Vn * 3 + (size_t)i * 3 + c] = m->posedirs[(size_t)k * V * 3 + (size_t)v * 3 + c];
      }
      for (int j = 0; j < J; ++j) lw[(size_t)i * J + j] = m->lbs_weights[(size_t)v * J + j];
    }
    dpb_body_tensors ms = *m;
    ms.V = Vn;
    ms.v_template = vt.data(); ms.shapedirs = sd.data(); ms.posedirs = pd.data();
    ms.lbs_weights = lw.data(); ms.J_regressor = jr.data();
    ms.n_extra = 0; ms.extra_vids = nullptr; ms.n_lmk = 0; ms.lmk_faces = nullptr; ms.lmk_bary = nullptr;
    rc = dpb_lbs_create(&h->sub, &ms, device);
  }
  if (rc != DPB_OK) { dpb_lbs_destroy(h); return rc; }
  *out = h;
  return DPB_OK;
}

extern "C" int dpb_lbs_destroy(dpb_lbs_t* h) {
  if (!h) return DPB_OK;
  DeviceGuard guard(h->device);
  if (h->sub) dpb_lbs_destroy(h->sub);
  h->sub = nullptr;
  lbs_tc_release(h);
  lbs_bwd_release(h);
  lbs_bwd_tc_release(h);
  lbs_skin_bwd_tc_release(h);
  void* ptrs[] = {h->v_template, h->shapedirs, h->posedirs, h->j_template, h->j_shapedirs, h->j_shapedirsT, h->parents, h->depth, h->child_ptr, h->child_idx,
                  h->ell_idx, h->ell_w, h->extra_vids, h->lmk_faces, h->lmk_bary, h->need_vids, h->extra_pos,
                  h->lmk_pos, h->need_index};
  for (void* p : ptrs) if (p) cudaFree(p);
  delete h;
  return DPB_OK;
}

extern "C" int dpb_lbs_num_joints_out(dpb_lbs_t* h) { return h ? h->n_out : DPB_EINVAL; }

extern "C" int dpb_lbs_set_const_tail(dpb_lbs_t* h, int n_var, const float* tail_pose) {
  if (!h) return fail(DPB_EINVAL, "dpb_lbs_set_const_tail: null handle");
  DPB_REQUIRE(n_var >= 1 && n_var < h->J && tail_pose, "dpb_lbs_set_const_tail: need 1 <= n_var < J and a tail pose");
  DeviceGuard guard(h->device);
  if (h->sub) {
    int rc = lbs_tc_make_tail(h->sub, n_var, tail_pose);
    if (rc != DPB_OK) return rc;
  }
  return lbs_tc_make_tail(h, n_var, tail_pose);
}

extern "C" size_t dpb_lbs_workspace_bytes(dpb_lbs_t* h, int64_t B, int flags) {
  (void)flags;
  if (!h || B <= 0) return 0;
  return lbs_ws_bytes(h, B, true);
}

extern "C" int dpb_lbs_forward(dpb_lbs_t* h, const float* betas, const float* full_pose, const float* transl,
                               float* verts, float* joints, int64_t B, int flags, void* ws, size_t ws_bytes,
                               void* stream) {
  if (!h) return fail(DPB_EINVAL, "dpb_lbs_forward: null handle");
  DeviceGuard guard(h->device);
  DPB_REQUIRE(betas && full_pose && joints, "dpb_lbs_forward: betas, full_pose and joints are required");
  if (B <= 0) return DPB_OK;
  cudaStream_t st = (cudaStream_t)stream;
  const bool compact = (verts == nullptr);
  LbsWs w;
  if (!lbs_carve(h, B, compact, ws, ws_bytes, &w)) return fail(DPB_ENOMEM, "dpb_lbs_forward: workspace too small");
  const int engine = flags & DPB_ENGINE_MASK;
  const int n_verts = compact ? h->n_need : h->V;
  float* vout = compact ? w.compact : verts;
  // hv = the body model whose vertices this call produces: the full one, or the compact set of the joints-only mode
  dpb_lbs* hv = compact ? h->sub : h;
  const bool use_tc = n_verts > 0 && hv && hv->tc_ready && w.featop &&
                      (engine == DPB_LBS_ENGINE_TC || (engine == DPB_ENGINE_AUTO && B >= 64));
  // const-tail calls (DPB_LBS_CONST_TAIL) read the pruned basis; everything else the full one
  const bool want_tail = (flags & DPB_LBS_CONST_TAIL) != 0;
  if (want_tail) DPB_REQUIRE(h->tailv.n_var > 0 || !h->tc_ready, "dpb_lbs_forward: DPB_LBS_CONST_TAIL without dpb_lbs_set_const_tail");
  // (the compact model's variants have the same K layout: the pose kernel's operands serve both)
  const LbsVariant var = !use_tc ? ((want_tail && h->tailv.dirs16) ? h->tailv : lbs_full_variant(h))
                                 : ((want_tail && hv->tailv.dirs16) ? hv->tailv : lbs_full_variant(hv));
  // blend + skinning in one CTA-pair kernel, chosen by the padded joint count: the 128-pose-group kernel for one
  // skinning K slab (jp = 32, SMPL), the 96-pose-group kernel for two (jp = 64, SMPL-X)
  const bool use_fused3 = use_tc && w.skinop && lbs_fused3_fits(hv, var);
  const bool use_fused = use_fused3 || (use_tc && w.skinop && lbs_fused2_fits(hv, var));
  // the fused kernel's operands come straight out of the pose kernel (pad rows of the last pose group are zeroed)
  __half* fop = use_fused ? w.featop : nullptr;
  __half* sop = use_fused ? w.skinop : nullptr;
  if (use_fused) {
    const int64_t B_pad = (B + 127) / 128 * 128;
    if (B_pad > B) {
      DPB_CUDA_CHECK(cudaMemsetAsync(w.featop + (size_t)B * var.kext, 0, (size_t)(B_pad - B) * var.kext * sizeof(__half), st));
      DPB_CUDA_CHECK(cudaMemsetAsync(w.skinop + (size_t)B * 12 * 2 * h->jp, 0,
                                     (size_t)(B_pad - B) * 12 * 2 * h->jp * sizeof(__half), st));
    }
  }
  // forward-only fused calls (DPB_LBS_NO_SAVE): nothing downstream reads the fp32 transforms / features
  const bool no_save = (flags & DPB_LBS_NO_SAVE) && use_fused;
  float* A_o = no_save ? nullptr : w.A;
  float* G_o = no_save ? nullptr : w.G;
  float* feat_o = no_save ? nullptr : w.feat;
  float* jrest_o = no_save ? nullptr : w.jrest;
  const unsigned pose_grid = (unsigned)((B + 3) / 4);
  if (h->J > 32)
    lbs_pose_kernel<2><<<pose_grid, 128, 0, st>>>(betas, full_pose, transl, h->j_template, h->j_shapedirsT, h->parents,
                                                   h->depth, h->J, h->S, h->max_depth, A_o, G_o, feat_o, jrest_o,
                                                   joints, h->n_out, B, fop, var.kext / 2, var.p_feat, sop, h->jp);
  else
    lbs_pose_kernel<1><<<pose_grid, 128, 0, st>>>(betas, full_pose, transl, h->j_template, h->j_shapedirsT, h->parents,
                                                   h->depth, h->J, h->S, h->max_depth, A_o, G_o, feat_o, jrest_o,
                                                   joints, h->n_out, B, fop, var.kext / 2, var.p_feat, sop, h->jp);
  DPB_CUDA_CHECK(cudaGetLastError());
  if (n_verts > 0) {
    if (!compact && engine == DPB_LBS_ENGINE_TC && !use_tc)
      return fail(DPB_EUNSUPPORTED, "dpb_lbs_forward: tensor-core engine unavailable");
    if (use_tc) {
      if (use_fused) {
        // the blended vertices stay in TMEM
        int rc = use_fused3 ? lbs_fused3(hv, var, w.featop, w.skinop, vout, B, st)
                            : lbs_fused2(hv, var, w.featop, w.skinop, vout, B, st);
        if (rc != DPB_OK) return rc;
      } else {
      // blend on tcgen05 (writes v_posed into verts), then skin in place with the transforms from the pose kernel
      int rc = lbs_tc_blend(hv, var, betas, w.feat, w.featop, vout, B, st);
      if (rc != DPB_OK) return rc;
      if (lbs_tc_skin_fits(hv)) {
        rc = lbs_tc_skin(hv, w.A, transl, w.skinop, vout, B, st);
        if (rc != DPB_OK) return rc;
      } else {
      size_t smem = ((size_t)LBS_TP * h->J * 12 + LBS_TP * 3) * 4;
      DPB_CUDA_CHECK(cudaFuncSetAttribute(lbs_vertex_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
      dim3 grid((n_verts + LBS_TV - 1) / LBS_TV, (unsigned)((B + LBS_TP - 1) / LBS_TP));
      DPB_REQUIRE(grid.y <= 65535u, "dpb_lbs_forward: batch too large for one call (max 65535*16 poses)");
      lbs_vertex_kernel<<<grid, LBS_TV, smem, st>>>(betas, transl, w.feat, w.A, hv->v_template, hv->shapedirs,
                                                    hv->posedirs, hv->ell_idx, hv->ell_w, nullptr, n_verts, hv->V, h->J,
                                                    0, 0, hv->nnz, vout, vout, B);
      DPB_CUDA_CHECK(cudaGetLastError());
      }
      }
    } else {
      size_t smem = ((size_t)h->P * LBS_TP + (size_t)h->S * LBS_TP + (size_t)LBS_TP * h->J * 12 + LBS_TP * 3) * 4;
      DPB_CUDA_CHECK(cudaFuncSetAttribute(lbs_vertex_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
      dim3 grid((n_verts + LBS_TV - 1) / LBS_TV, (unsigned)((B + LBS_TP - 1) / LBS_TP));
      DPB_REQUIRE(grid.y <= 65535u, "dpb_lbs_forward: batch too large for one call (max 65535*16 poses)");
      lbs_vertex_kernel<<<grid, LBS_TV, smem, st>>>(betas, transl, w.feat, w.A, h->v_template, h->shapedirs,
                                                    h->posedirs, h->ell_idx, h->ell_w,
                                                    compact ? h->need_vids : nullptr, n_verts, h->V, h->J, h->S, h->P,
                                                    h->nnz, nullptr, vout, B);
      DPB_CUDA_CHECK(cudaGetLastError());
    }
  }
  const int per = h->n_extra + h->n_lmk;
  if (per > 0) {
    int64_t n = B * per;
    lbs_gather_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(
        vout, n_verts, compact ? h->extra_pos : h->extra_vids, h->n_extra, compact ? h->lmk_pos : h->lmk_faces,
        h->lmk_bary, h->n_lmk, h->J, h->n_out, joints, B);
    DPB_CUDA_CHECK(cudaGetLastError());
  }
  return DPB_OK;
}
