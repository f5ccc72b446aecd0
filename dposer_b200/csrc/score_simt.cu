// fp32 engine of the score network: time-path table, tiled SGEMM with per-row time bias,
// GroupNorm+SiLU(+residual).  This is the exact path (fp32 FFMA, fp32 accumulate); the
// tcgen05 engine in score_tc.cu is the throughput path and is validated against this one
// on the device as well as against the CPU oracle.
//
// Math follows ScoreModelFC.forward (reference lib/algorithms/advanced/model.py:141-196).
#include "score.h"
#include "train.h"

namespace dpb {

// ------------------------------------------------------------------ time path
// grid: (ceil(n / TT_LABELS), TT_SPLIT) CTAs of 256 threads.  A CTA handles TT_LABELS labels (weights are
// read once per TT_LABELS labels); blockIdx.y selects 1/TT_SPLIT of the 5x1024 projection outputs.  The
// 512x512 shared embed is recomputed by every split (cheap) so a single label still spreads over TT_SPLIT SMs.
constexpr int TT_LABELS = 8;
constexpr int TT_SPLIT = 16;

struct PtrPack {
  const float* t_w[5];
  const float* t_b[5];
  const float* lin_b[5];
};

__global__ void __launch_bounds__(256) time_table_kernel(
    const float* __restrict__ labels, int n, const float* __restrict__ freqs,
    const float* __restrict__ temb_w, const float* __restrict__ temb_b,
    const PtrPack p, float* __restrict__ table) {
  __shared__ float emb0[TT_LABELS][E];
  __shared__ float emb1[TT_LABELS][E];
  const int l0 = blockIdx.x * TT_LABELS;
  const int nl = min(TT_LABELS, n - l0);
  // sinusoidal embedding: [sin(label*f_k) | cos(label*f_k)]  (model.py:37-51)
  for (int i = threadIdx.x; i < TT_LABELS * E; i += blockDim.x) {
    int li = i / E, c = i % E;
    float v = 0.f;
    if (li < nl) {
      float arg = labels[l0 + li] * freqs[c % (E / 2)];
      v = (c < E / 2) ? sinf(arg) : cosf(arg);
    }
    emb0[li][c] = v;
  }
  __syncthreads();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  // shared_time_embed: temb = SiLU(W_s emb0 + b_s)   (model.py:124-127,164)
  for (int o = warp; o < E; o += 8) {
    float acc[TT_LABELS];
#pragma unroll
    for (int li = 0; li < TT_LABELS; ++li) acc[li] = 0.f;
    const float* wr = temb_w + (size_t)o * E;
    for (int k = lane; k < E; k += 32) {
      float w = wr[k];
#pragma unroll
      for (int li = 0; li < TT_LABELS; ++li) acc[li] = fmaf(w, emb0[li][k], acc[li]);
    }
#pragma unroll
    for (int li = 0; li < TT_LABELS; ++li) {
      float v = acc[li];
      for (int s = 16; s > 0; s >>= 1) v += __shfl_xor_sync(0xffffffffu, v, s);
      if (lane == 0) {
        v += temb_b[o];
        emb1[li][o] = v / (1.0f + expf(-v));
      }
    }
  }
  __syncthreads();
  // five projections W_lt temb + b_lt, with the x-path bias b_l folded in
  constexpr int PER_SPLIT = NL * H / TT_SPLIT;
  for (int oo = warp; oo < PER_SPLIT; oo += 8) {
    const int o = blockIdx.y * PER_SPLIT + oo;
    const int layer = o / H, c = o % H;
    float acc[TT_LABELS];
#pragma unroll
    for (int li = 0; li < TT_LABELS; ++li) acc[li] = 0.f;
    const float* wr = p.t_w[layer] + (size_t)c * E;
    for (int k = lane; k < E; k += 32) {
      float w = wr[k];
#pragma unroll
      for (int li = 0; li < TT_LABELS; ++li) acc[li] = fmaf(w, emb1[li][k], acc[li]);
    }
#pragma unroll
    for (int li = 0; li < TT_LABELS; ++li) {
      float v = acc[li];
      for (int s = 16; s > 0; s >>= 1) v += __shfl_xor_sync(0xffffffffu, v, s);
      if (lane == 0 && li < nl)
        table[((size_t)(l0 + li) * NL + layer) * H + c] = (v + p.t_b[layer][c]) + p.lin_b[layer][c];
    }
  }
}

// ------------------------------------------------------------------ SGEMM  C = A W^T + bias
// A [M,K] row-major, W [N,K] row-major, C [M,N].  64x64 tile, BK=16, 256 threads, 4x4 micro-tile.
// bias: table + layer*H, row -> entry t_index[m] (stride NL*H) or entry 0; bias==nullptr -> none.
constexpr int BM = 64, BN = 64, BK = 16;

__global__ void __launch_bounds__(256) sgemm_bias_kernel(const float* __restrict__ A, const float* __restrict__ W,
                                                         float* __restrict__ C, int64_t M, int N, int K,
                                                         const float* __restrict__ bias,
                                                         const int32_t* __restrict__ t_index, int bias_stride,
                                                         const float* __restrict__ col_bias, int64_t bias_rows) {
  __shared__ float As[BK][BM + 4];
  __shared__ float Ws[BK][BN + 4];
  const int tid = threadIdx.x;
  const int64_t m0 = (int64_t)blockIdx.y * BM;
  const int n0 = blockIdx.x * BN;
  const int tx = tid & 15, ty = tid >> 4;  // micro-tile: rows ty*4.., cols tx*4..
  // loader mapping: each thread loads one float4 of A and one of W per k-tile
  const int lr = tid >> 2, lk = (tid & 3) * 4;  // row 0..63, k offset 0,4,8,12
  float acc[4][4] = {};
  for (int k0 = 0; k0 < K; k0 += BK) {
    float4 a = make_float4(0.f, 0.f, 0.f, 0.f);
    if (m0 + lr < M) a = *reinterpret_cast<const float4*>(A + (m0 + lr) * K + k0 + lk);
    float4 w = *reinterpret_cast<const float4*>(W + (size_t)(n0 + lr) * K + k0 + lk);
    As[lk + 0][lr] = a.x; As[lk + 1][lr] = a.y; As[lk + 2][lr] = a.z; As[lk + 3][lr] = a.w;
    Ws[lk + 0][lr] = w.x; Ws[lk + 1][lr] = w.y; Ws[lk + 2][lr] = w.z; Ws[lk + 3][lr] = w.w;
    __syncthreads();
#pragma unroll
    for (int kk = 0; kk < BK; ++kk) {
      float4 av = *reinterpret_cast<const float4*>(&As[kk][ty * 4]);
      float4 wv = *reinterpret_cast<const float4*>(&Ws[kk][tx * 4]);
      float ar[4] = {av.x, av.y, av.z, av.w}, wr[4] = {wv.x, wv.y, wv.z, wv.w};
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(ar[i], wr[j], acc[i][j]);
    }
    __syncthreads();
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    int64_t m = m0 + ty * 4 + i;
    if (m >= M) continue;
    const bool biased = m < bias_rows;          // rows beyond carry tangents (JVP): the affine part drops out
    const float* brow = nullptr;
    if (bias && biased) brow = bias + (size_t)(t_index ? t_index[m] : 0) * bias_stride;
    float4 o;
    float* op = &o.x;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      int n = n0 + tx * 4 + j;
      float v = acc[i][j];
      if (brow) v += brow[n];
      if (col_bias && biased) v += col_bias[n];
      op[j] = v;
    }
    *reinterpret_cast<float4*>(C + m * N + n0 + tx * 4) = o;
  }
}

// ------------------------------------------------------------------ GroupNorm(32x32) + SiLU (+ residual)
// one CTA (256 threads) per row; thread owns 4 consecutive channels; a group = 8 consecutive lanes.
__global__ void __launch_bounds__(256) gn_silu_kernel(const float* __restrict__ in, const float* __restrict__ gamma,
                                                      const float* __restrict__ beta,
                                                      const float* residual, float* out, int64_t M) {
  // residual and out may alias (in-place residual update of the stream h)
  const int64_t m = blockIdx.x;
  if (m >= M) return;
  const int c = threadIdx.x * 4;
  float4 v = *reinterpret_cast<const float4*>(in + m * H + c);
  float s = (v.x + v.y) + (v.z + v.w);
  s += __shfl_xor_sync(0xffffffffu, s, 1);
  s += __shfl_xor_sync(0xffffffffu, s, 2);
  s += __shfl_xor_sync(0xffffffffu, s, 4);
  const float mean = s * (1.0f / GROUP);
  float dx = v.x - mean, dy = v.y - mean, dz = v.z - mean, dw = v.w - mean;
  float q = (dx * dx + dy * dy) + (dz * dz + dw * dw);
  q += __shfl_xor_sync(0xffffffffu, q, 1);
  q += __shfl_xor_sync(0xffffffffu, q, 2);
  q += __shfl_xor_sync(0xffffffffu, q, 4);
  const float rstd = 1.0f / sqrtf(q * (1.0f / GROUP) + GN_EPS);  // biased variance, eps 1e-5
  float4 g = *reinterpret_cast<const float4*>(gamma + c);
  float4 b = *reinterpret_cast<const float4*>(beta + c);
  float y[4] = {dx * rstd * g.x + b.x, dy * rstd * g.y + b.y, dz * rstd * g.z + b.z, dw * rstd * g.w + b.w};
  float4 o;
  float* op = &o.x;
#pragma unroll
  for (int i = 0; i < 4; ++i) op[i] = y[i] / (1.0f + expf(-y[i]));
  if (residual) {
    float4 r = *reinterpret_cast<const float4*>(residual + m * H + c);
    o.x += r.x; o.y += r.y; o.z += r.z; o.w += r.w;
  }
  *reinterpret_cast<float4*>(out + m * H + c) = o;
}

// Forward-mode twin of gn_silu_kernel: row m of `in` is the primal pre-activation, row M + m its tangent; writes
// SiLU(GN(h)) and its directional derivative (+ the residual stream's primal / tangent).  GroupNorm's JVP inside a
// group: n = (h - mu) rstd,  dn = rstd (dh - mean(dh)) - n rstd mean(n dh);  SiLU'(y) = s + y s (1 - s), s = sigmoid(y).
__global__ void __launch_bounds__(256) gn_silu_jvp_kernel(const float* __restrict__ in, const float* __restrict__ gamma,
                                                          const float* __restrict__ beta, const float* residual,
                                                          float* out, int64_t M) {
  const int64_t m = blockIdx.x;
  if (m >= M) return;
  const int c = threadIdx.x * 4;
  const float4 v = *reinterpret_cast<const float4*>(in + m * H + c);
  const float4 d = *reinterpret_cast<const float4*>(in + (M + m) * H + c);
  auto gsum = [](float s) {
    s += __shfl_xor_sync(0xffffffffu, s, 1);
    s += __shfl_xor_sync(0xffffffffu, s, 2);
    s += __shfl_xor_sync(0xffffffffu, s, 4);
    return s;
  };
  const float mean = gsum((v.x + v.y) + (v.z + v.w)) * (1.0f / GROUP);
  const float dmean = gsum((d.x + d.y) + (d.z + d.w)) * (1.0f / GROUP);
  const float hx[4] = {v.x - mean, v.y - mean, v.z - mean, v.w - mean};
  const float dx[4] = {d.x - dmean, d.y - dmean, d.z - dmean, d.w - dmean};
  const float q = gsum((hx[0] * hx[0] + hx[1] * hx[1]) + (hx[2] * hx[2] + hx[3] * hx[3]));
  const float rstd = 1.0f / sqrtf(q * (1.0f / GROUP) + GN_EPS);
  float n[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) n[i] = hx[i] * rstd;
  const float ndh = gsum((n[0] * dx[0] + n[1] * dx[1]) + (n[2] * dx[2] + n[3] * dx[3])) * (1.0f / GROUP);
  const float4 g = *reinterpret_cast<const float4*>(gamma + c);
  const float4 b = *reinterpret_cast<const float4*>(beta + c);
  const float gg[4] = {g.x, g.y, g.z, g.w}, bb[4] = {b.x, b.y, b.z, b.w};
  float4 o, od;
  float *op = &o.x, *odp = &od.x;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const float y = n[i] * gg[i] + bb[i];
    const float dy = gg[i] * rstd * (dx[i] - n[i] * ndh);
    const float sg = 1.0f / (1.0f + expf(-y));
    op[i] = y * sg;
    odp[i] = dy * (sg + y * sg * (1.0f - sg));
  }
  if (residual) {
    const float4 r = *reinterpret_cast<const float4*>(residual + m * H + c);
    const float4 rd = *reinterpret_cast<const float4*>(residual + (M + m) * H + c);
    o.x += r.x; o.y += r.y; o.z += r.z; o.w += r.w;
    od.x += rd.x; od.y += rd.y; od.z += rd.z; od.w += rd.w;
  }
  *reinterpret_cast<float4*>(out + m * H + c) = o;
  *reinterpret_cast<float4*>(out + (M + m) * H + c) = od;
}

// x [B,D] -> xpad [B,PDP]  (D = 63 / 126, PDP = 64 / 128)
template <int PDP>
__global__ void pad_x_kernel(const float* __restrict__ x, float* __restrict__ xp, int64_t B) {
  constexpr int PD = pose_dim_of(PDP);
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= B * PDP) return;
  int64_t r = i / PDP;
  int c = (int)(i % PDP);
  xp[i] = (c < PD) ? x[r * PD + c] : 0.f;
}

static void launch_pad_x(const float* x, float* xp, int64_t B, int dp, cudaStream_t st) {
  const int64_t n = B * dp;
  if (dp == DP128) pad_x_kernel<DP128><<<(unsigned)((n + 255) / 256), 256, 0, st>>>(x, xp, B);
  else pad_x_kernel<DP><<<(unsigned)((n + 255) / 256), 256, 0, st>>>(x, xp, B);
}

int simt_time_table(dpb_score* h, const float* labels, int n, float* table, cudaStream_t st) {
  if (n <= 0) return DPB_OK;
  // pointer tables live in constant kernel-parameter space (no device allocation in the call)
  PtrPack p;
  for (int l = 0; l < NL; ++l) { p.t_w[l] = h->t_w[l]; p.t_b[l] = h->t_b[l]; p.lin_b[l] = h->lin_b[l]; }
  dim3 grid((n + TT_LABELS - 1) / TT_LABELS, TT_SPLIT);
  time_table_kernel<<<grid, 256, 0, st>>>(labels, n, h->emb_freqs, h->temb_w, h->temb_b, p, table);
  DPB_CUDA_CHECK(cudaGetLastError());
  return DPB_OK;
}

size_t simt_forward_ws_bytes(int64_t B, int dp) {
  // xpad [B,DP] + three [B,1024] fp32 buffers
  return align_up((size_t)B * dp * 4, 256) + 3 * align_up((size_t)B * H * 4, 256) + 1024;
}

int simt_forward_raw(dpb_score* h, const float* x, const float* table, const int32_t* t_index, float* raw,
                     int64_t B, void* ws, size_t ws_bytes, cudaStream_t st) {
  if (B <= 0) return DPB_OK;
  const int dp = h->pose_dp;
  WsCarver c(ws, ws_bytes);
  float* xp = c.take<float>((size_t)B * dp);
  float* pre = c.take<float>((size_t)B * H);   // pre-activation scratch
  float* hbuf = c.take<float>((size_t)B * H);  // residual stream
  float* tbuf = c.take<float>((size_t)B * H);  // block intermediate
  if (!c.ok() || ws == nullptr) return fail(DPB_ENOMEM, "score forward: workspace too small");
  const int stride = NL * H;
  dim3 gemm_grid(H / BN, (unsigned)((B + BM - 1) / BM));
  launch_pad_x(x, xp, B, dp, st);
  // pre_dense + pre_gnorm + act   (model.py:166-169)
  sgemm_bias_kernel<<<gemm_grid, 256, 0, st>>>(xp, h->pre_w, pre, B, H, dp, table, t_index, stride, nullptr, B);
  gn_silu_kernel<<<(unsigned)B, 256, 0, st>>>(pre, h->gn_w[0], h->gn_b[0], nullptr, hbuf, B);
  for (int blk = 0; blk < 2; ++blk) {  // model.py:172-187
    int l1 = 1 + 2 * blk, l2 = 2 + 2 * blk;
    sgemm_bias_kernel<<<gemm_grid, 256, 0, st>>>(hbuf, h->blk_w[l1 - 1], pre, B, H, H, table + (size_t)l1 * H,
                                                 t_index, stride, nullptr, B);
    gn_silu_kernel<<<(unsigned)B, 256, 0, st>>>(pre, h->gn_w[l1], h->gn_b[l1], nullptr, tbuf, B);
    sgemm_bias_kernel<<<gemm_grid, 256, 0, st>>>(tbuf, h->blk_w[l2 - 1], pre, B, H, H, table + (size_t)l2 * H,
                                                 t_index, stride, nullptr, B);
    gn_silu_kernel<<<(unsigned)B, 256, 0, st>>>(pre, h->gn_w[l2], h->gn_b[l2], hbuf, hbuf, B);
  }
  // post_dense (model.py:189), N padded to DP (64 or 128)
  dim3 post_grid(dp / BN, (unsigned)((B + BM - 1) / BM));
  sgemm_bias_kernel<<<post_grid, 256, 0, st>>>(hbuf, h->post_w, raw, B, dp, H, nullptr, nullptr, 0, h->post_b, B);
  DPB_CUDA_CHECK(cudaGetLastError());
  return DPB_OK;
}

// raw[0:B] = net(x) and raw[B:2B] = (d net / d x) v  (both before the sigma division), fp32 engine: every GEMM runs on
// the stacked rows [primal ; tangent] (the tangent rows skip the bias), every GroupNorm + SiLU on its forward-mode twin.
// ws: simt_forward_ws_bytes(2 B, DP).  Serves the Hutchinson divergence of lib/algorithms/advanced/likelihood.py:26-37:
// eps . (J eps) is the scalar the reference gets from autograd's eps . (J^T eps).
int simt_forward_jvp_raw(dpb_score* h, const float* x, const float* v, const float* table, const int32_t* t_index,
                         float* raw, int64_t B, void* ws, size_t ws_bytes, cudaStream_t st) {
  if (B <= 0) return DPB_OK;
  const int64_t B2 = 2 * B;
  const int dp = h->pose_dp;
  WsCarver c(ws, ws_bytes);
  float* xp = c.take<float>((size_t)B2 * dp);
  float* pre = c.take<float>((size_t)B2 * H);
  float* hbuf = c.take<float>((size_t)B2 * H);
  float* tbuf = c.take<float>((size_t)B2 * H);
  if (!c.ok() || ws == nullptr) return fail(DPB_ENOMEM, "score jvp: workspace too small");
  const int stride = NL * H;
  dim3 gemm_grid(H / BN, (unsigned)((B2 + BM - 1) / BM));
  launch_pad_x(x, xp, B, dp, st);
  launch_pad_x(v, xp + (size_t)B * dp, B, dp, st);
  sgemm_bias_kernel<<<gemm_grid, 256, 0, st>>>(xp, h->pre_w, pre, B2, H, dp, table, t_index, stride, nullptr, B);
  gn_silu_jvp_kernel<<<(unsigned)B, 256, 0, st>>>(pre, h->gn_w[0], h->gn_b[0], nullptr, hbuf, B);
  for (int blk = 0; blk < 2; ++blk) {
    int l1 = 1 + 2 * blk, l2 = 2 + 2 * blk;
    sgemm_bias_kernel<<<gemm_grid, 256, 0, st>>>(hbuf, h->blk_w[l1 - 1], pre, B2, H, H, table + (size_t)l1 * H,
                                                 t_index, stride, nullptr, B);
    gn_silu_jvp_kernel<<<(unsigned)B, 256, 0, st>>>(pre, h->gn_w[l1], h->gn_b[l1], nullptr, tbuf, B);
    sgemm_bias_kernel<<<gemm_grid, 256, 0, st>>>(tbuf, h->blk_w[l2 - 1], pre, B2, H, H, table + (size_t)l2 * H,
                                                 t_index, stride, nullptr, B);
    gn_silu_jvp_kernel<<<(unsigned)B, 256, 0, st>>>(pre, h->gn_w[l2], h->gn_b[l2], hbuf, hbuf, B);
  }
  dim3 post_grid(dp / BN, (unsigned)((B2 + BM - 1) / BM));
  sgemm_bias_kernel<<<post_grid, 256, 0, st>>>(hbuf, h->post_w, raw, B2, dp, H, nullptr, nullptr, 0, h->post_b, B);
  DPB_CUDA_CHECK(cudaGetLastError());
  return DPB_OK;
}


// ------------------------------------------------------------------ the same JVP with every contraction on tcgen05
// (gemm_tc.cu: fp16 [hi | lo] operands, three products, fp32 accumulation in TMEM -- ~1e-6 relative, so it stands in for
// the fp32 SGEMM above).  Batch-uniform time only (one table row, the likelihood's case): the affine part of a layer is a
// column bias applied to the primal rows.  The weight operands are built once per handle, at the handle's padded width.
struct JvpOps {
  __half* pool = nullptr;
  Op16 Wpre, W[4], Wpost;
};

static Op16 carve_op16(WsCarver& ws, int64_t rows, int64_t kp) {
  Op16 o;
  o.ptr = ws.take<__half>((size_t)rows * 2 * kp);
  o.ld = 2 * kp;
  o.rows = rows;
  o.lo = (int)kp;
  return o;
}

static size_t jvp_weight_layout(JvpOps* o, int dp, void* base, size_t cap) {
  WsCarver ws(base, cap);
  o->Wpre = carve_op16(ws, H, dp);
  for (int l = 0; l < 4; ++l) o->W[l] = carve_op16(ws, H, H);
  o->Wpost = carve_op16(ws, dp, H);
  return align_up(ws.off, 256);
}

struct JvpWs {
  float *xp, *pre, *hbuf, *tbuf;
  Op16 xp16, a16;
};

static size_t jvp_ws_layout(JvpWs* w, int64_t B2, int dp, void* base, size_t cap) {
  WsCarver ws(base, cap);
  w->xp = ws.take<float>((size_t)B2 * dp);
  w->pre = ws.take<float>((size_t)B2 * H);
  w->hbuf = ws.take<float>((size_t)B2 * H);
  w->tbuf = ws.take<float>((size_t)B2 * H);
  w->xp16 = carve_op16(ws, B2, dp);
  w->a16 = carve_op16(ws, B2, H);
  return align_up(ws.off, 256);
}

size_t score_jvp_tc_ws_bytes(int64_t B, int dp) {
  JvpWs w;
  return jvp_ws_layout(&w, 2 * B, dp, nullptr, ~(size_t)0) + 1024;
}

void score_jvp_tc_release(dpb_score* h) {
  JvpOps* o = static_cast<JvpOps*>(h->jvp_ops);
  if (!o) return;
  if (o->pool) cudaFree(o->pool);
  delete o;
  h->jvp_ops = nullptr;
}

int score_jvp_tc_raw(dpb_score* h, const float* x, const float* v, const float* table, float* raw, int64_t B, void* ws,
                     size_t ws_bytes, cudaStream_t st) {
  if (B <= 0) return DPB_OK;
  int rc = DPB_OK;
  const int dp = h->pose_dp;
  JvpOps* o = static_cast<JvpOps*>(h->jvp_ops);
  if (!o) {
    if ((rc = gemm_tc_init()) != DPB_OK) return rc;
    o = new JvpOps();
    const size_t bytes = jvp_weight_layout(o, dp, nullptr, ~(size_t)0);
    if (cudaMalloc((void**)&o->pool, bytes) != cudaSuccess) { delete o; return fail(DPB_ENOMEM, "score jvp: weight operands"); }
    jvp_weight_layout(o, dp, o->pool, bytes);
    h->jvp_ops = o;
    if ((rc = split16(h->pre_w, H, dp, dp, &o->Wpre, nullptr, st)) != DPB_OK) return rc;
    for (int l = 0; l < 4; ++l)
      if ((rc = split16(h->blk_w[l], H, H, H, &o->W[l], nullptr, st)) != DPB_OK) return rc;
    if ((rc = split16(h->post_w, dp, H, H, &o->Wpost, nullptr, st)) != DPB_OK) return rc;
  }
  const int64_t B2 = 2 * B;
  JvpWs w;
  if (ws == nullptr || jvp_ws_layout(&w, B2, dp, ws, ws_bytes) > ws_bytes) return fail(DPB_ENOMEM, "score jvp: workspace too small");
  const int M = (int)B2, Bi = (int)B;
  launch_pad_x(x, w.xp, B, dp, st);
  launch_pad_x(v, w.xp + (size_t)B * dp, B, dp, st);
#define JTRY(expr) do { rc = (expr); if (rc != DPB_OK) return rc; } while (0)
  JTRY(split16(w.xp, M, dp, dp, &w.xp16, nullptr, st));
  JTRY(gemm_tc(w.xp16, o->Wpre, M, H, dp, w.pre, H, table, nullptr, nullptr, 0, st, Bi));
  gn_silu_jvp_kernel<<<(unsigned)B, 256, 0, st>>>(w.pre, h->gn_w[0], h->gn_b[0], nullptr, w.hbuf, B);
  for (int blk = 0; blk < 2; ++blk) {
    const int l1 = 1 + 2 * blk, l2 = 2 + 2 * blk;
    JTRY(split16(w.hbuf, M, H, H, &w.a16, nullptr, st));
    JTRY(gemm_tc(w.a16, o->W[l1 - 1], M, H, H, w.pre, H, table + (size_t)l1 * H, nullptr, nullptr, 0, st, Bi));
    gn_silu_jvp_kernel<<<(unsigned)B, 256, 0, st>>>(w.pre, h->gn_w[l1], h->gn_b[l1], nullptr, w.tbuf, B);
    JTRY(split16(w.tbuf, M, H, H, &w.a16, nullptr, st));
    JTRY(gemm_tc(w.a16, o->W[l2 - 1], M, H, H, w.pre, H, table + (size_t)l2 * H, nullptr, nullptr, 0, st, Bi));
    gn_silu_jvp_kernel<<<(unsigned)B, 256, 0, st>>>(w.pre, h->gn_w[l2], h->gn_b[l2], w.hbuf, w.hbuf, B);
  }
  JTRY(split16(w.hbuf, M, H, H, &w.a16, nullptr, st));
  JTRY(gemm_tc(w.a16, o->Wpost, M, dp, H, raw, dp, h->post_b, nullptr, nullptr, 0, st, Bi));
#undef JTRY
  DPB_CUDA_CHECK(cudaGetLastError());
  return DPB_OK;
}

}  // namespace dpb
