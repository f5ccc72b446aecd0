// Training step of the score network on the device: denoising score-matching loss with per-row random times, its
// gradient with respect to every parameter, Adam with warm-up / gradient clipping, the EMA update, and the forward /
// backward halves + small kernels the auxiliary (DDIM chain + body model) loss chains together.
// Reference: lib/algorithms/advanced/losses.py:31-57 (optimizer, optimize_fn), :61-137 (get_sde_loss_fn), :187-275
// (get_step_fn), lib/algorithms/advanced/model.py:141-196 (forward in train mode, dropout active),
// lib/algorithms/ema.py:10-98.  The reference differentiates with autograd; here the backward pass is written out:
//
//   stage s = 0..4 (pre, b1_dense1, b1_dense2, b2_dense1, b2_dense2):
//     u_s = in_s W_s^T + b_s + temb Wt_s^T + bt_s ;  a_s = dropout(SiLU(GroupNorm_s(u_s))) ;  residual after stages 2, 4
//   res = h W_post^T + b_post ;  e = res_c res + z_c z ;  loss = mean_b row_w_b sum_k e^2
//
// Every contraction (9 forward, 18 backward) is the split-fp16 tcgen05 GEMM of gemm_tc.cu; the per-row time path is
// two GEMMs (shared embedding, then all five 512 -> 1024 projections at once) and its cotangent one GEMM over the
// concatenated stage cotangents.  Column sums (bias / GroupNorm affine gradients) and the gradient norm are reduced
// in a fixed order: the step is deterministic for a given seed.
#include <cmath>
#include <cstring>

#include "score.h"
#include "train.h"

struct dpb_train {
  int device = 0;
  int64_t B = 0, Bp = 0;
  int pose_dim = 63, pose_dp = 64;        // network width D (63 axis-angle, 126 rot6d) and its padded width DP (64, 128)
  char* pool = nullptr;
  size_t pool_bytes = 0;
  float *xp, *z, *temb0, *q, *temb, *tproj, *u[5], *act[5], *res, *gres, *Gall, *gA, *gB, *gtemb, *gq, *t1, *t2;
  float *mean[5], *rstd[5], *loss_rows;
  dpb::Op16 xp16, xpT16, temb0_16, temb0T16, temb16, tembT16, X16[5], XT16[5], G16, GT16, gres16, gresT16, gqT16;
  dpb::Op16 Wpre16, WpreT16, W16[4], WT16[4], Wpost16, WpostT16, Ws16, Wt16, WtT16;
  const uint64_t* seed_dev = nullptr;     // when set, the Philox seed is read from device memory (graph replay)
  cudaStream_t side = nullptr;            // weight-gradient GEMMs run beside the cotangent chain
  cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
};

namespace dpb {
namespace trn {

constexpr int SS_BLOCKS = 512;

// perturbed = mean_c x + std_c z (losses.py:112-115), z from Philox or given; sinusoidal embedding of the label (model.py:37-51).
// Thread t < PDP / 4 owns columns 4t..4t+3 and draws them with Philox counter t: at 126 threads 16..31 add columns 64..127.
template <int PDP>
__global__ void __launch_bounds__(256) prep_kernel(const float* __restrict__ batch, const float* __restrict__ rows,
                                                   const float* __restrict__ z_given, uint64_t seed,
                                                   const uint64_t* __restrict__ seed_dev,
                                                   const float* __restrict__ freqs, float* __restrict__ xp,
                                                   float* __restrict__ z, float* __restrict__ temb0, int64_t B) {
  constexpr int PD = pose_dim_of(PDP);
  if (seed_dev) seed = *seed_dev;
  const int64_t b = blockIdx.x;
  const int t = threadIdx.x;
  const float label = rows[b], mc = rows[B + b], sc = rows[2 * B + b];
  if (t < PDP / 4) {
    float zz[4];
    if (z_given) {
#pragma unroll
      for (int i = 0; i < 4; ++i) zz[i] = (4 * t + i < PD) ? z_given[b * PD + 4 * t + i] : 0.f;
    } else {
      normal4(seed, (uint64_t)b, 0u, 0u, (uint32_t)t, zz);
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int k = 4 * t + i;
      const float zv = k < PD ? zz[i] : 0.f;
      z[b * PDP + k] = zv;
      xp[b * PDP + k] = k < PD ? mc * batch[b * PD + k] + sc * zv : 0.f;
    }
  }
  const float arg = label * freqs[t];
  temb0[b * E + t] = sinf(arg);
  temb0[b * E + E / 2 + t] = cosf(arg);
}

__global__ void silu_fwd_kernel(const float* __restrict__ q, float* __restrict__ out, int64_t n) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) { const float v = q[i]; out[i] = v / (1.0f + expf(-v)); }
}

__global__ void silu_bwd_kernel(const float* __restrict__ q, const float* __restrict__ g, float* __restrict__ out, int64_t n) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) {
    const float v = q[i], s = 1.0f / (1.0f + expf(-v));
    out[i] = g[i] * s * (1.0f + v * (1.0f - s));
  }
}

__device__ __forceinline__ float keep_scale(const uint8_t* mask_given, uint64_t seed, int stage, int64_t b, int c, float p,
                                            int64_t B) {
  if (p <= 0.f) return 1.0f;
  bool keep;
  if (mask_given) {
    keep = mask_given[((size_t)stage * B + b) * H + c] != 0;
  } else {
    uint32_t r[4];
    philox4x32_10((uint32_t)b, (uint32_t)(b >> 32), 0x5EED0000u + (uint32_t)stage, (uint32_t)(c >> 2), (uint32_t)seed,
                  (uint32_t)(seed >> 32), r);
    keep = (float)r[c & 3] * 2.3283064365386963e-10f >= p;       // bernoulli(1 - p)
  }
  return keep ? 1.0f / (1.0f - p) : 0.f;
}

// one warp = one (row, GroupNorm group): a = dropout(SiLU(gamma xhat + beta)), out = (resid +) a
__global__ void __launch_bounds__(256) gn_act_fwd_kernel(const float* __restrict__ u, const float* __restrict__ gamma,
                                                         const float* __restrict__ beta, const float* __restrict__ resid,
                                                         float* __restrict__ out, float* __restrict__ mean,
                                                         float* __restrict__ rstd, const uint8_t* __restrict__ mask_given,
                                                         uint64_t seed, const uint64_t* __restrict__ seed_dev, int stage,
                                                         float p, int64_t B) {
  if (seed_dev) seed = *seed_dev;
  const int64_t w = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (w >= B * 32) return;
  const int64_t b = w >> 5;
  const int c = (int)(w & 31) * GROUP + lane;
  const float x = u[b * H + c];
  float s = x;
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  const float mu = s * (1.0f / GROUP);
  const float d = x - mu;
  float v = d * d;
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  const float rs = rsqrtf(v * (1.0f / GROUP) + GN_EPS);
  const float n = gamma[c] * (d * rs) + beta[c];
  float a = n / (1.0f + expf(-n));
  a *= keep_scale(mask_given, seed, stage, b, c, p, B);
  out[b * H + c] = resid ? resid[b * H + c] + a : a;
  if (lane == 0) { mean[w] = mu; rstd[w] = rs; }
}

// cotangent of the stage input u given the cotangent of its output; t1 = g_n, t2 = g_n xhat (column sums -> d beta, d gamma)
__global__ void __launch_bounds__(256) gn_act_bwd_kernel(const float* __restrict__ gout, const float* __restrict__ u,
                                                         const float* __restrict__ gamma, const float* __restrict__ beta,
                                                         const float* __restrict__ mean, const float* __restrict__ rstd,
                                                         float* __restrict__ gu, int64_t ldg, float* __restrict__ t1,
                                                         float* __restrict__ t2, const uint8_t* __restrict__ mask_given,
                                                         uint64_t seed, const uint64_t* __restrict__ seed_dev, int stage,
                                                         float p, int64_t B) {
  if (seed_dev) seed = *seed_dev;
  const int64_t w = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (w >= B * 32) return;
  const int64_t b = w >> 5;
  const int c = (int)(w & 31) * GROUP + lane;
  const float rs = rstd[w];
  const float xh = (u[b * H + c] - mean[w]) * rs;
  const float n = gamma[c] * xh + beta[c];
  const float sg = 1.0f / (1.0f + expf(-n));
  const float gn = gout[b * H + c] * keep_scale(mask_given, seed, stage, b, c, p, B) * sg * (1.0f + n * (1.0f - sg));
  const float gx = gn * gamma[c];
  float m1 = gx, m2 = gx * xh;
  for (int o = 16; o > 0; o >>= 1) {
    m1 += __shfl_xor_sync(0xffffffffu, m1, o);
    m2 += __shfl_xor_sync(0xffffffffu, m2, o);
  }
  gu[b * ldg + c] = rs * (gx - m1 * (1.0f / GROUP) - xh * m2 * (1.0f / GROUP));
  t1[b * H + c] = gn;
  t2[b * H + c] = gn * xh;
}

// dst[c] = scale * sum_r src[r, c], rows added in a fixed order (32 row lanes, then a fixed tree)
__global__ void __launch_bounds__(1024) colsum_kernel(const float* __restrict__ src, int64_t R, int Cc, int64_t ld,
                                                      float scale, float* __restrict__ dst1, float* __restrict__ dst2,
                                                      int acc) {
  __shared__ float part[32][33];
  const int c = blockIdx.x * 32 + threadIdx.x;
  float s = 0.f;
  if (c < Cc)
    for (int64_t r = threadIdx.y; r < R; r += 32) s += src[r * ld + c];
  part[threadIdx.y][threadIdx.x] = s;
  __syncthreads();
  if (threadIdx.y == 0 && c < Cc) {
    float t = 0.f;
#pragma unroll
    for (int i = 0; i < 32; ++i) t += part[i][threadIdx.x];
    t *= scale;
    dst1[c] = acc ? dst1[c] + t : t;
    if (dst2) dst2[c] = acc ? dst2[c] + t : t;
  }
}

// the three column sums of one stage's backward in one launch (blockIdx.y picks the source): d beta, d gamma, d bias
__global__ void __launch_bounds__(1024) colsum3_kernel(const float* __restrict__ s0, const float* __restrict__ s1,
                                                       const float* __restrict__ s2, int64_t ld2, int64_t R,
                                                       float* __restrict__ d0, float* __restrict__ d1,
                                                       float* __restrict__ d2a, float* __restrict__ d2b, int acc) {
  __shared__ float part[32][33];
  const int which = blockIdx.y;
  const float* src = which == 0 ? s0 : which == 1 ? s1 : s2;
  const int64_t ld = which == 2 ? ld2 : H;
  const int c = blockIdx.x * 32 + threadIdx.x;
  float s = 0.f;
  for (int64_t r = threadIdx.y; r < R; r += 32) s += src[r * ld + c];
  part[threadIdx.y][threadIdx.x] = s;
  __syncthreads();
  if (threadIdx.y == 0) {
    float t = 0.f;
#pragma unroll
    for (int i = 0; i < 32; ++i) t += part[i][threadIdx.x];
    if (which == 0) d0[c] = acc ? d0[c] + t : t;
    else if (which == 1) d1[c] = acc ? d1[c] + t : t;
    else { d2a[c] = acc ? d2a[c] + t : t; d2b[c] = acc ? d2b[c] + t : t; }
  }
}

// e = res_c res + z_c z ; loss_row = row_w sum e^2 ; d loss / d res = 2 row_w res_c e / B   (losses.py:124-131)
template <int PDP>
__global__ void __launch_bounds__(256) loss_kernel(const float* __restrict__ res, const float* __restrict__ z,
                                                   const float* __restrict__ rows, float* __restrict__ gres,
                                                   float* __restrict__ loss_rows, int64_t B) {
  const int64_t b = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (b >= B) return;
  constexpr int PD = pose_dim_of(PDP);
  const float rc = rows[3 * B + b], zc = rows[4 * B + b], w = rows[5 * B + b];
  float acc = 0.f;
#pragma unroll
  for (int h2 = 0; h2 < PDP / 32; ++h2) {
    const int k = lane + 32 * h2;
    float e = 0.f;
    if (k < PD) e = rc * res[b * PDP + k] + zc * z[b * PDP + k];
    acc += e * e;
    gres[b * PDP + k] = k < PD ? 2.0f * w * rc * e / (float)B : 0.f;
  }
  for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  if (lane == 0) loss_rows[b] = w * acc;
}

__global__ void __launch_bounds__(256) sumsq_partial_kernel(const float* __restrict__ x, int64_t n, double* __restrict__ part) {
  __shared__ double sh[256];
  double s = 0.0;
  for (int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x; i < n; i += (int64_t)gridDim.x * 256) {
    const double v = x[i];
    s += v * v;
  }
  sh[threadIdx.x] = s;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if (threadIdx.x < o) sh[threadIdx.x] += sh[threadIdx.x + o];
    __syncthreads();
  }
  if (threadIdx.x == 0) part[blockIdx.x] = sh[0];
}

__global__ void __launch_bounds__(256) sumsq_final_kernel(const double* __restrict__ part, int n, double* __restrict__ out) {
  __shared__ double sh[256];
  double s = 0.0;
  for (int i = threadIdx.x; i < n; i += 256) s += part[i];
  sh[threadIdx.x] = s;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if (threadIdx.x < o) sh[threadIdx.x] += sh[threadIdx.x + o];
    __syncthreads();
  }
  if (threadIdx.x == 0) *out = sh[0];
}

// torch.nn.utils.clip_grad_norm_ (coefficient max_norm / (norm + 1e-6) clamped to 1) folded into torch.optim.Adam's update
__global__ void adam_weights_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m,
                                    float* __restrict__ v, int64_t n, float step_size, float beta1, float beta2,
                                    float inv_sqrt_bc2, float eps, float wd, const double* __restrict__ gnorm_sq,
                                    float grad_clip, const float* __restrict__ hyper_dev) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  if (hyper_dev) { step_size = hyper_dev[0]; inv_sqrt_bc2 = hyper_dev[1]; }
  float coef = 1.0f;
  if (gnorm_sq && grad_clip >= 0.f) coef = fminf(grad_clip / ((float)sqrt(*gnorm_sq) + 1e-6f), 1.0f);
  float gi = g[i] * coef;
  if (wd != 0.f) gi += wd * p[i];
  const float mi = beta1 * m[i] + (1.0f - beta1) * gi;
  const float vi = beta2 * v[i] + (1.0f - beta2) * gi * gi;
  m[i] = mi;
  v[i] = vi;
  p[i] -= step_size * (mi / (sqrtf(vi) * inv_sqrt_bc2 + eps));
}

// s -= (1 - decay) (s - p)   (ema.py:48-50)
__global__ void ema_kernel(float* __restrict__ s, const float* __restrict__ p, int64_t n, float omd,
                           const float* __restrict__ omd_dev) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (omd_dev) omd = *omd_dev;
  if (i < n) s[i] -= omd * (s[i] - p[i]);
}

static Op16 carve16(WsCarver& ws, int64_t rows, int64_t kp) {
  Op16 o;
  o.ptr = ws.take<__half>((size_t)rows * 2 * kp);
  o.ld = 2 * kp;
  o.rows = rows;
  o.lo = (int)kp;
  return o;
}

static size_t layout(dpb_train* h, void* base, size_t cap) {
  WsCarver ws(base, cap);
  const int64_t B = h->B, Bp = h->Bp, DP = h->pose_dp;
  h->xp = ws.take<float>(B * DP); h->z = ws.take<float>(B * DP);
  h->temb0 = ws.take<float>(B * E); h->q = ws.take<float>(B * E); h->temb = ws.take<float>(B * E);
  h->tproj = ws.take<float>(B * NL * H);
  for (int s = 0; s < NL; ++s) {
    h->u[s] = ws.take<float>(B * H); h->act[s] = ws.take<float>(B * H);
    h->mean[s] = ws.take<float>(B * 32); h->rstd[s] = ws.take<float>(B * 32);
  }
  h->res = ws.take<float>(B * DP); h->gres = ws.take<float>(B * DP);
  h->Gall = ws.take<float>(B * NL * H);
  h->gA = ws.take<float>(B * H); h->gB = ws.take<float>(B * H);
  h->gtemb = ws.take<float>(B * E); h->gq = ws.take<float>(B * E);
  h->t1 = ws.take<float>(B * H); h->t2 = ws.take<float>(B * H);
  h->loss_rows = ws.take<float>(B);
  h->xp16 = carve16(ws, B, DP); h->xpT16 = carve16(ws, DP, Bp);
  h->temb0_16 = carve16(ws, B, E); h->temb0T16 = carve16(ws, E, Bp);
  h->temb16 = carve16(ws, B, E); h->tembT16 = carve16(ws, E, Bp);
  for (int s = 0; s < NL; ++s) { h->X16[s] = carve16(ws, B, H); h->XT16[s] = carve16(ws, H, Bp); }
  h->G16 = carve16(ws, B, NL * H); h->GT16 = carve16(ws, NL * H, Bp);
  h->gres16 = carve16(ws, B, DP); h->gresT16 = carve16(ws, DP, Bp);
  h->gqT16 = carve16(ws, E, Bp);
  h->Wpre16 = carve16(ws, H, DP); h->WpreT16 = carve16(ws, DP, H);
  for (int l = 0; l < 4; ++l) { h->W16[l] = carve16(ws, H, H); h->WT16[l] = carve16(ws, H, H); }
  h->Wpost16 = carve16(ws, DP, H); h->WpostT16 = carve16(ws, H, DP);
  h->Ws16 = carve16(ws, E, E);
  h->Wt16 = carve16(ws, NL * H, E); h->WtT16 = carve16(ws, E, NL * H);
  return align_up(ws.off, 256);
}

}  // namespace trn
}  // namespace dpb

using namespace dpb;

extern "C" int dpb_train_create_dim(dpb_train** out, int64_t batch, int pose_dim, int device) {
  if (pose_dim != DPB_POSE_DIM && pose_dim != DPB_POSE_DIM_ROT6D)
    return fail(DPB_EUNSUPPORTED, "dpb_train_create_dim: pose_dim must be 63 (axis-angle) or 126 (rot6d)");
  DPB_REQUIRE(out && batch > 0, "dpb_train_create_dim: bad argument");
  DeviceGuard guard(device);
  int rc = gemm_tc_init();
  if (rc != DPB_OK) return rc;
  dpb_train* h = new dpb_train();
  h->device = device;
  h->B = batch;
  h->pose_dim = pose_dim;
  h->pose_dp = pose_dim == D126 ? DP128 : DP;
  h->Bp = (batch + 63) / 64 * 64;
  h->pool_bytes = trn::layout(h, nullptr, ~(size_t)0);
  cudaError_t e = cudaMalloc((void**)&h->pool, h->pool_bytes);
  if (e != cudaSuccess) { delete h; return fail(DPB_ENOMEM, std::string("dpb_train_create_dim: ") + cudaGetErrorString(e)); }
  cudaMemset(h->pool, 0, h->pool_bytes);                  // operand pads (k >= K, rows >= valid) stay zero for good
  trn::layout(h, h->pool, h->pool_bytes);
  cudaStreamCreateWithFlags(&h->side, cudaStreamNonBlocking);
  cudaEventCreateWithFlags(&h->ev_fork, cudaEventDisableTiming);
  cudaEventCreateWithFlags(&h->ev_join, cudaEventDisableTiming);
  *out = h;
  return DPB_OK;
}

extern "C" int dpb_train_set_seed_pointer(dpb_train* h, const uint64_t* seed_dev) {
  DPB_REQUIRE(h, "dpb_train_set_seed_pointer: bad argument");
  h->seed_dev = seed_dev;
  return DPB_OK;
}

extern "C" int dpb_train_destroy(dpb_train* h) {
  if (!h) return DPB_OK;
  DeviceGuard guard(h->device);
  if (h->pool) cudaFree(h->pool);
  if (h->side) cudaStreamDestroy(h->side);
  if (h->ev_fork) cudaEventDestroy(h->ev_fork);
  if (h->ev_join) cudaEventDestroy(h->ev_join);
  delete h;
  return DPB_OK;
}

namespace dpb {
namespace trn {

// x [B,D] -> xp [B,DP] (pad columns zero); sinusoidal embedding of the per-row label
template <int PDP>
__global__ void __launch_bounds__(256) prep_given_kernel(const float* __restrict__ x, const float* __restrict__ labels,
                                                         const float* __restrict__ freqs, float* __restrict__ xp,
                                                         float* __restrict__ temb0, int64_t B) {
  constexpr int PD = pose_dim_of(PDP);
  const int64_t b = blockIdx.x;
  const int t = threadIdx.x;
  if (t < PDP) xp[b * PDP + t] = t < PD ? x[b * PD + t] : 0.f;
  const float arg = labels[b] * freqs[t];
  temb0[b * E + t] = sinf(arg);
  temb0[b * E + E / 2 + t] = cosf(arg);
}

// [B,D] <-> [B,DP] copies of the network output / its cotangent
__global__ void pad_cols_kernel(const float* __restrict__ src, int ls, float* __restrict__ dst, int ld, int cols, int64_t B) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= B * ld) return;
  const int64_t b = i / ld;
  const int c = (int)(i % ld);
  dst[i] = c < cols ? src[b * ls + c] : 0.f;
}

struct Ptrs {
  const float *Wl[4], *Wt[5], *bl[5], *bt[5], *gam[5], *bet[5];
  explicit Ptrs(const dpb_train_tensors* P) {
    for (int l = 0; l < 4; ++l) Wl[l] = P->blk_w[l];
    Wt[0] = P->pre_t_w; bl[0] = P->pre_b; bt[0] = P->pre_t_b; gam[0] = P->pre_gn_w; bet[0] = P->pre_gn_b;
    for (int l = 0; l < 4; ++l) {
      Wt[l + 1] = P->blk_t_w[l]; bl[l + 1] = P->blk_b[l]; bt[l + 1] = P->blk_t_b[l];
      gam[l + 1] = P->blk_gn_w[l]; bet[l + 1] = P->blk_gn_b[l];
    }
  }
};

#define TRY(expr) do { rc = (expr); if (rc != DPB_OK) return rc; } while (0)

// fp16 [hi | lo] operands of the current weights (they change every step); `back`: the transposed copies too
static int weight_operands(dpb_train* h, const dpb_train_tensors* P, bool back, cudaStream_t st) {
  int rc = DPB_OK;
  const Ptrs w(P);
  const int D = h->pose_dim;
  TRY(split16(P->pre_w, H, D, D, &h->Wpre16, back ? &h->WpreT16 : nullptr, st));
  for (int l = 0; l < 4; ++l) TRY(split16(w.Wl[l], H, H, H, &h->W16[l], back ? &h->WT16[l] : nullptr, st));
  TRY(split16(P->post_w, D, H, H, &h->Wpost16, back ? &h->WpostT16 : nullptr, st));
  TRY(split16(P->temb_w, E, E, E, &h->Ws16, nullptr, st));
  for (int s = 0; s < NL; ++s) {
    const Op16 r = h->Wt16.block(s * H, 0), c = h->WtT16.block(0, s * H);
    TRY(split16(w.Wt[s], H, E, E, &r, back ? &c : nullptr, st));
  }
  return DPB_OK;
}

// h->xp, h->temb0 -> h->res (activations and, with `back`, the transposed operands stay in the handle)
static int forward(dpb_train* h, const dpb_train_tensors* P, const uint8_t* mask_given, float drop_p, uint64_t seed,
                   bool back, cudaStream_t st) {
  int rc = DPB_OK;
  const Ptrs w(P);
  const int64_t B = h->B;
  const int Bi = (int)B, D = h->pose_dim, DP = h->pose_dp;
  const unsigned gw = (unsigned)((B * 32 + 7) / 8);
  TRY(split16(h->xp, Bi, DP, DP, &h->xp16, back ? &h->xpT16 : nullptr, st));
  TRY(split16(h->temb0, Bi, E, E, &h->temb0_16, back ? &h->temb0T16 : nullptr, st));
  TRY(gemm_tc(h->temb0_16, h->Ws16, Bi, E, E, h->q, E, P->temb_b, nullptr, nullptr, 0, st));
  silu_fwd_kernel<<<(unsigned)((B * E + 255) / 256), 256, 0, st>>>(h->q, h->temb, B * E);
  TRY(split16(h->temb, Bi, E, E, &h->temb16, back ? &h->tembT16 : nullptr, st));
  TRY(gemm_tc(h->temb16, h->Wt16, Bi, NL * H, E, h->tproj, NL * H, nullptr, nullptr, nullptr, 0, st));
  for (int s = 0; s < NL; ++s) {
    const Op16& in = s == 0 ? h->xp16 : h->X16[s - 1];
    const Op16& wop = s == 0 ? h->Wpre16 : h->W16[s - 1];
    TRY(gemm_tc(in, wop, Bi, H, s == 0 ? DP : H, h->u[s], H, w.bl[s], w.bt[s], h->tproj + (size_t)s * H, NL * H, st));
    const float* resid = (s == 2) ? h->act[0] : (s == 4) ? h->act[2] : nullptr;
    gn_act_fwd_kernel<<<gw, 256, 0, st>>>(h->u[s], w.gam[s], w.bet[s], resid, h->act[s], h->mean[s], h->rstd[s], mask_given,
                                          seed, h->seed_dev, s, drop_p, B);
    TRY(split16(h->act[s], Bi, H, H, &h->X16[s], back ? &h->XT16[s] : nullptr, st));
  }
  TRY(gemm_tc(h->X16[4], h->Wpost16, Bi, D, H, h->res, DP, P->post_b, nullptr, nullptr, 0, st));
  return DPB_OK;
}

// h->gres (cotangent of res) -> every parameter gradient (overwritten, or added to with `acc`) and, if asked, the
// cotangent of the network input g_x [B,D]
static int backward(dpb_train* h, const dpb_train_tensors* P, const dpb_train_tensors* G, const uint8_t* mask_given,
                    float drop_p, uint64_t seed, bool acc, float* g_x, cudaStream_t st) {
  int rc = DPB_OK;
  const Ptrs w(P);
  const int64_t B = h->B;
  const int Bi = (int)B, D = h->pose_dim, DP = h->pose_dp;
  const unsigned gw = (unsigned)((B * 32 + 7) / 8);
  float* gWl[4] = {(float*)G->blk_w[0], (float*)G->blk_w[1], (float*)G->blk_w[2], (float*)G->blk_w[3]};
  float* gWt[5] = {(float*)G->pre_t_w, (float*)G->blk_t_w[0], (float*)G->blk_t_w[1], (float*)G->blk_t_w[2], (float*)G->blk_t_w[3]};
  float* gbl[5] = {(float*)G->pre_b, (float*)G->blk_b[0], (float*)G->blk_b[1], (float*)G->blk_b[2], (float*)G->blk_b[3]};
  float* gbt[5] = {(float*)G->pre_t_b, (float*)G->blk_t_b[0], (float*)G->blk_t_b[1], (float*)G->blk_t_b[2], (float*)G->blk_t_b[3]};
  float* ggam[5] = {(float*)G->pre_gn_w, (float*)G->blk_gn_w[0], (float*)G->blk_gn_w[1], (float*)G->blk_gn_w[2], (float*)G->blk_gn_w[3]};
  float* gbet[5] = {(float*)G->pre_gn_b, (float*)G->blk_gn_b[0], (float*)G->blk_gn_b[1], (float*)G->blk_gn_b[2], (float*)G->blk_gn_b[3]};
  const dim3 cs(32, 32);
  const int ia = acc ? 1 : 0;
  auto addc = [&](float* c) -> const float* { return acc ? c : nullptr; };      // C += ... through the GEMM's added matrix
  TRY(split16(h->gres, Bi, DP, DP, &h->gres16, &h->gresT16, st));
  // weight-gradient GEMMs leave the critical path (the cotangent chain): they run on a side stream, forked after the
  // operand they read is written and joined at the end (works the same under stream capture)
  cudaStream_t sd = h->side ? h->side : st;
  auto fork = [&]() { if (sd != st) { cudaEventRecord(h->ev_fork, st); cudaStreamWaitEvent(sd, h->ev_fork, 0); } };
  fork();
  TRY(gemm_tc(h->gresT16, h->XT16[4], D, H, Bi, (float*)G->post_w, H, nullptr, nullptr, addc((float*)G->post_w), H, sd));   // dW_post
  colsum_kernel<<<DP / 32, cs, 0, st>>>(h->gres, B, D, DP, 1.0f, (float*)G->post_b, nullptr, ia);
  TRY(gemm_tc(h->gres16, h->WpostT16, Bi, H, DP, h->gA, H, nullptr, nullptr, nullptr, 0, st));                   // d h''
  // cotangent buffers: gA carries d h'' -> d h' -> d h (outputs of the even stages), gB the odd stages' outputs
  for (int s = NL - 1; s >= 0; --s) {
    float* gu = h->Gall + (size_t)s * H;
    const float* gout = (s & 1) ? h->gB : h->gA;
    gn_act_bwd_kernel<<<gw, 256, 0, st>>>(gout, h->u[s], w.gam[s], w.bet[s], h->mean[s], h->rstd[s], gu, NL * H, h->t1, h->t2,
                                          mask_given, seed, h->seed_dev, s, drop_p, B);
    colsum3_kernel<<<dim3(H / 32, 3), cs, 0, st>>>(h->t1, h->t2, gu, NL * H, B, gbet[s], ggam[s], gbl[s], gbt[s], ia);
    const Op16 grow = h->G16.block(0, s * H), gcol = h->GT16.block(s * H, 0);
    TRY(split16(gu, Bi, H, NL * H, &grow, &gcol, st));
    fork();
    if (s == 0) {
      TRY(gemm_tc(gcol, h->xpT16, H, D, Bi, (float*)G->pre_w, D, nullptr, nullptr, addc((float*)G->pre_w), D, sd));   // dW_pre
      if (g_x) TRY(gemm_tc(grow, h->WpreT16, Bi, D, H, g_x, D, nullptr, nullptr, nullptr, 0, st));                    // d x
    } else {
      TRY(gemm_tc(gcol, h->XT16[s - 1], H, H, Bi, gWl[s - 1], H, nullptr, nullptr, addc(gWl[s - 1]), H, sd));         // dW_s
      if (s & 1)     // input of stage 3 / 1 is h' / h, which also feeds the residual: d h' = g_u3 W_3 + d h''  (in place)
        TRY(gemm_tc(grow, h->WT16[s - 1], Bi, H, H, h->gA, H, nullptr, nullptr, h->gA, H, st));
      else           // input of stage 4 / 2 is a_3 / a_1
        TRY(gemm_tc(grow, h->WT16[s - 1], Bi, H, H, h->gB, H, nullptr, nullptr, nullptr, 0, st));
    }
    TRY(gemm_tc(gcol, h->tembT16, H, E, Bi, gWt[s], E, nullptr, nullptr, addc(gWt[s]), E, sd));                       // dWt_s
  }
  // time path: d temb = sum_s g_u_s Wt_s (one GEMM over the concatenated cotangents), through SiLU, into the shared layer
  TRY(gemm_tc(h->G16, h->WtT16, Bi, E, NL * H, h->gtemb, E, nullptr, nullptr, nullptr, 0, st));
  silu_bwd_kernel<<<(unsigned)((B * E + 255) / 256), 256, 0, st>>>(h->q, h->gtemb, h->gq, B * E);
  TRY(split16(h->gq, Bi, E, E, nullptr, &h->gqT16, st));
  TRY(gemm_tc(h->gqT16, h->temb0T16, E, E, Bi, (float*)G->temb_w, E, nullptr, nullptr, addc((float*)G->temb_w), E, st));  // dW_s
  colsum_kernel<<<E / 32, cs, 0, st>>>(h->gq, B, E, E, 1.0f, (float*)G->temb_b, nullptr, ia);
  if (sd != st) { cudaEventRecord(h->ev_join, sd); cudaStreamWaitEvent(st, h->ev_join, 0); }
  return DPB_OK;
}
#undef TRY

}  // namespace trn
}  // namespace dpb

extern "C" int dpb_train_loss_grad(dpb_train* h, const dpb_train_tensors* P, const dpb_train_tensors* G, const float* batch,
                                   const float* rows, const float* z_given, const uint8_t* mask_given, float drop_p,
                                   uint64_t seed, float* loss, float* loss_rows, void* stream) {
  DPB_REQUIRE(h && P && batch && rows && loss, "dpb_train_loss_grad: bad argument");
  DPB_REQUIRE(drop_p >= 0.f && drop_p < 1.f, "dpb_train_loss_grad: dropout probability must be in [0, 1)");
  DeviceGuard guard(h->device);
  cudaStream_t st = (cudaStream_t)stream;
  const int64_t B = h->B;
  int rc = trn::weight_operands(h, P, G != nullptr, st);
  if (rc != DPB_OK) return rc;
  const bool wide = h->pose_dp == DP128;
  if (wide) trn::prep_kernel<DP128><<<(unsigned)B, 256, 0, st>>>(batch, rows, z_given, seed, h->seed_dev, P->emb_freqs, h->xp, h->z, h->temb0, B);
  else trn::prep_kernel<DP><<<(unsigned)B, 256, 0, st>>>(batch, rows, z_given, seed, h->seed_dev, P->emb_freqs, h->xp, h->z, h->temb0, B);
  if ((rc = trn::forward(h, P, mask_given, drop_p, seed, G != nullptr, st)) != DPB_OK) return rc;
  float* lrows = loss_rows ? loss_rows : h->loss_rows;
  const unsigned gl = (unsigned)((B + 7) / 8);
  if (wide) trn::loss_kernel<DP128><<<gl, 256, 0, st>>>(h->res, h->z, rows, h->gres, lrows, B);
  else trn::loss_kernel<DP><<<gl, 256, 0, st>>>(h->res, h->z, rows, h->gres, lrows, B);
  trn::colsum_kernel<<<1, dim3(32, 32), 0, st>>>(lrows, B, 1, 1, 1.0f / (float)B, loss, nullptr, 0);
  DPB_CUDA_CHECK(cudaGetLastError());
  if (!G) return DPB_OK;
  if ((rc = trn::backward(h, P, G, mask_given, drop_p, seed, false, nullptr, st)) != DPB_OK) return rc;
  DPB_CUDA_CHECK(cudaGetLastError());
  return DPB_OK;
}

// The two halves on their own, for losses that chain several network evaluations (the auxiliary loss of losses.py:91-106,
// 244-258: a DDIM chain under the optimiser).  One handle = the activations of ONE evaluation.
extern "C" int dpb_train_forward(dpb_train* h, const dpb_train_tensors* P, const float* x, const float* labels,
                                 const uint8_t* mask_given, float drop_p, uint64_t seed, float* res, void* stream) {
  DPB_REQUIRE(h && P && x && labels && res, "dpb_train_forward: bad argument");
  DPB_REQUIRE(drop_p >= 0.f && drop_p < 1.f, "dpb_train_forward: dropout probability must be in [0, 1)");
  DeviceGuard guard(h->device);
  cudaStream_t st = (cudaStream_t)stream;
  const int64_t B = h->B;
  int rc = trn::weight_operands(h, P, true, st);
  if (rc != DPB_OK) return rc;
  const int D = h->pose_dim, DP = h->pose_dp;
  if (DP == DP128) trn::prep_given_kernel<DP128><<<(unsigned)B, 256, 0, st>>>(x, labels, P->emb_freqs, h->xp, h->temb0, B);
  else trn::prep_given_kernel<dpb::DP><<<(unsigned)B, 256, 0, st>>>(x, labels, P->emb_freqs, h->xp, h->temb0, B);
  if ((rc = trn::forward(h, P, mask_given, drop_p, seed, true, st)) != DPB_OK) return rc;
  trn::pad_cols_kernel<<<(unsigned)((B * D + 255) / 256), 256, 0, st>>>(h->res, DP, res, D, D, B);
  DPB_CUDA_CHECK(cudaGetLastError());
  return DPB_OK;
}

extern "C" int dpb_train_backward(dpb_train* h, const dpb_train_tensors* P, const dpb_train_tensors* G, const float* g_res,
                                  const uint8_t* mask_given, float drop_p, uint64_t seed, int accumulate, float* g_x,
                                  void* stream) {
  DPB_REQUIRE(h && P && G && g_res, "dpb_train_backward: bad argument");
  DeviceGuard guard(h->device);
  cudaStream_t st = (cudaStream_t)stream;
  const int64_t B = h->B;
  const int D = h->pose_dim, DP = h->pose_dp;
  trn::pad_cols_kernel<<<(unsigned)((B * DP + 255) / 256), 256, 0, st>>>(g_res, D, h->gres, DP, D, B);
  int rc = trn::backward(h, P, G, mask_given, drop_p, seed, accumulate != 0, g_x, st);
  if (rc != DPB_OK) return rc;
  DPB_CUDA_CHECK(cudaGetLastError());
  return DPB_OK;
}

namespace dpb {
namespace trn {

// out[b,c] = a[b] x[b,c] + b[b] y[b,c]  (y may be null): the DDIM chain's affine steps and their adjoints
__global__ void rows_axpby_kernel(const float* __restrict__ a, const float* __restrict__ x, const float* __restrict__ bb,
                                  const float* __restrict__ y, float* __restrict__ out, int cols, int64_t B) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= B * cols) return;
  const int64_t b = i / cols;
  float v = a[b] * x[i];
  if (y) v += bb[b] * y[i];
  out[i] = v;
}

// row_loss[b] = w[b] sum_i (p[b,i] - q[b,i])^2 ;  grad_q[b,i] = -2 scale w[b] (p - q)   (weighted MSE of losses.py:253-254)
__global__ void __launch_bounds__(256) wsqdiff_kernel(const float* __restrict__ p, const float* __restrict__ q,
                                                      const float* __restrict__ w, int64_t n, float scale,
                                                      float* __restrict__ row_loss, float* __restrict__ grad_q) {
  __shared__ float sh[256];
  const int64_t b = blockIdx.x;
  const float wb = w[b];
  float s = 0.f;
  for (int64_t i = threadIdx.x; i < n; i += 256) {
    const float d = p[b * n + i] - q[b * n + i];
    s += d * d;
    if (grad_q) grad_q[b * n + i] = -2.0f * scale * wb * d;
  }
  sh[threadIdx.x] = s;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if (threadIdx.x < o) sh[threadIdx.x] += sh[threadIdx.x + o];
    __syncthreads();
  }
  if (threadIdx.x == 0) row_loss[b] = wb * sh[0];
}

}  // namespace trn
}  // namespace dpb

extern "C" int dpb_rows_axpby(const float* a, const float* x, const float* b, const float* y, float* out, int cols,
                              int64_t B, void* stream) {
  DPB_REQUIRE(a && x && out && cols > 0 && B >= 0 && (!y || b), "dpb_rows_axpby: bad argument");
  if (B == 0) return DPB_OK;
  PtrDeviceGuard guard(out);
  trn::rows_axpby_kernel<<<(unsigned)((B * cols + 255) / 256), 256, 0, (cudaStream_t)stream>>>(a, x, b, y, out, cols, B);
  DPB_CUDA_CHECK(cudaGetLastError());
  return DPB_OK;
}

// loss[0] = scale * sum_b w[b] sum_i (p - q)^2 (rows added in a fixed order); grad_q optional; row_scratch DEVICE [B]
extern "C" int dpb_weighted_sqdiff(const float* p, const float* q, const float* w, int64_t B, int64_t n, float scale,
                                   float* loss, float* grad_q, float* row_scratch, void* stream) {
  DPB_REQUIRE(p && q && w && loss && row_scratch && B > 0 && n > 0, "dpb_weighted_sqdiff: bad argument");
  PtrDeviceGuard guard(p);
  cudaStream_t st = (cudaStream_t)stream;
  trn::wsqdiff_kernel<<<(unsigned)B, 256, 0, st>>>(p, q, w, n, scale, row_scratch, grad_q);
  trn::colsum_kernel<<<1, dim3(32, 32), 0, st>>>(row_scratch, B, 1, 1, scale, loss, nullptr, 0);
  DPB_CUDA_CHECK(cudaGetLastError());
  return DPB_OK;
}

// ---- C = A B^T through the same split-fp16 tensor-core GEMM (utility / unit-test entry; operands converted per call)
static size_t gemm_nt_layout(int M, int N, int K, void* base, size_t cap, Op16* a, Op16* b) {
  WsCarver ws(base, cap);
  const int64_t kp = (K + 63) / 64 * 64;
  *a = trn::carve16(ws, M, kp);
  *b = trn::carve16(ws, N, kp);
  return align_up(ws.off, 256);
}

extern "C" size_t dpb_gemm_nt_workspace_bytes(int M, int N, int K) {
  Op16 a, b;
  return gemm_nt_layout(M, N, K, nullptr, ~(size_t)0, &a, &b);
}

extern "C" int dpb_gemm_nt(const float* A, const float* B, const float* bias, float* C, int M, int N, int K, void* ws,
                           size_t ws_bytes, void* stream) {
  DPB_REQUIRE(A && B && C && ws && M > 0 && N > 0 && K > 0, "dpb_gemm_nt: bad argument");
  DPB_REQUIRE(ws_bytes >= dpb_gemm_nt_workspace_bytes(M, N, K), "dpb_gemm_nt: workspace too small");
  PtrDeviceGuard guard(C);
  cudaStream_t st = (cudaStream_t)stream;
  int rc = gemm_tc_init();
  if (rc != DPB_OK) return rc;
  Op16 a, b;
  const size_t used = gemm_nt_layout(M, N, K, ws, ws_bytes, &a, &b);
  DPB_CUDA_CHECK(cudaMemsetAsync(ws, 0, used, st));
  if ((rc = split16(A, M, K, K, &a, nullptr, st)) != DPB_OK) return rc;
  if ((rc = split16(B, N, K, K, &b, nullptr, st)) != DPB_OK) return rc;
  return gemm_tc(a, b, M, N, K, C, N, bias, nullptr, nullptr, 0, st);
}

extern "C" size_t dpb_train_adam_scratch_bytes(void) { return (size_t)(trn::SS_BLOCKS + 1) * sizeof(double); }

// scratch[0] = sum_i g_i^2 (double), partial sums added in a fixed order
extern "C" int dpb_train_grad_norm(const float* g, int64_t n, void* scratch, void* stream) {
  DPB_REQUIRE(g && scratch && n >= 0, "dpb_train_grad_norm: bad argument");
  PtrDeviceGuard guard(g);
  cudaStream_t st = (cudaStream_t)stream;
  double* sc = static_cast<double*>(scratch);
  trn::sumsq_partial_kernel<<<trn::SS_BLOCKS, 256, 0, st>>>(g, n, sc + 1);
  trn::sumsq_final_kernel<<<1, 256, 0, st>>>(sc + 1, trn::SS_BLOCKS, sc);
  DPB_CUDA_CHECK(cudaGetLastError());
  return DPB_OK;
}

extern "C" int dpb_train_adam(float* p, const float* g, float* m, float* v, int64_t n, float lr, float beta1, float beta2,
                              float eps, float weight_decay, int64_t step, float grad_clip, const float* hyper_dev,
                              void* scratch, void* stream) {
  DPB_REQUIRE(p && g && m && v && n >= 0 && step >= 1, "dpb_train_adam: bad argument");
  DPB_REQUIRE(grad_clip < 0.f || scratch, "dpb_train_adam: gradient clipping needs the scratch buffer");
  PtrDeviceGuard guard(p);
  cudaStream_t st = (cudaStream_t)stream;
  if (grad_clip >= 0.f) {
    int rc = dpb_train_grad_norm(g, n, scratch, stream);
    if (rc != DPB_OK) return rc;
  }
  // torch computes the bias corrections in double on the host (torch/optim/adam.py)
  const double bc1 = 1.0 - std::pow((double)beta1, (double)step), bc2 = 1.0 - std::pow((double)beta2, (double)step);
  const float step_size = (float)((double)lr / bc1), inv_sqrt_bc2 = (float)(1.0 / std::sqrt(bc2));
  trn::adam_weights_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(
      p, g, m, v, n, step_size, beta1, beta2, inv_sqrt_bc2, eps, weight_decay,
      grad_clip >= 0.f ? static_cast<const double*>(scratch) : nullptr, grad_clip, hyper_dev);
  DPB_CUDA_CHECK(cudaGetLastError());
  return DPB_OK;
}

extern "C" int dpb_ema_update(float* shadow, const float* p, int64_t n, float one_minus_decay, const float* omd_dev,
                              void* stream) {
  DPB_REQUIRE(shadow && p && n >= 0, "dpb_ema_update: bad argument");
  if (n == 0) return DPB_OK;
  PtrDeviceGuard guard(shadow);
  trn::ema_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(shadow, p, n, one_minus_decay, omd_dev);
  DPB_CUDA_CHECK(cudaGetLastError());
  return DPB_OK;
}
