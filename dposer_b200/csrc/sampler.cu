// Elementwise pieces of the sampler / prior loss for the fp32 engine, Langevin corrector
// kernels, Philox fill.  The tcgen05 engine fuses the same update into its last-layer
// epilogue (score_tc.cu) using the identical formulas and the identical Philox addressing.
//
// Reference: EulerMaruyamaPredictor.update_fn sampling.py:182-188, imputation :413-422,
// LangevinCorrector.update_fn :282-302, prior loss run/completion.py:131-149.
#include "score.h"

namespace dpb {

// Every kernel here is templated on the padded pose width PDP (64 for the 63-D network, 128 for the 126-D one);
// PD = pose_dim_of(PDP) is the unpadded width and PQ = PDP / 4 the column quads of a row.
#define DPB_POSE_WIDTH_CONSTS \
  constexpr int PD = pose_dim_of(PDP); constexpr int PQ = PDP / 4; constexpr int PQ_LOG2 = PQ == 32 ? 5 : 4; \
  (void)PQ; (void)PQ_LOG2;

// one thread per (row, quad of 4 columns): PQ quads per row
template <int PDP>
__global__ void em_update_kernel(float* __restrict__ x_io, const float* __restrict__ raw,
                                 const float* __restrict__ coef, const float* __restrict__ obs,
                                 const float* __restrict__ mask, const float* __restrict__ noise, int noise_k,
                                 uint64_t seed, uint32_t step, float* __restrict__ traj,
                                 float* __restrict__ x_mean_out, int64_t B, int impute) {
  DPB_POSE_WIDTH_CONSTS
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= B * PQ) return;
  const int64_t row = i >> PQ_LOG2;
  const int quad = (int)(i & (PQ - 1));
  const float a = coef[0], b = coef[1], c = coef[2], alpha = coef[3], sd = coef[4];
  float zp[4], zi[4] = {0, 0, 0, 0};
  const size_t plane = (size_t)B * PD;
  if (noise) {
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      int col = quad * 4 + j;
      size_t e = (size_t)row * PD + col;
      bool ok = col < PD;
      if (noise_k == 3) {  // planes: [draw after corrector | predictor draw | draw after predictor]
        zp[j] = ok ? noise[plane + e] : 0.f;
        zi[j] = ok ? noise[2 * plane + e] : 0.f;
      } else {
        zp[j] = ok ? noise[e] : 0.f;
      }
    }
  } else {
    normal4(seed, (uint64_t)row, step, 1, quad, zp, PQ);
    if (impute) normal4(seed, (uint64_t)row, step, 2, quad, zi, PQ);
  }
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    int col = quad * 4 + j;
    if (col >= PD) continue;
    size_t e = (size_t)row * PD + col;
    // x already carries the imputation of the corrector slot (impute_kernel ran before the score eval)
    float x = x_io[e];
    float xm = a * x + b * raw[(size_t)row * PDP + col];
    float xn = xm + c * zp[j];
    if (impute) {
      float m = mask[e];
      xn = xn * (1.0f - m) + (alpha * obs[e] + zi[j] * sd) * m;   // sampling.py:413-422 after the predictor
    }
    x_io[e] = xn;
    if (traj) traj[e] = xn;
    if (x_mean_out) x_mean_out[e] = xm;
  }
}

// imputation that precedes the score evaluation of a step (corrector slot, sampling.py:459)
template <int PDP>
__global__ void impute_kernel(float* __restrict__ x_io, const float* __restrict__ coef,
                              const float* __restrict__ obs, const float* __restrict__ mask,
                              const float* __restrict__ noise, uint64_t seed, uint32_t step, int64_t B) {
  DPB_POSE_WIDTH_CONSTS
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= B * PQ) return;
  const int64_t row = i >> PQ_LOG2;
  const int quad = (int)(i & (PQ - 1));
  const float alpha = coef[3], sd = coef[4];
  float z[4];
  if (noise) {
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      int col = quad * 4 + j;
      z[j] = col < PD ? noise[(size_t)row * PD + col] : 0.f;
    }
  } else {
    normal4(seed, (uint64_t)row, step, 0, quad, z, PQ);
  }
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    int col = quad * 4 + j;
    if (col >= PD) continue;
    size_t e = (size_t)row * PD + col;
    float m = mask[e];
    x_io[e] = x_io[e] * (1.0f - m) + (alpha * obs[e] + z[j] * sd) * m;
  }
}

template <int PDP>
__global__ void scale_out_kernel(const float* __restrict__ raw, const float* __restrict__ row_scale, float scale,
                                 float* __restrict__ out, int64_t B) {
  DPB_POSE_WIDTH_CONSTS
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= B * PD) return;
  int64_t row = i / PD;
  int col = (int)(i % PD);
  float s = row_scale ? row_scale[row] : scale;
  out[i] = raw[row * PDP + col] * s;
}

// ------------------------------------------------------------------ Langevin
template <int PDP>
__global__ void __launch_bounds__(256) langevin_norms_kernel(const float* __restrict__ grad,
                                                             const float* __restrict__ noise,
                                                             float* __restrict__ sums, int64_t B) {
  DPB_POSE_WIDTH_CONSTS
  // one warp per row
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  int64_t row = (int64_t)blockIdx.x * 8 + warp;
  float g = 0.f, z = 0.f;
  if (row < B) {
    for (int c = lane; c < PD; c += 32) {
      float a = grad[row * PD + c], b = noise[row * PD + c];
      g = fmaf(a, a, g);
      z = fmaf(b, b, z);
    }
  }
  for (int s = 16; s > 0; s >>= 1) {
    g += __shfl_xor_sync(0xffffffffu, g, s);
    z += __shfl_xor_sync(0xffffffffu, z, s);
  }
  __shared__ float sg[8], sz[8];
  if (lane == 0) { sg[warp] = row < B ? sqrtf(g) : 0.f; sz[warp] = row < B ? sqrtf(z) : 0.f; }
  __syncthreads();
  if (threadIdx.x == 0) {
    float a = 0.f, b = 0.f;
    for (int w = 0; w < 8; ++w) { a += sg[w]; b += sz[w]; }
    atomicAdd(&sums[0], a);
    atomicAdd(&sums[1], b);
  }
}

template <int PDP>
__global__ void langevin_update_kernel(float* __restrict__ x_io, float* __restrict__ x_mean,
                                       const float* __restrict__ grad, const float* __restrict__ noise,
                                       const float* __restrict__ sums, float snr, float alpha, int64_t B) {
  DPB_POSE_WIDTH_CONSTS
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= B * PD) return;
  // both means share the divisor, so the ratio of sums equals the ratio of means (sampling.py:296-298)
  float r = snr * sums[1] / sums[0];
  float step = r * r * 2.0f * alpha;
  float xm = x_io[i] + step * grad[i];
  if (x_mean) x_mean[i] = xm;
  x_io[i] = xm + sqrtf(step * 2.0f) * noise[i];
}

template <int PDP>
__global__ void normal_fill_kernel(float* __restrict__ out, int64_t B, uint64_t seed, uint32_t step, uint32_t slot) {
  DPB_POSE_WIDTH_CONSTS
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= B * PQ) return;
  const int64_t row = i >> PQ_LOG2;
  const int quad = (int)(i & (PQ - 1));
  float z[4];
  normal4(seed, (uint64_t)row, step, slot, quad, z, PQ);
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    int col = quad * 4 + j;
    if (col < PD) out[(size_t)row * PD + col] = z[j];
  }
}

// ------------------------------------------------------------------ prior loss (fp32 engine)
template <int PDP>
__global__ void perturb_kernel(const float* __restrict__ x0, const float* __restrict__ z, uint64_t seed,
                               uint32_t step, float alpha, float sd, float* __restrict__ xt, int64_t B) {
  DPB_POSE_WIDTH_CONSTS
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= B * PQ) return;
  const int64_t row = i >> PQ_LOG2;
  const int quad = (int)(i & (PQ - 1));
  float zz[4];
  if (z) {
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      int col = quad * 4 + j;
      zz[j] = col < PD ? z[(size_t)row * PD + col] : 0.f;
    }
  } else {
    normal4(seed, (uint64_t)row, step, 3, quad, zz, PQ);
  }
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    int col = quad * 4 + j;
    if (col < PD) xt[(size_t)row * PD + col] = alpha * x0[(size_t)row * PD + col] + sd * zz[j];
  }
}

// one warp per row; loss_out accumulated with one atomic per CTA
template <int PDP>
__global__ void __launch_bounds__(256) prior_loss_kernel(const float* __restrict__ x0, const float* __restrict__ xt,
                                                         const float* __restrict__ raw, float alpha, float sd,
                                                         float inv_sigma_std, float w, float inv_div,
                                                         float* __restrict__ loss_out, float* __restrict__ grad_out,
                                                         float* __restrict__ row_loss, int64_t B) {
  DPB_POSE_WIDTH_CONSTS
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  int64_t row = (int64_t)blockIdx.x * 8 + warp;
  float acc = 0.f;
  if (row < B) {
    for (int c = lane; c < PD; c += 32) {
      size_t e = (size_t)row * PD + c;
      float score = -raw[(size_t)row * PDP + c] * inv_sigma_std;       // utils.py:162
      float x0h = (xt[e] + (sd * sd) * score) / alpha;                  // completion.py:107
      float d = x0[e] - x0h;
      acc = fmaf(w * d, d, acc);
      if (grad_out) grad_out[e] = 2.0f * w * d * inv_div;
    }
  }
  for (int s = 16; s > 0; s >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, s);
  __shared__ float sacc[8];
  if (lane == 0) {
    sacc[warp] = acc;
    if (row_loss && row < B) row_loss[row] = acc;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    float a = 0.f;
    for (int k = 0; k < 8; ++k) a += sacc[k];
    atomicAdd(loss_out, a * inv_div);
  }
}

// ------------------------------------------------------------------ host-side launchers used by api.cu
static inline unsigned blocks_for(int64_t n, int bs) { return (unsigned)((n + bs - 1) / bs); }

// `dp` is the padded pose width of the score handle (64 or 128); it selects the kernel instantiation
#define DPB_BY_WIDTH(dp, call) \
  do { if ((dp) == ::dpb::DP128) { constexpr int W = ::dpb::DP128; call; } else { constexpr int W = ::dpb::DP; call; } } while (0)

int launch_em_update(float* x_io, const float* raw, const float* coef, const float* obs, const float* mask,
                     const float* noise, int noise_k, uint64_t seed, uint32_t step, float* traj, float* x_mean,
                     int64_t B, int impute, int dp, cudaStream_t st) {
  DPB_BY_WIDTH(dp, (em_update_kernel<W><<<blocks_for(B * (W / 4), 256), 256, 0, st>>>(
                       x_io, raw, coef, obs, mask, noise, noise_k, seed, step, traj, x_mean, B, impute)));
  DPB_CUDA_CHECK(cudaGetLastError());
  return DPB_OK;
}

int launch_impute(float* x_io, const float* coef, const float* obs, const float* mask, const float* noise,
                  uint64_t seed, uint32_t step, int64_t B, int dp, cudaStream_t st) {
  DPB_BY_WIDTH(dp, (impute_kernel<W><<<blocks_for(B * (W / 4), 256), 256, 0, st>>>(x_io, coef, obs, mask, noise, seed,
                                                                                   step, B)));
  DPB_CUDA_CHECK(cudaGetLastError());
  return DPB_OK;
}

int launch_scale_out(const float* raw, const float* row_scale, float scale, float* out, int64_t B, int dp,
                     cudaStream_t st) {
  DPB_BY_WIDTH(dp, (scale_out_kernel<W><<<blocks_for(B * pose_dim_of(W), 256), 256, 0, st>>>(raw, row_scale, scale, out,
                                                                                            B)));
  DPB_CUDA_CHECK(cudaGetLastError());
  return DPB_OK;
}

int launch_perturb(const float* x0, const float* z, uint64_t seed, uint32_t step, float alpha, float sd, float* xt,
                   int64_t B, int dp, cudaStream_t st) {
  DPB_BY_WIDTH(dp, (perturb_kernel<W><<<blocks_for(B * (W / 4), 256), 256, 0, st>>>(x0, z, seed, step, alpha, sd, xt,
                                                                                    B)));
  DPB_CUDA_CHECK(cudaGetLastError());
  return DPB_OK;
}

int launch_prior_loss(const float* x0, const float* xt, const float* raw, float alpha, float sd, float inv_sigma_std,
                      float w, float inv_div, float* loss_out, float* grad_out, float* row_loss, int64_t B, int dp,
                      cudaStream_t st) {
  DPB_CUDA_CHECK(cudaMemsetAsync(loss_out, 0, sizeof(float), st));
  DPB_BY_WIDTH(dp, (prior_loss_kernel<W><<<blocks_for(B, 8), 256, 0, st>>>(x0, xt, raw, alpha, sd, inv_sigma_std, w,
                                                                           inv_div, loss_out, grad_out, row_loss, B)));
  DPB_CUDA_CHECK(cudaGetLastError());
  return DPB_OK;
}

static int dp_of_dim(int pose_dim) { return pose_dim == D126 ? DP128 : pose_dim == D ? DP : 0; }

}  // namespace dpb

// ------------------------------------------------------------------ C ABI (stateless helpers)
extern "C" int dpb_langevin_norms_dim(const float* grad, const float* noise, float* sums, int64_t B, int pose_dim,
                                      void* stream) {
  const int dp = dpb::dp_of_dim(pose_dim);
  if (!dp) return dpb::fail(DPB_EUNSUPPORTED, "dpb_langevin_norms_dim: pose_dim must be 63 or 126");
  if (!grad || !noise || !sums || B <= 0) return dpb::fail(DPB_EINVAL, "dpb_langevin_norms: bad argument");
  dpb::PtrDeviceGuard guard(grad);
  DPB_BY_WIDTH(dp, (dpb::langevin_norms_kernel<W><<<dpb::blocks_for(B, 8), 256, 0, (cudaStream_t)stream>>>(grad, noise,
                                                                                                          sums, B)));
  DPB_CUDA_CHECK(cudaGetLastError());
  return DPB_OK;
}

extern "C" int dpb_langevin_norms(const float* grad, const float* noise, float* sums, int64_t B, void* stream) {
  return dpb_langevin_norms_dim(grad, noise, sums, B, DPB_POSE_DIM, stream);
}

extern "C" int dpb_langevin_update_dim(float* x_io, float* x_mean, const float* grad, const float* noise,
                                       const float* sums, float snr, float alpha, int64_t B, int pose_dim,
                                       void* stream) {
  const int dp = dpb::dp_of_dim(pose_dim);
  if (!dp) return dpb::fail(DPB_EUNSUPPORTED, "dpb_langevin_update_dim: pose_dim must be 63 or 126");
  if (!x_io || !grad || !noise || !sums || B <= 0) return dpb::fail(DPB_EINVAL, "dpb_langevin_update: bad argument");
  dpb::PtrDeviceGuard guard(x_io);
  DPB_BY_WIDTH(dp, (dpb::langevin_update_kernel<W><<<dpb::blocks_for(B * pose_dim, 256), 256, 0, (cudaStream_t)stream>>>(
                       x_io, x_mean, grad, noise, sums, snr, alpha, B)));
  DPB_CUDA_CHECK(cudaGetLastError());
  return DPB_OK;
}

extern "C" int dpb_langevin_update(float* x_io, float* x_mean, const float* grad, const float* noise,
                                   const float* sums, float snr, float alpha, int64_t B, void* stream) {
  return dpb_langevin_update_dim(x_io, x_mean, grad, noise, sums, snr, alpha, B, DPB_POSE_DIM, stream);
}

extern "C" int dpb_normal_fill_dim(float* out, int64_t B, uint64_t seed, uint64_t step, int slot, int pose_dim,
                                   void* stream) {
  const int dp = dpb::dp_of_dim(pose_dim);
  if (!dp) return dpb::fail(DPB_EUNSUPPORTED, "dpb_normal_fill_dim: pose_dim must be 63 or 126");
  if (!out || B <= 0) return dpb::fail(DPB_EINVAL, "dpb_normal_fill: bad argument");
  dpb::PtrDeviceGuard guard(out);
  DPB_BY_WIDTH(dp, (dpb::normal_fill_kernel<W><<<dpb::blocks_for(B * (W / 4), 256), 256, 0, (cudaStream_t)stream>>>(
                       out, B, seed, (uint32_t)step, (uint32_t)slot)));
  DPB_CUDA_CHECK(cudaGetLastError());
  return DPB_OK;
}

extern "C" int dpb_normal_fill(float* out, int64_t B, uint64_t seed, uint64_t step, int slot, void* stream) {
  return dpb_normal_fill_dim(out, B, seed, step, slot, DPB_POSE_DIM, stream);
}
