// Dormand-Prince RK45 on device vectors: the arithmetic of scipy.integrate.RK45 (which the reference drives through
// solve_ivp in lib/algorithms/advanced/likelihood.py:93-101 and sampling.py:520-524) with the state kept on the GPU in
// fp64; the host keeps only the step-size controller and reads ONE scalar (the error norm) per attempted step.
//   k      DEVICE fp32 [7, n]   stage derivatives (the network produces fp32; scipy widens the same values to fp64)
//   stage  y + h * sum_j a[s][j] k_j  (s = 1..5), or the 5th-order solution y + h * sum_j b_j k_j (s = 6)
//   error  sum_i ( h * sum_j e_j k_j[i] / (atol + rtol max(|y_i|, |y_new_i|)) )^2, added in a fixed order
#include "common.cuh"

namespace dpb {
namespace rk {

__constant__ double A[6][5] = {
    {0, 0, 0, 0, 0},
    {1.0 / 5, 0, 0, 0, 0},
    {3.0 / 40, 9.0 / 40, 0, 0, 0},
    {44.0 / 45, -56.0 / 15, 32.0 / 9, 0, 0},
    {19372.0 / 6561, -25360.0 / 2187, 64448.0 / 6561, -212.0 / 729, 0},
    {9017.0 / 3168, -355.0 / 33, 46732.0 / 5247, 49.0 / 176, -5103.0 / 18656}};
__constant__ double Bc[6] = {35.0 / 384, 0, 500.0 / 1113, 125.0 / 192, -2187.0 / 6784, 11.0 / 84};
__constant__ double Ec[7] = {-71.0 / 57600, 0, 71.0 / 16695, -71.0 / 1920, 17253.0 / 339200, -22.0 / 525, 1.0 / 40};
constexpr int PART = 512;

__global__ void stage_kernel(const double* __restrict__ y, const float* __restrict__ k, int64_t n, double h, int stage,
                             double* __restrict__ y_out, float* __restrict__ x_out, int64_t nx) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  double acc = 0.0;
  if (stage <= 5) {
    for (int j = 0; j < stage; ++j) acc += A[stage][j] * (double)k[(size_t)j * n + i];   // K[:s].T @ a[:s], in order
  } else {
    for (int j = 0; j < 6; ++j) acc += Bc[j] * (double)k[(size_t)j * n + i];
  }
  const double v = y[i] + acc * h;
  if (y_out) y_out[i] = v;
  if (x_out && i < nx) x_out[i] = (float)v;
}

__global__ void __launch_bounds__(256) error_partial_kernel(const double* __restrict__ y, const double* __restrict__ y_new,
                                                            const float* __restrict__ k, int64_t n, double h, double rtol,
                                                            double atol, double* __restrict__ part) {
  __shared__ double sh[256];
  double s = 0.0;
  for (int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x; i < n; i += (int64_t)gridDim.x * 256) {
    double e = 0.0;
    for (int j = 0; j < 7; ++j) e += Ec[j] * (double)k[(size_t)j * n + i];
    const double scale = atol + fmax(fabs(y[i]), fabs(y_new[i])) * rtol;
    const double r = e * h / scale;
    s += r * r;
  }
  sh[threadIdx.x] = s;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if (threadIdx.x < o) sh[threadIdx.x] += sh[threadIdx.x + o];
    __syncthreads();
  }
  if (threadIdx.x == 0) part[blockIdx.x] = sh[0];
}

__global__ void __launch_bounds__(256) error_final_kernel(const double* __restrict__ part, double* __restrict__ out) {
  __shared__ double sh[256];
  double s = 0.0;
  for (int i = threadIdx.x; i < PART; i += 256) s += part[i];
  sh[threadIdx.x] = s;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if (threadIdx.x < o) sh[threadIdx.x] += sh[threadIdx.x + o];
    __syncthreads();
  }
  if (threadIdx.x == 0) *out = sh[0];
}

// right-hand side of the probability-flow ODE from the network outputs (likelihood.py:58-66 / sampling.py:505-509):
// k[b*PD + c] = fx x - 0.5 g2 score ;  k[B*PD + b] = fx sum_c eps^2 - 0.5 g2 sum_c jv eps   (jv / eps null: drift only),
// PD = the pose width (63 axis-angle, 126 rot6d)
template <int PD>
__global__ void __launch_bounds__(256) pf_rhs_kernel(const float* __restrict__ x, const float* __restrict__ score,
                                                     const float* __restrict__ jv, const float* __restrict__ eps, float fx,
                                                     float g2, float* __restrict__ kout, int64_t B) {
  const int64_t b = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (b >= B) return;
  float d1 = 0.f, d2 = 0.f;
  for (int c = lane; c < PD; c += 32) {
    const size_t i = (size_t)b * PD + c;
    kout[i] = fx * x[i] - 0.5f * g2 * score[i];
    if (jv) { const float e = eps[i]; d1 += e * e; d2 += jv[i] * e; }
  }
  if (!jv) return;
  for (int o = 16; o > 0; o >>= 1) {
    d1 += __shfl_xor_sync(0xffffffffu, d1, o);
    d2 += __shfl_xor_sync(0xffffffffu, d2, o);
  }
  if (lane == 0) kout[(size_t)B * PD + b] = fx * d1 - 0.5f * g2 * d2;
}

}  // namespace rk
}  // namespace dpb

using namespace dpb;

extern "C" size_t dpb_rk45_scratch_bytes(void) { return (size_t)(rk::PART + 1) * sizeof(double); }

extern "C" int dpb_rk45_stage(const double* y, const float* k, int64_t n, double h, int stage, double* y_out, float* x_out,
                              int64_t nx, void* stream) {
  DPB_REQUIRE(y && k && n > 0 && stage >= 1 && stage <= 6 && (y_out || x_out), "dpb_rk45_stage: bad argument");
  PtrDeviceGuard guard(y);
  rk::stage_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(y, k, n, h, stage, y_out, x_out, nx);
  DPB_CUDA_CHECK(cudaGetLastError());
  return DPB_OK;
}

extern "C" int dpb_rk45_error(const double* y, const double* y_new, const float* k, int64_t n, double h, double rtol,
                              double atol, void* scratch, void* stream) {
  DPB_REQUIRE(y && y_new && k && scratch && n > 0, "dpb_rk45_error: bad argument");
  PtrDeviceGuard guard(y);
  cudaStream_t st = (cudaStream_t)stream;
  double* sc = static_cast<double*>(scratch);
  rk::error_partial_kernel<<<rk::PART, 256, 0, st>>>(y, y_new, k, n, h, rtol, atol, sc + 1);
  rk::error_final_kernel<<<1, 256, 0, st>>>(sc + 1, sc);
  DPB_CUDA_CHECK(cudaGetLastError());
  return DPB_OK;
}

extern "C" int dpb_pf_ode_rhs_dim(const float* x, const float* score, const float* jv, const float* eps, float fx, float g2,
                                  float* k_out, int64_t B, int pose_dim, void* stream) {
  if (pose_dim != DPB_POSE_DIM && pose_dim != DPB_POSE_DIM_ROT6D)
    return fail(DPB_EUNSUPPORTED, "dpb_pf_ode_rhs_dim: pose_dim must be 63 (axis-angle) or 126 (rot6d)");
  DPB_REQUIRE(x && score && k_out && B > 0 && (!jv || eps), "dpb_pf_ode_rhs_dim: bad argument");
  PtrDeviceGuard guard(x);
  const unsigned grid = (unsigned)((B + 7) / 8);
  cudaStream_t st = (cudaStream_t)stream;
  if (pose_dim == D126) rk::pf_rhs_kernel<D126><<<grid, 256, 0, st>>>(x, score, jv, eps, fx, g2, k_out, B);
  else rk::pf_rhs_kernel<D><<<grid, 256, 0, st>>>(x, score, jv, eps, fx, g2, k_out, B);
  DPB_CUDA_CHECK(cudaGetLastError());
  return DPB_OK;
}
