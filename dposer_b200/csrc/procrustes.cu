// Similarity (Procrustes) alignment of batched point sets and the aligned error, PA-MPJPE / PA-MPVPE
// (compute_similarity_transform / reconstruction_error of the reference's lib/utils/transforms.py).  The definition
// is in dposer_b200/metric.py's docstring.  Per row, in fp64:
//   pass 1  the moments of the selected points, shifted by the first selected point (so that a large translation
//           does not cancel): sums of a = S1 - o1, b = S2 - o2, a.a and a b^T;
//   solve   K = X1^T X2 and var1 from the moments; the proper rotation maximising trace(R K) is the top eigenvector
//           of Horn's symmetric 4x4 quaternion matrix of K (cyclic Jacobi, at most PA_SWEEPS sweeps), and
//           trace(R K) / var1 the scale;
//   pass 2  err = mean over the selected points of ||s R x1 + t - x2||, and the aligned points when asked for.
// Two layouts, picked from n_points by the host:
//   warp  (n_points <= PA_WARP_MAX_POINTS): a warp owns 32 consecutive rows.  For each row its lanes stride over
//         the points and reduce by a butterfly; the 32 solves then run one per lane; pass 2 again row by row.
//   CTA   (larger n_points): one CTA per row, two CTAs per SM; pass 2 walks the row backwards so that it starts with
//         the points pass 1 read last, which are the likeliest to still be in L2.
// Every reduction has a fixed order and there are no atomics, so the output is bit-identical across runs; nothing is
// allocated and nothing synchronises with the host.
#include <math.h>

#include "common.cuh"

namespace dpb {
namespace pa {

constexpr int NM = 16;                  // moments: sum a (3), sum b (3), sum a.a (1), sum a b^T (9)
constexpr int NS = 12;                  // solution: A = s R (9, row-major), t (3)
constexpr int PA_SWEEPS = 12;
constexpr int PA_WARP_MAX_POINTS = 512;
constexpr int WARP_THREADS = 256;       // 8 warps, 256 rows per CTA
constexpr int WARP_ROWS = WARP_THREADS;
constexpr int CTA_THREADS = 512;

__device__ __forceinline__ void load3(const float* p, double& x, double& y, double& z) {
  x = (double)__ldg(p);
  y = (double)__ldg(p + 1);
  z = (double)__ldg(p + 2);
}

// pass 1 of one point: m += moments of (p1 - o, p2 - o2)
__device__ __forceinline__ void accumulate(double m[NM], const float* p1, const float* p2, const double o[6]) {
  double a0, a1, a2, b0, b1, b2;
  load3(p1, a0, a1, a2);
  load3(p2, b0, b1, b2);
  a0 -= o[0]; a1 -= o[1]; a2 -= o[2];
  b0 -= o[3]; b1 -= o[4]; b2 -= o[5];
  m[0] += a0; m[1] += a1; m[2] += a2;
  m[3] += b0; m[4] += b1; m[5] += b2;
  m[6] = fma(a0, a0, fma(a1, a1, fma(a2, a2, m[6])));
  m[7] = fma(a0, b0, m[7]);  m[8] = fma(a0, b1, m[8]);  m[9] = fma(a0, b2, m[9]);
  m[10] = fma(a1, b0, m[10]); m[11] = fma(a1, b1, m[11]); m[12] = fma(a1, b2, m[12]);
  m[13] = fma(a2, b0, m[13]); m[14] = fma(a2, b1, m[14]); m[15] = fma(a2, b2, m[15]);
}

// y = A x1 + t, in fp64; returns ||y - x2||
__device__ __forceinline__ double transform(const double* sol, const float* p1, const float* p2, float* out) {
  double x0, x1, x2, z0, z1, z2;
  load3(p1, x0, x1, x2);
  load3(p2, z0, z1, z2);
  const double y0 = fma(sol[0], x0, fma(sol[1], x1, fma(sol[2], x2, sol[9])));
  const double y1 = fma(sol[3], x0, fma(sol[4], x1, fma(sol[5], x2, sol[10])));
  const double y2 = fma(sol[6], x0, fma(sol[7], x1, fma(sol[8], x2, sol[11])));
  if (out) {
    out[0] = (float)y0;
    out[1] = (float)y1;
    out[2] = (float)y2;
  }
  const double d0 = y0 - z0, d1 = y1 - z1, d2 = y2 - z2;
  return sqrt(fma(d0, d0, fma(d1, d1, d2 * d2)));
}

// One Jacobi rotation of the symmetric 4x4 a, annihilating a[p][q]; v accumulates the eigenvectors (columns).
template <int p, int q>
__device__ __forceinline__ void jacobi_rotate(double a[4][4], double v[4][4]) {
  const double apq = a[p][q];
  if (apq == 0.0) return;
  const double theta = (a[q][q] - a[p][p]) / (2.0 * apq);
  const double t = copysign(1.0, theta) / (fabs(theta) + sqrt(fma(theta, theta, 1.0)));
  const double c = rsqrt(fma(t, t, 1.0)), s = t * c;
  a[p][p] -= t * apq;
  a[q][q] += t * apq;
  a[p][q] = a[q][p] = 0.0;
#pragma unroll
  for (int r = 0; r < 4; ++r) {
    if (r != p && r != q) {
      const double arp = a[r][p], arq = a[r][q];
      a[r][p] = a[p][r] = c * arp - s * arq;
      a[r][q] = a[q][r] = s * arp + c * arq;
    }
    const double vrp = v[r][p], vrq = v[r][q];
    v[r][p] = c * vrp - s * vrq;
    v[r][q] = s * vrp + c * vrq;
  }
}

// Moments of n selected points (shift o) -> solution {A = s R, t}, and params {s, R, t} when params is not null;
// NaN everywhere for a non-finite row or var1 == 0.
__device__ void solve(const double m[NM], double n, const double o[6], double sol[NS], float* params) {
  bool ok = true;
#pragma unroll
  for (int i = 0; i < NM; ++i) ok = ok && isfinite(m[i]);
  const double inv_n = 1.0 / n;
  const double ma0 = m[0] * inv_n, ma1 = m[1] * inv_n, ma2 = m[2] * inv_n;   // means of a and b
  const double mb0 = m[3] * inv_n, mb1 = m[4] * inv_n, mb2 = m[5] * inv_n;
  const double var1 = m[6] - (m[0] * ma0 + m[1] * ma1 + m[2] * ma2);
  if (!ok || !(var1 > 0.0)) {
#pragma unroll
    for (int i = 0; i < NS; ++i) sol[i] = __longlong_as_double(0x7ff8000000000000ll);
    if (params)
      for (int i = 0; i < 13; ++i) params[i] = __int_as_float(0x7fc00000);
    return;
  }
  // K[i][j] = sum X1_i X2_j = sum a_i b_j - n ma_i mb_j
  const double ma[3] = {ma0, ma1, ma2}, mb[3] = {mb0, mb1, mb2};
  double K[3][3];
#pragma unroll
  for (int i = 0; i < 3; ++i)
#pragma unroll
    for (int j = 0; j < 3; ++j) K[i][j] = m[7 + 3 * i + j] - n * ma[i] * mb[j];
  // Horn (1987): the top eigenvector of N is the unit quaternion of the best proper rotation X1 -> X2
  double a[4][4], v[4][4];
  a[0][0] = K[0][0] + K[1][1] + K[2][2];
  a[1][1] = K[0][0] - K[1][1] - K[2][2];
  a[2][2] = -K[0][0] + K[1][1] - K[2][2];
  a[3][3] = -K[0][0] - K[1][1] + K[2][2];
  a[0][1] = a[1][0] = K[1][2] - K[2][1];
  a[0][2] = a[2][0] = K[2][0] - K[0][2];
  a[0][3] = a[3][0] = K[0][1] - K[1][0];
  a[1][2] = a[2][1] = K[0][1] + K[1][0];
  a[1][3] = a[3][1] = K[2][0] + K[0][2];
  a[2][3] = a[3][2] = K[1][2] + K[2][1];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) v[i][j] = i == j ? 1.0 : 0.0;
  for (int sweep = 0; sweep < PA_SWEEPS; ++sweep) {
    const double off = a[0][1] * a[0][1] + a[0][2] * a[0][2] + a[0][3] * a[0][3] + a[1][2] * a[1][2] +
                       a[1][3] * a[1][3] + a[2][3] * a[2][3];
    const double diag = a[0][0] * a[0][0] + a[1][1] * a[1][1] + a[2][2] * a[2][2] + a[3][3] * a[3][3];
    if (!(off > 1e-34 * diag)) break;
    jacobi_rotate<0, 1>(a, v);
    jacobi_rotate<0, 2>(a, v);
    jacobi_rotate<0, 3>(a, v);
    jacobi_rotate<1, 2>(a, v);
    jacobi_rotate<1, 3>(a, v);
    jacobi_rotate<2, 3>(a, v);
  }
  // the column of the largest eigenvalue (the first on a tie)
  double w = v[0][0], x = v[1][0], y = v[2][0], z = v[3][0], top = a[0][0];
#pragma unroll
  for (int k = 1; k < 4; ++k)
    if (a[k][k] > top) {
      top = a[k][k];
      w = v[0][k]; x = v[1][k]; y = v[2][k]; z = v[3][k];
    }
  const double inv = 1.0 / (w * w + x * x + y * y + z * z);
  double R[3][3];
  R[0][0] = (w * w + x * x - y * y - z * z) * inv;
  R[0][1] = 2.0 * (x * y - w * z) * inv;
  R[0][2] = 2.0 * (x * z + w * y) * inv;
  R[1][0] = 2.0 * (x * y + w * z) * inv;
  R[1][1] = (w * w - x * x + y * y - z * z) * inv;
  R[1][2] = 2.0 * (y * z - w * x) * inv;
  R[2][0] = 2.0 * (x * z - w * y) * inv;
  R[2][1] = 2.0 * (y * z + w * x) * inv;
  R[2][2] = (w * w - x * x - y * y + z * z) * inv;
  double tr = 0.0;                                   // trace(R K)
#pragma unroll
  for (int i = 0; i < 3; ++i)
#pragma unroll
    for (int j = 0; j < 3; ++j) tr = fma(R[i][j], K[j][i], tr);
  const double s = tr / var1;
  // mu1 = o1 + ma, mu2 = o2 + mb;  t = mu2 - s R mu1
  const double mu1[3] = {o[0] + ma0, o[1] + ma1, o[2] + ma2};
#pragma unroll
  for (int i = 0; i < 3; ++i) {
#pragma unroll
    for (int j = 0; j < 3; ++j) sol[3 * i + j] = s * R[i][j];
    sol[9 + i] = (o[3 + i] + mb[i]) - (sol[3 * i] * mu1[0] + sol[3 * i + 1] * mu1[1] + sol[3 * i + 2] * mu1[2]);
  }
  if (params) {
    params[0] = (float)s;
#pragma unroll
    for (int i = 0; i < 3; ++i) {
#pragma unroll
      for (int j = 0; j < 3; ++j) params[1 + 3 * i + j] = (float)R[i][j];
      params[10 + i] = (float)sol[9 + i];
    }
  }
}

__device__ __forceinline__ double warp_sum(double x) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) x += __shfl_xor_sync(0xffffffffu, x, o);
  return x;
}

// ------------------------------------------------------------------ warp layout: a warp owns 32 rows
__global__ void __launch_bounds__(WARP_THREADS) pa_warp_kernel(const float* __restrict__ s1,
                                                               const float* __restrict__ s2, int64_t B, int n_points,
                                                               const int32_t* __restrict__ idx, int n_idx,
                                                               float* __restrict__ err, float* __restrict__ aligned,
                                                               float* __restrict__ params) {
  __shared__ double sh[WARP_THREADS / 32][32][NM];   // per row: the moments, then the solution
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int64_t row0 = (int64_t)blockIdx.x * WARP_ROWS + warp * 32;
  if (row0 >= B) return;
  const int rows = B - row0 < 32 ? (int)(B - row0) : 32;
  const int n = idx ? n_idx : n_points;
  const int p0 = idx ? __ldg(idx) : 0;
  double (*msh)[NM] = sh[warp];

  for (int r = 0; r < rows; ++r) {
    const size_t base = (size_t)(row0 + r) * n_points * 3;
    double o[6];
    load3(s1 + base + (size_t)p0 * 3, o[0], o[1], o[2]);
    load3(s2 + base + (size_t)p0 * 3, o[3], o[4], o[5]);
    double m[NM];
#pragma unroll
    for (int i = 0; i < NM; ++i) m[i] = 0.0;
    for (int k = lane; k < n; k += 32) {
      const size_t p = (size_t)(idx ? __ldg(idx + k) : k) * 3;
      accumulate(m, s1 + base + p, s2 + base + p, o);
    }
#pragma unroll
    for (int i = 0; i < NM; ++i) m[i] = warp_sum(m[i]);
    if (lane < NM) {
      double mine = m[0];
#pragma unroll
      for (int i = 1; i < NM; ++i) mine = lane == i ? m[i] : mine;
      msh[r][lane] = mine;
    }
  }
  __syncwarp();

  // one solve per lane: lane r solves row r
  double sol[NS];
  if (lane < rows) {
    const size_t base = (size_t)(row0 + lane) * n_points * 3 + (size_t)p0 * 3;
    double m[NM], o[6];
#pragma unroll
    for (int i = 0; i < NM; ++i) m[i] = msh[lane][i];
    load3(s1 + base, o[0], o[1], o[2]);
    load3(s2 + base, o[3], o[4], o[5]);
    solve(m, (double)n, o, sol, params ? params + (row0 + lane) * 13 : nullptr);
  }
  __syncwarp();
  if (lane < rows) {
#pragma unroll
    for (int i = 0; i < NS; ++i) msh[lane][i] = sol[i];
  }
  __syncwarp();

  double my_err = 0.0;
  for (int r = 0; r < rows; ++r) {
    const size_t base = (size_t)(row0 + r) * n_points * 3;
    const double* sr = msh[r];
    double e = 0.0;
    if (idx || !aligned) {
      for (int k = lane; k < n; k += 32) {
        const size_t p = (size_t)(idx ? __ldg(idx + k) : k) * 3;
        e += transform(sr, s1 + base + p, s2 + base + p, nullptr);
      }
    }
    if (aligned) {
      for (int k = lane; k < n_points; k += 32) {
        const size_t p = (size_t)k * 3;
        const double d = transform(sr, s1 + base + p, s2 + base + p, aligned + base + p);
        if (!idx) e += d;
      }
    }
    e = warp_sum(e);
    if (lane == r) my_err = e;
  }
  if (lane < rows) err[row0 + lane] = (float)(my_err / (double)n);
}

// ------------------------------------------------------------------ CTA layout: one CTA per row
// fixed-order sum over the CTA of NV values per thread; the result is in out[0..NV) for every thread
template <int NV>
__device__ __forceinline__ void cta_sum(double v[NV], double (*part)[NM], double* out) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int i = 0; i < NV; ++i) v[i] = warp_sum(v[i]);
  if (lane == 0) {
#pragma unroll
    for (int i = 0; i < NV; ++i) part[warp][i] = v[i];
  }
  __syncthreads();
  if (threadIdx.x < NV) {
    double s = 0.0;
#pragma unroll
    for (int w = 0; w < CTA_THREADS / 32; ++w) s += part[w][threadIdx.x];
    out[threadIdx.x] = s;
  }
  __syncthreads();
}

__global__ void __launch_bounds__(CTA_THREADS, 2) pa_cta_kernel(const float* __restrict__ s1,
                                                                const float* __restrict__ s2, int n_points,
                                                                const int32_t* __restrict__ idx, int n_idx,
                                                                float* __restrict__ err, float* __restrict__ aligned,
                                                                float* __restrict__ params) {
  __shared__ double part[CTA_THREADS / 32][NM];
  __shared__ double tot[NM];
  __shared__ double sol_sh[NS];
  const int64_t row = blockIdx.x;
  const size_t base = (size_t)row * n_points * 3;
  const int n = idx ? n_idx : n_points;
  const int p0 = idx ? __ldg(idx) : 0;
  double o[6];
  load3(s1 + base + (size_t)p0 * 3, o[0], o[1], o[2]);
  load3(s2 + base + (size_t)p0 * 3, o[3], o[4], o[5]);
  {
    double m[NM];
#pragma unroll
    for (int i = 0; i < NM; ++i) m[i] = 0.0;
    for (int k = threadIdx.x; k < n; k += CTA_THREADS) {
      const size_t p = (size_t)(idx ? __ldg(idx + k) : k) * 3;
      accumulate(m, s1 + base + p, s2 + base + p, o);
    }
    cta_sum<NM>(m, part, tot);
  }
  if (threadIdx.x == 0) {
    double sol[NS];
    solve(tot, (double)n, o, sol, params ? params + row * 13 : nullptr);
#pragma unroll
    for (int i = 0; i < NS; ++i) sol_sh[i] = sol[i];
  }
  __syncthreads();
  double sol[NS];
#pragma unroll
  for (int i = 0; i < NS; ++i) sol[i] = sol_sh[i];
  // backwards over the row; each thread takes the points it took in pass 1
  const int tid = threadIdx.x;
  double e[1] = {0.0};
  if (idx || !aligned) {
    for (int k = tid < n ? tid + (n - 1 - tid) / CTA_THREADS * CTA_THREADS : -1; k >= 0; k -= CTA_THREADS) {
      const size_t p = (size_t)(idx ? __ldg(idx + k) : k) * 3;
      e[0] += transform(sol, s1 + base + p, s2 + base + p, nullptr);
    }
  }
  if (aligned) {
    for (int k = tid < n_points ? tid + (n_points - 1 - tid) / CTA_THREADS * CTA_THREADS : -1; k >= 0;
         k -= CTA_THREADS) {
      const size_t p = (size_t)k * 3;
      const double d = transform(sol, s1 + base + p, s2 + base + p, aligned + base + p);
      if (!idx) e[0] += d;
    }
  }
  cta_sum<1>(e, part, tot);
  if (threadIdx.x == 0) err[row] = (float)(tot[0] / (double)n);
}

}  // namespace pa
}  // namespace dpb

extern "C" int dpb_procrustes(const float* s1, const float* s2, int64_t B, int n_points, const int32_t* idx,
                              int n_idx, float* err, float* aligned, float* params, void* stream) {
  using namespace dpb;
  if (!s1 || !s2 || !err || B <= 0 || B > INT32_MAX || n_points <= 0 || n_points > INT32_MAX / 3 ||
      (idx && n_idx <= 0))
    return fail(DPB_EINVAL, "dpb_procrustes: bad argument");
  PtrDeviceGuard guard(s1);
  cudaStream_t st = (cudaStream_t)stream;
  if (n_points <= pa::PA_WARP_MAX_POINTS)
    pa::pa_warp_kernel<<<(unsigned)((B + pa::WARP_ROWS - 1) / pa::WARP_ROWS), pa::WARP_THREADS, 0, st>>>(
        s1, s2, B, n_points, idx, n_idx, err, aligned, params);
  else
    pa::pa_cta_kernel<<<(unsigned)B, pa::CTA_THREADS, 0, st>>>(s1, s2, n_points, idx, n_idx, err, aligned, params);
  DPB_CUDA_CHECK(cudaGetLastError());
  return DPB_OK;
}
