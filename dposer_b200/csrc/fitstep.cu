// Kernels that close the fitting loops on the device (no eager framework ops inside an Adam step):
//
//   motion_data_kernel / motion_temporal_kernel   run/motion_denoising.py:255-262 -- the temporal vertex term
//       mean ||v[t] - v[t+1]|| and the joint data term mean ||Jtr[:, :22] - noisy||, value AND cotangents, per
//       60-frame sequence (adjacent rows of different sequences are not differenced, SURVEY App. B-7; the
//       `if data_term > 0` NaN guard is a per-sequence device predicate, App. B-8)
//   camera_fit_kernel                              lib/body_model/fitting_losses.py:106-136, value and cotangents
//   adam_kernel                                    torch.optim.Adam's update (the reference's optimiser in
//       run/completion.py:178, run/motion_denoising.py:217, run/smplify.py:206,236), fused with the gradient assembly
//   affine_cols_kernel                             Posenormalizer z-score (lib/dataset/AMASS.py:187-259)
//   axis_to_rot6d kernels                          Posenormalizer.offline_normalize(from_axis=True) of a rot6d prior
//       (run/smplify.py:109-115, lib/utils/transforms.py:237-255) and its vector-Jacobian product
//   joint_map kernels                             lib/body_model/smpl.py:70 joints[:, joint_map] and its adjoint
#include <cmath>

#include "common.cuh"

namespace dpb {

// ---- data term: one block per sequence.  g_joints[rows, n_out, 3] gets the cotangent of the first n_data joints
// (zero elsewhere); seq_terms[seq*2 + 1] = the sequence's data term.
__global__ void __launch_bounds__(256) motion_data_kernel(const float* __restrict__ joints,
                                                          const float* __restrict__ target, int seq_len, int n_out,
                                                          int n_data, float w_data, float* __restrict__ g_joints,
                                                          float* __restrict__ seq_terms) {
  const int64_t row0 = (int64_t)blockIdx.x * seq_len;
  const int n = seq_len * n_data;
  float acc = 0.f;
  for (int i = threadIdx.x; i < n; i += 256) {
    const int f = i / n_data, j = i % n_data;
    const float* a = joints + ((row0 + f) * n_out + j) * 3;
    const float* t = target + ((row0 + f) * n_data + j) * 3;
    const float dx = a[0] - t[0], dy = a[1] - t[1], dz = a[2] - t[2];
    acc += sqrtf(dx * dx + dy * dy + dz * dz);
  }
  __shared__ float part[8];
  __shared__ float total;
  for (int s = 16; s > 0; s >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, s);
  if ((threadIdx.x & 31) == 0) part[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0)
    total = (((part[0] + part[1]) + (part[2] + part[3])) + ((part[4] + part[5]) + (part[6] + part[7]))) / (float)n;
  __syncthreads();
  const float data = total;
  if (seq_terms && threadIdx.x == 0) seq_terms[blockIdx.x * 2 + 1] = data;
  // reference: `if data_term > 0` (false for NaN and 0) -- the term is dropped for this sequence only
  const float c = (data > 0.f) ? w_data / (float)n : 0.f;
  for (int i = threadIdx.x; i < seq_len * n_out; i += 256) {
    const int f = i / n_out, j = i % n_out;
    float* g = g_joints + ((row0 + f) * n_out + j) * 3;
    float gx = 0.f, gy = 0.f, gz = 0.f;
    if (j < n_data && c != 0.f) {
      const float* a = joints + ((row0 + f) * n_out + j) * 3;
      const float* t = target + ((row0 + f) * n_data + j) * 3;
      const float dx = a[0] - t[0], dy = a[1] - t[1], dz = a[2] - t[2];
      const float d2 = dx * dx + dy * dy + dz * dz;
      const float s = d2 > 0.f ? c * rsqrtf(d2) : 0.f;   // (the reference's sqrt backward gives NaN at exactly 0)
      gx = s * dx; gy = s * dy; gz = s * dz;
    }
    g[0] = gx; g[1] = gy; g[2] = gz;
  }
}

// ---- temporal term: grid (ceil(V/128), n_seq); a thread owns one vertex and walks the sequence's frames, so every
// vertex is read once and its cotangent written once (coalesced across the 128 vertices of the block).
__global__ void __launch_bounds__(128) motion_temporal_kernel(const float* __restrict__ verts, int seq_len, int V,
                                                              float w_temp, float* __restrict__ g_verts,
                                                              float* __restrict__ seq_terms) {
  const int v = blockIdx.x * 128 + threadIdx.x;
  const int64_t row0 = (int64_t)blockIdx.y * seq_len;
  const float c = w_temp / ((float)(seq_len - 1) * (float)V);
  float acc = 0.f;
  if (v < V) {
    const size_t stride = (size_t)V * 3;
    const float* p = verts + (size_t)row0 * stride + (size_t)v * 3;
    float* g = g_verts + (size_t)row0 * stride + (size_t)v * 3;
    float cx = p[0], cy = p[1], cz = p[2];     // current frame
    float gx = 0.f, gy = 0.f, gz = 0.f;        // cotangent of the current frame from the previous pair
    for (int f = 0; f + 1 < seq_len; ++f) {
      const float* q = p + (size_t)(f + 1) * stride;
      const float nx = q[0], ny = q[1], nz = q[2];
      const float dx = cx - nx, dy = cy - ny, dz = cz - nz;
      const float d2 = dx * dx + dy * dy + dz * dz;
      const float r = d2 > 0.f ? rsqrtf(d2) : 0.f;
      acc += d2 * r;                            // ||d||
      const float ux = c * r * dx, uy = c * r * dy, uz = c * r * dz;
      float* o = g + (size_t)f * stride;
      o[0] = gx + ux; o[1] = gy + uy; o[2] = gz + uz;
      gx = -ux; gy = -uy; gz = -uz;
      cx = nx; cy = ny; cz = nz;
    }
    float* o = g + (size_t)(seq_len - 1) * stride;
    o[0] = gx; o[1] = gy; o[2] = gz;
  }
  if (seq_terms) {   // reporting only (fp32 atomics: order-dependent in the last bits; the cotangents do not depend on it)
    for (int s = 16; s > 0; s >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, s);
    if ((threadIdx.x & 31) == 0) atomicAdd(seq_terms + blockIdx.y * 2, acc / ((float)(seq_len - 1) * (float)V));
  }
}

// ---- camera fitting loss (fitting_losses.py:106-136): thread per sample
__global__ void camera_fit_kernel(const float* __restrict__ joints, const float* __restrict__ kp2d,
                                  const float* __restrict__ conf, const float* __restrict__ center,
                                  const float* __restrict__ cam_t, const float* __restrict__ cam_est,
                                  const float* __restrict__ focal_b, float focal, float depth_w, int K,
                                  float* __restrict__ loss, float* __restrict__ g_joints,
                                  float* __restrict__ g_cam, int64_t B) {
  const int64_t b = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  const int op[4] = {9, 12, 2, 5};        // OP RHip, OP LHip, OP RShoulder, OP LShoulder (constants.JOINT_IDS)
  const int gt[4] = {27, 28, 33, 34};     // Right Hip, Left Hip, Right Shoulder, Left Shoulder
  if (focal_b) focal = focal_b[b];
  float cmin = conf[b * K + op[0]];
  for (int i = 1; i < 4; ++i) cmin = fminf(cmin, conf[b * K + op[i]]);
  const bool valid = cmin > 0.f;          // all four OpenPose detections present, else the GT slots
  if (g_joints)
    for (int i = 0; i < K * 3; ++i) g_joints[b * K * 3 + i] = 0.f;
  const float cx = center[b * 2], cy = center[b * 2 + 1];
  float acc = 0.f;
  for (int i = 0; i < 4; ++i) {
    const int k = valid ? op[i] : gt[i];
    const float* X = joints + (b * K + k) * 3;
    const float iz = 1.0f / X[2];
    const float ex = kp2d[(b * K + k) * 2] - (focal * X[0] * iz + cx);
    const float ey = kp2d[(b * K + k) * 2 + 1] - (focal * X[1] * iz + cy);
    acc += ex * ex + ey * ey;
    if (g_joints) {
      float* G = g_joints + (b * K + k) * 3;
      G[0] = -2.f * ex * focal * iz;
      G[1] = -2.f * ey * focal * iz;
      G[2] = 2.f * (ex * X[0] + ey * X[1]) * focal * iz * iz;
    }
  }
  const float dz = cam_t[b * 3 + 2] - cam_est[b * 3 + 2];
  loss[b] = acc + depth_w * depth_w * dz * dz;
  if (g_cam) {
    g_cam[b * 3] = 0.f;
    g_cam[b * 3 + 1] = 0.f;
    g_cam[b * 3 + 2] = 2.f * depth_w * depth_w * dz;
  }
}

// ---- Adam (torch.optim.Adam, amsgrad off, weight decay 0): grad = s1 g1 + s2 col_scale2[c] g2 + s3 g3, all strided views
__global__ void adam_kernel(float* __restrict__ param, int64_t ld_p, float* __restrict__ m, float* __restrict__ v,
                            const float* __restrict__ g1, int64_t ld1, float s1, const float* __restrict__ g2,
                            int64_t ld2, float s2, const float* __restrict__ col_scale2,
                            const float* __restrict__ g3, int64_t ld3, float s3, int64_t rows, int cols,
                            float step_size, float beta1, float beta2, float inv_sqrt_bc2, float eps) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= rows * cols) return;
  const int64_t r = i / cols;
  const int c = (int)(i % cols);
  float g = s1 * g1[r * ld1 + c];
  if (g2) g += s2 * (col_scale2 ? col_scale2[c] : 1.0f) * g2[r * ld2 + c];
  if (g3) g += s3 * g3[r * ld3 + c];
  const float mi = beta1 * m[i] + (1.0f - beta1) * g;          // exp_avg.lerp_(grad, 1 - beta1)
  const float vi = beta2 * v[i] + (1.0f - beta2) * g * g;      // exp_avg_sq.mul_(beta2).addcmul_(grad, grad, 1 - beta2)
  m[i] = mi;
  v[i] = vi;
  const float denom = sqrtf(vi) * inv_sqrt_bc2 + eps;          // (exp_avg_sq.sqrt() / bias_correction2_sqrt).add_(eps)
  param[r * ld_p + c] -= step_size * (mi / denom);             // param.addcdiv_(exp_avg, denom, value=-lr / bias_correction1)
}

__global__ void affine_cols_kernel(const float* __restrict__ x, int64_t ldx, const float* __restrict__ mean,
                                   const float* __restrict__ sd, float* __restrict__ out, int64_t ldo, int64_t rows,
                                   int cols, int inverse, float squash) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= rows * cols) return;
  const int64_t r = i / cols;
  const int c = (int)(i % cols);
  float xv = x[r * ldx + c];
  if (squash > 0.f) xv = tanhf(xv * squash);
  out[r * ldo + c] = inverse ? xv * sd[c] + mean[c] : (xv - mean[c]) / sd[c];
}

// ---- axis-angle -> normalised rot6d, one thread per (row, joint).  With theta = |a| and K = [a]x:
//   R = I + A K + B K^2,                       A = sin t / t, B = (1 - cos t) / t^2
//   dR/da_i = C a_i K + A [e_i]x + D a_i K^2 + B ([e_i]x K + K [e_i]x),   C = A' / t, D = B' / t
// rot6d = (R00, R01, R10, R11, R20, R21), transforms.axis_angle_to_rot6d's [:, :3, :2] layout.
//
// Series branch: below theta = 1.2 the four coefficients come from their Taylor series through theta^8, above it from
// the closed forms.  In fp32 the closed forms lose to cancellation as theta falls (C and D worst, D ~ 1e-6 relative at
// 1.2 and 2e-6 at 0.9); the five-term series is within 2.5e-7 relative everywhere below 1.2 (its first dropped term is
// largest for A: theta^10 / 11!).  The three-term series (through theta^4) cannot do this: where its truncation error
// falls to 1e-6 (theta ~ 0.5), the closed form of D is already 1e-5 off.  Both figures are measured against fp64.
// theta = 0 lands in the series branch and needs no special case; a non-finite coordinate fails the comparison,
// takes the closed form and turns the joint's outputs into NaN (every output entry carries a B or D factor).
struct Rot6dCoefs {
  float A, B, C, D;
};

__device__ __forceinline__ Rot6dCoefs rot6d_coefs(float t2) {
  Rot6dCoefs k;
  if (t2 < 1.44f) {
    k.A = 1.f + t2 * (-1.f / 6 + t2 * (1.f / 120 + t2 * (-1.f / 5040 + t2 * (1.f / 362880))));
    k.B = 0.5f + t2 * (-1.f / 24 + t2 * (1.f / 720 + t2 * (-1.f / 40320 + t2 * (1.f / 3628800))));
    k.C = -1.f / 3 + t2 * (1.f / 30 + t2 * (-1.f / 840 + t2 * (1.f / 45360 + t2 * (-1.f / 3991680))));
    k.D = -1.f / 12 + t2 * (1.f / 180 + t2 * (-1.f / 6720 + t2 * (1.f / 453600 + t2 * (-1.f / 47900160))));
  } else {
    const float t = sqrtf(t2);
    float s, c;
    sincosf(t, &s, &c);
    const float it2 = 1.f / t2;
    k.A = s / t;
    k.B = (1.f - c) * it2;
    k.C = (t * c - s) / (t2 * t);
    k.D = (t * s - 2.f * (1.f - c)) * (it2 * it2);
  }
  return k;
}

__global__ void __launch_bounds__(256) axis_to_rot6d_kernel(const float* __restrict__ x, int64_t ldx,
                                                             const float* __restrict__ mean, const float* __restrict__ sd,
                                                             float* __restrict__ out, int64_t ldo, int64_t rows, int nj) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= rows * nj) return;
  const int64_t r = i / nj;
  const int j = (int)(i % nj);
  const float* a = x + r * ldx + 3 * j;
  const float a0 = a[0], a1 = a[1], a2 = a[2];
  const float q0 = a0 * a0, q1 = a1 * a1, q2 = a2 * a2;
  const Rot6dCoefs k = rot6d_coefs(q0 + q1 + q2);
  // K^2 = a a^T - theta^2 I; its diagonal as -(sum of the other two squares), free of cancellation
  const float rot[6] = {1.f - k.B * (q1 + q2), -k.A * a2 + k.B * a0 * a1,
                        k.A * a2 + k.B * a0 * a1, 1.f - k.B * (q0 + q2),
                        -k.A * a1 + k.B * a0 * a2, k.A * a0 + k.B * a1 * a2};
  float* o = out + r * ldo + 6 * j;
#pragma unroll
  for (int c = 0; c < 6; ++c) o[c] = (rot[c] - mean[6 * j + c]) / sd[6 * j + c];
}

// g_x_i = <G, dR/da_i> with G = the cotangent of R (rows 0..2, columns 0..1 from g / std, column 2 zero):
//   g_x = a (C <G,K> + D (a^T G a - theta^2 tr G) - 2 B tr G) + A w + B (G a + G^T a),
// where w = (G21 - G12, G02 - G20, G10 - G01) is the vector of G's skew part (<G, [v]x> = v . w).
__global__ void __launch_bounds__(256) axis_to_rot6d_vjp_kernel(const float* __restrict__ x, int64_t ldx,
                                                                 const float* __restrict__ sd, const float* __restrict__ g,
                                                                 int64_t ldg, float* __restrict__ g_x, int64_t ldgx,
                                                                 int64_t rows, int nj) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= rows * nj) return;
  const int64_t r = i / nj;
  const int j = (int)(i % nj);
  const float* a = x + r * ldx + 3 * j;
  const float a0 = a[0], a1 = a[1], a2 = a[2];
  const float t2 = a0 * a0 + a1 * a1 + a2 * a2;
  const Rot6dCoefs k = rot6d_coefs(t2);
  const float* gr = g + r * ldg + 6 * j;
  const float G00 = gr[0] / sd[6 * j], G01 = gr[1] / sd[6 * j + 1], G10 = gr[2] / sd[6 * j + 2],
              G11 = gr[3] / sd[6 * j + 3], G20 = gr[4] / sd[6 * j + 4], G21 = gr[5] / sd[6 * j + 5];
  const float w0 = G21, w1 = -G20, w2 = G10 - G01;           // G02 = G12 = 0
  const float trG = G00 + G11;
  const float Ga0 = G00 * a0 + G01 * a1, Ga1 = G10 * a0 + G11 * a1, Ga2 = G20 * a0 + G21 * a1;    // G a
  const float Gta0 = G00 * a0 + G10 * a1 + G20 * a2, Gta1 = G01 * a0 + G11 * a1 + G21 * a2;       // G^T a (third: 0)
  const float aGa = a0 * Ga0 + a1 * Ga1 + a2 * Ga2;
  const float s = k.C * (a0 * w0 + a1 * w1 + a2 * w2) + k.D * (aGa - t2 * trG) - 2.f * k.B * trG;
  float* o = g_x + r * ldgx + 3 * j;
  o[0] = s * a0 + k.A * w0 + k.B * (Ga0 + Gta0);
  o[1] = s * a1 + k.A * w1 + k.B * (Ga1 + Gta1);
  o[2] = s * a2 + k.A * w2 + k.B * Ga2;
}

// cotangent of mean((x*m - o*m)^2) (nn.MSELoss 'mean' on masked tensors, run/completion.py:197): 2 m^2 (x - o) / n
__global__ void masked_mse_grad_kernel(const float* __restrict__ x, const float* __restrict__ o,
                                       const float* __restrict__ m, float* __restrict__ g, int64_t n) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float mi = m[i];
  g[i] = 2.0f * mi * (x[i] * mi - o[i] * mi) / (float)n;
}

__global__ void joint_gather_kernel(const float* __restrict__ joints, int n_in, const int32_t* __restrict__ map,
                                    int n_map, float* __restrict__ out, int64_t B) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= B * n_map * 3) return;
  const int64_t b = i / (n_map * 3);
  const int k = (int)((i / 3) % n_map), c = (int)(i % 3);
  out[i] = joints[(b * n_in + map[k]) * 3 + c];
}

// adjoint of the gather: the map has repeated entries (smpl.py:53-58), so one thread per (sample, coordinate) adds its
// n_map contributions in a fixed order (deterministic, no atomics)
__global__ void joint_scatter_kernel(const float* __restrict__ g_out, int n_map, const int32_t* __restrict__ map,
                                     int n_in, float* __restrict__ g_in, int64_t B) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= B * 3) return;
  const int64_t b = i / 3;
  const int c = (int)(i % 3);
  float* gi = g_in + b * n_in * 3 + c;
  for (int j = 0; j < n_in; ++j) gi[j * 3] = 0.f;
  for (int k = 0; k < n_map; ++k) gi[map[k] * 3] += g_out[(b * n_map + k) * 3 + c];
}

// zero-padded 3-tap smoothing along the frames of each sequence (gaussian_smoothing(window_size=3), lib/utils/misc.py:84-95,
// as applied per sequence by run/motion_denoising.py:281-285); the first / last frame of a sequence keep their values
__global__ void seq_smooth3_kernel(const float* __restrict__ x, float* __restrict__ out, int L, int C, float w0, float w1,
                                   float w2, int keep_ends, int64_t rows) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= rows * C) return;
  const int64_t r = i / C;
  const int f = (int)(r % L);
  const float xm = f > 0 ? x[i - C] : 0.f, xp = f < L - 1 ? x[i + C] : 0.f, x0 = x[i];
  out[i] = (keep_ends && (f == 0 || f == L - 1)) ? x0 : w0 * xm + w1 * x0 + w2 * xp;
}

}  // namespace dpb

using namespace dpb;

extern "C" int dpb_motion_loss(const float* verts, const float* joints, const float* target, int64_t rows,
                               int seq_len, int V, int n_out, int n_data, float w_temp, float w_data, float* g_verts,
                               float* g_joints, float* seq_terms, void* stream) {
  DPB_REQUIRE(verts && joints && target && g_verts && g_joints, "dpb_motion_loss: null argument");
  DPB_REQUIRE(seq_len >= 2 && rows > 0 && rows % seq_len == 0, "dpb_motion_loss: rows must be whole sequences of >= 2 frames");
  DPB_REQUIRE(V > 0 && n_data > 0 && n_data <= n_out, "dpb_motion_loss: bad sizes");
  PtrDeviceGuard guard(verts);
  cudaStream_t st = (cudaStream_t)stream;
  const int64_t n_seq = rows / seq_len;
  DPB_REQUIRE(n_seq <= 65535, "dpb_motion_loss: at most 65535 sequences per call");
  if (seq_terms) DPB_CUDA_CHECK(cudaMemsetAsync(seq_terms, 0, (size_t)n_seq * 2 * sizeof(float), st));
  motion_data_kernel<<<(unsigned)n_seq, 256, 0, st>>>(joints, target, seq_len, n_out, n_data, w_data, g_joints, seq_terms);
  motion_temporal_kernel<<<dim3((unsigned)((V + 127) / 128), (unsigned)n_seq), 128, 0, st>>>(verts, seq_len, V, w_temp,
                                                                                            g_verts, seq_terms);
  DPB_CUDA_CHECK(cudaGetLastError());
  return DPB_OK;
}

extern "C" int dpb_camera_fit_loss(const float* joints, const float* joints_2d, const float* conf, const float* center,
                                   const float* cam_t, const float* cam_t_est, const float* focal_b, float focal,
                                   float depth_weight, int n_joints, float* loss, float* g_joints, float* g_cam_t,
                                   int64_t B, void* stream) {
  DPB_REQUIRE(joints && joints_2d && conf && center && cam_t && cam_t_est && loss, "dpb_camera_fit_loss: null argument");
  DPB_REQUIRE(n_joints > 34, "dpb_camera_fit_loss: needs the 49-joint SMPLify layout (torso joints up to index 34)");
  if (B <= 0) return DPB_OK;
  PtrDeviceGuard guard(joints);
  camera_fit_kernel<<<(unsigned)((B + 127) / 128), 128, 0, (cudaStream_t)stream>>>(
      joints, joints_2d, conf, center, cam_t, cam_t_est, focal_b, focal, depth_weight, n_joints, loss, g_joints, g_cam_t, B);
  DPB_CUDA_CHECK(cudaGetLastError());
  return DPB_OK;
}

extern "C" int dpb_adam_step(float* param, int64_t ld_p, float* m, float* v, const float* g1, int64_t ld1, float s1,
                             const float* g2, int64_t ld2, float s2, const float* col_scale2, const float* g3,
                             int64_t ld3, float s3, int64_t rows, int cols, float lr, float beta1, float beta2,
                             float eps, int step, void* stream) {
  DPB_REQUIRE(param && m && v && g1 && rows >= 0 && cols > 0 && step >= 1, "dpb_adam_step: bad argument");
  if (rows == 0) return DPB_OK;
  PtrDeviceGuard guard(param);
  // torch computes the bias corrections in double on the host (torch/optim/adam.py _single_tensor_adam)
  const double bc1 = 1.0 - std::pow((double)beta1, step), bc2 = 1.0 - std::pow((double)beta2, step);
  const float step_size = (float)((double)lr / bc1), inv_sqrt_bc2 = (float)(1.0 / std::sqrt(bc2));
  const int64_t n = rows * cols;
  adam_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(param, ld_p, m, v, g1, ld1, s1, g2, ld2, s2,
                                                                            col_scale2, g3, ld3, s3, rows, cols, step_size,
                                                                            beta1, beta2, inv_sqrt_bc2, eps);
  DPB_CUDA_CHECK(cudaGetLastError());
  return DPB_OK;
}

extern "C" int dpb_affine_cols(const float* x, int64_t ldx, const float* mean, const float* sd, float* out,
                               int64_t ldo, int64_t rows, int cols, int inverse, float squash, void* stream) {
  DPB_REQUIRE(x && mean && sd && out && cols > 0 && ldo >= cols, "dpb_affine_cols: bad argument");
  if (rows <= 0) return DPB_OK;
  PtrDeviceGuard guard(x);
  const int64_t n = rows * cols;
  affine_cols_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(x, ldx, mean, sd, out, ldo, rows, cols, inverse, squash);
  DPB_CUDA_CHECK(cudaGetLastError());
  return DPB_OK;
}

extern "C" int dpb_axis_to_rot6d_cols(const float* x, int64_t ldx, const float* mean, const float* sd, float* out,
                                      int64_t ldo, int64_t rows, int n_joints, void* stream) {
  DPB_REQUIRE(x && mean && sd && out && n_joints > 0 && rows >= 0, "dpb_axis_to_rot6d_cols: bad argument");
  DPB_REQUIRE(ldx >= 3 * (int64_t)n_joints && ldo >= 6 * (int64_t)n_joints,
              "dpb_axis_to_rot6d_cols: row strides must cover 3 * n_joints inputs and 6 * n_joints outputs");
  if (rows == 0) return DPB_OK;
  PtrDeviceGuard guard(x);
  const int64_t n = rows * n_joints;
  axis_to_rot6d_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(x, ldx, mean, sd, out, ldo, rows,
                                                                                      n_joints);
  DPB_CUDA_CHECK(cudaGetLastError());
  return DPB_OK;
}

extern "C" int dpb_axis_to_rot6d_cols_vjp(const float* x, int64_t ldx, const float* sd, const float* g, int64_t ldg,
                                          float* g_x, int64_t ldgx, int64_t rows, int n_joints, void* stream) {
  DPB_REQUIRE(x && sd && g && g_x && n_joints > 0 && rows >= 0, "dpb_axis_to_rot6d_cols_vjp: bad argument");
  DPB_REQUIRE(ldx >= 3 * (int64_t)n_joints && ldg >= 6 * (int64_t)n_joints && ldgx >= 3 * (int64_t)n_joints,
              "dpb_axis_to_rot6d_cols_vjp: row strides must cover 3 * n_joints inputs / gradients and 6 * n_joints "
              "cotangents");
  if (rows == 0) return DPB_OK;
  PtrDeviceGuard guard(x);
  const int64_t n = rows * n_joints;
  axis_to_rot6d_vjp_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(x, ldx, sd, g, ldg, g_x, ldgx,
                                                                                          rows, n_joints);
  DPB_CUDA_CHECK(cudaGetLastError());
  return DPB_OK;
}

extern "C" int dpb_masked_mse_grad(const float* x, const float* obs, const float* mask, float* grad, int64_t n,
                                   void* stream) {
  DPB_REQUIRE(x && obs && mask && grad, "dpb_masked_mse_grad: null argument");
  if (n <= 0) return DPB_OK;
  PtrDeviceGuard guard(x);
  masked_mse_grad_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(x, obs, mask, grad, n);
  DPB_CUDA_CHECK(cudaGetLastError());
  return DPB_OK;
}

extern "C" int dpb_joint_map_gather(const float* joints, int n_in, const int32_t* map, int n_map, float* out,
                                    int64_t B, void* stream) {
  DPB_REQUIRE(joints && map && out && n_in > 0 && n_map > 0, "dpb_joint_map_gather: bad argument");
  if (B <= 0) return DPB_OK;
  PtrDeviceGuard guard(joints);
  const int64_t n = B * n_map * 3;
  joint_gather_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(joints, n_in, map, n_map, out, B);
  DPB_CUDA_CHECK(cudaGetLastError());
  return DPB_OK;
}

extern "C" int dpb_joint_map_scatter(const float* g_out, int n_map, const int32_t* map, int n_in, float* g_in,
                                     int64_t B, void* stream) {
  DPB_REQUIRE(g_out && map && g_in && n_in > 0 && n_map > 0, "dpb_joint_map_scatter: bad argument");
  if (B <= 0) return DPB_OK;
  PtrDeviceGuard guard(g_out);
  const int64_t n = B * 3;
  joint_scatter_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(g_out, n_map, map, n_in, g_in, B);
  DPB_CUDA_CHECK(cudaGetLastError());
  return DPB_OK;
}

extern "C" int dpb_seq_smooth3(const float* x, float* out, int64_t rows, int seq_len, int cols, float w0, float w1, float w2,
                               int keep_ends, void* stream) {
  DPB_REQUIRE(x && out && x != out && rows > 0 && seq_len > 0 && cols > 0 && rows % seq_len == 0, "dpb_seq_smooth3: bad argument");
  PtrDeviceGuard guard(x);
  const int64_t n = rows * cols;
  seq_smooth3_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(x, out, seq_len, cols, w0, w1, w2, keep_ends, rows);
  DPB_CUDA_CHECK(cudaGetLastError());
  return DPB_OK;
}
