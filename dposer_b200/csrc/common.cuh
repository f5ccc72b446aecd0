// Shared device/host helpers for libdposer_b200 (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <cuda_fp16.h>
#include <cuda_bf16.h>
#include <stdint.h>
#include <string>

#include "../../include/dposer_b200.h"

namespace dpb {

// ---------------------------------------------------------------- errors
void set_error(const std::string& msg);
int fail(int code, const std::string& msg);

#define DPB_CUDA_CHECK(expr)                                                                  \
  do {                                                                                        \
    cudaError_t _e = (expr);                                                                  \
    if (_e != cudaSuccess)                                                                    \
      return ::dpb::fail(DPB_ECUDA, std::string(#expr) + ": " + cudaGetErrorString(_e));      \
  } while (0)

#define DPB_REQUIRE(cond, msg)                                   \
  do {                                                           \
    if (!(cond)) return ::dpb::fail(DPB_EINVAL, std::string(msg)); \
  } while (0)

static inline size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

// Makes `device` current for the duration of an entry point and restores the caller's device afterwards
// (torch tracks its own current device; the library must not change it behind torch's back).
struct DeviceGuard {
  int prev = -1;
  bool switched = false;
  explicit DeviceGuard(int device) {
    if (cudaGetDevice(&prev) == cudaSuccess && prev != device) switched = cudaSetDevice(device) == cudaSuccess;
  }
  ~DeviceGuard() {
    if (switched) cudaSetDevice(prev);
  }
};
// device that owns a device pointer (entry points without a handle); -1 if it cannot be determined
static inline int device_of(const void* p) {
  cudaPointerAttributes a;
  if (!p || cudaPointerGetAttributes(&a, p) != cudaSuccess || a.type != cudaMemoryTypeDevice) {
    cudaGetLastError();
    return -1;
  }
  return a.device;
}
struct PtrDeviceGuard : DeviceGuard {
  static int pick(const void* p) {
    int d = device_of(p), cur = 0;
    if (d < 0) { cudaGetDevice(&cur); return cur; }
    return d;
  }
  explicit PtrDeviceGuard(const void* p) : DeviceGuard(pick(p)) {}
};

// carve sub-buffers out of the caller's workspace (256-byte aligned)
struct WsCarver {
  char* base;
  size_t off = 0, cap;
  WsCarver(void* p, size_t bytes) : base(static_cast<char*>(p)), cap(bytes) {}
  template <class T>
  T* take(size_t n) {
    off = align_up(off, 256);
    T* r = reinterpret_cast<T*>(base + off);
    off += n * sizeof(T);
    return r;
  }
  bool ok() const { return off <= cap; }
};

// ---------------------------------------------------------------- geometry
constexpr int D = DPB_POSE_DIM;     // 63
constexpr int DP = 64;              // padded pose dim
// The pose width is a property of the score handle: 63 (axis-angle) or 126 (rot6d), padded to DP = 64 or 128.
// Kernels that depend on it are templated on the padded width; D and DP above are the 63-D instantiation.
constexpr int D126 = DPB_POSE_DIM_ROT6D;
constexpr int DP128 = 128;
__host__ __device__ constexpr int pose_dim_of(int dp) { return dp == DP128 ? D126 : D; }
constexpr int H = DPB_HIDDEN;       // 1024
constexpr int E = DPB_EMBED;        // 512
constexpr int NL = DPB_NUM_DENSE;   // 5 hidden-producing dense layers
constexpr int GROUP = 32;           // channels per GroupNorm group (1024/32)
constexpr float GN_EPS = 1e-5f;

// ---------------------------------------------------------------- Philox4x32-10 + Box-Muller
// One counter = (row, step, slot*quads + quad) -> 4 normals for columns 4*quad..4*quad+3 of `row`, where
// quads = DP/4 is the number of column quads of the padded row: 16 for the 63-D layout, 32 for the 126-D one.
// Every (slot, column) of a row therefore has its own counter word (slots 0..4 are in use); the 126-D layout
// is a different stream from the 63-D one, not an extension of it.  Both engines (fp32 and tcgen05) call this
// with the same arguments, so the same seed gives the same noise on either path.
__host__ __device__ __forceinline__ uint32_t mulhilo32(uint32_t a, uint32_t b, uint32_t* hi) {
#ifdef __CUDA_ARCH__
  *hi = __umulhi(a, b);
  return a * b;
#else
  uint64_t p = (uint64_t)a * b;
  *hi = (uint32_t)(p >> 32);
  return (uint32_t)p;
#endif
}

__host__ __device__ __forceinline__ void philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3,
                                                       uint32_t k0, uint32_t k1, uint32_t out[4]) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    uint32_t hi0, hi1;
    uint32_t lo0 = mulhilo32(0xD2511F53u, c0, &hi0);
    uint32_t lo1 = mulhilo32(0xCD9E8D57u, c2, &hi1);
    uint32_t n0 = hi1 ^ c1 ^ k0, n1 = lo1, n2 = hi0 ^ c3 ^ k1, n3 = lo0;
    c0 = n0; c1 = n1; c2 = n2; c3 = n3;
    k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
  }
  out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}

__device__ __forceinline__ void normal4(uint64_t seed, uint64_t row, uint32_t step, uint32_t slot, uint32_t quad,
                                        float z[4], uint32_t quads = 16) {
  uint32_t r[4];
  philox4x32_10((uint32_t)row, (uint32_t)(row >> 32), step, slot * quads + quad, (uint32_t)seed,
                (uint32_t)(seed >> 32), r);
  // uniforms in (0,1]
  const float s = 2.3283064365386963e-10f;  // 2^-32
  float u0 = ((float)r[0] + 1.0f) * s, u1 = (float)r[1] * s;
  float u2 = ((float)r[2] + 1.0f) * s, u3 = (float)r[3] * s;
  u0 = fminf(u0, 1.0f); u2 = fminf(u2, 1.0f);
  float m0 = sqrtf(-2.0f * logf(u0)), m1 = sqrtf(-2.0f * logf(u2));
  float s0, c0, s1, c1;
  sincospif(2.0f * u1, &s0, &c0);
  sincospif(2.0f * u3, &s1, &c1);
  z[0] = m0 * c0; z[1] = m0 * s0; z[2] = m1 * c1; z[3] = m1 * s1;
}

__device__ __forceinline__ float silu(float v) { return v / (1.0f + __expf(-v)); }

}  // namespace dpb
