// Self-intersection metric (reference self_intersections_percentage, lib/utils/metric.py:41-89, which runs pymeshlab
// on the CPU): per-face selection and per-mesh selected-face counts of a batch of meshes that share one topology.
// The decision rule is specified in dposer_b200/metric.py; oracle/selfisect_ref.py restates it in numpy.
//
// One persistent CTA per SM walks the meshes b = blockIdx.x, blockIdx.x + gridDim.x, ...  Per mesh:
//   1. face AABBs (fp32, exact min / max) into the CTA's workspace slice, mesh bounds, finiteness of every face vertex;
//   2. a uniform grid over the mesh bounds in shared memory, built by a counting sort of (cell, face) entries over the
//      cells each face AABB overlaps; cells are coarsened until the entries fit (one cell holds every face, so the
//      coarsening ends);
//   3. every pair of faces listed in a cell whose closed AABBs overlap is tested in the cell that holds the lower
//      corner of the overlap -- exactly once: the cell map is monotone, so that cell lies in both faces' ranges;
//   4. the narrow phase in fp64 with explicitly rounded operations (__dmul_rn / __dadd_rn / __dsub_rn are never fused
//      into FMAs), in the oracle's association, so both take every decision on the same fp64 value;
//   5. selected faces as a bitset (atomicOr is idempotent), counted with popc: integer sums, deterministic.
// No host synchronisation, no allocation: the workspace comes from the caller, the call can be graph-captured.
#include <algorithm>

#include "common.cuh"

struct dpb_selfisect {
  int device = 0, V = 0, nF = 0, sm_count = 0;
  int32_t* faces = nullptr;  // DEVICE [nF,3]
};

namespace dpb {
namespace si {

constexpr int THREADS = 512;
constexpr int CMAX = 16384;   // grid cells
constexpr int FMAX = 32768;   // faces (16-bit ids in the cell lists, selection bitset of FMAX bits)
constexpr int ECAP = 73728;   // (cell, face) entries
constexpr int MAX_DIM = 1024; // cells per axis
constexpr size_t SMEM = (size_t)CMAX * 4 + FMAX / 8 + (size_t)ECAP * 2;  // 217 088 B
constexpr int NWARP = THREADS / 32;

struct V3 {
  double x, y, z;
};
__device__ __forceinline__ V3 sub(V3 a, V3 b) { return {__dsub_rn(a.x, b.x), __dsub_rn(a.y, b.y), __dsub_rn(a.z, b.z)}; }
__device__ __forceinline__ V3 cross(V3 a, V3 b) {
  return {__dsub_rn(__dmul_rn(a.y, b.z), __dmul_rn(a.z, b.y)), __dsub_rn(__dmul_rn(a.z, b.x), __dmul_rn(a.x, b.z)),
          __dsub_rn(__dmul_rn(a.x, b.y), __dmul_rn(a.y, b.x))};
}
__device__ __forceinline__ double dot(V3 a, V3 b) {
  return __dadd_rn(__dadd_rn(__dmul_rn(a.x, b.x), __dmul_rn(a.y, b.y)), __dmul_rn(a.z, b.z));
}
__device__ __forceinline__ V3 midpoint(V3 a, V3 b) {
  return {__dmul_rn(__dadd_rn(a.x, b.x), 0.5), __dmul_rn(__dadd_rn(a.y, b.y), 0.5), __dmul_rn(__dadd_rn(a.z, b.z), 0.5)};
}
// orientation of (p, q, r) in the plane with normal n
__device__ __forceinline__ double orient(V3 n, V3 p, V3 q, V3 r) { return dot(n, cross(sub(q, p), sub(r, p))); }
__device__ __forceinline__ bool on_segment(V3 p, V3 c, V3 e) {
  return dot(sub(p, c), sub(e, c)) >= 0 && dot(sub(p, e), sub(c, e)) >= 0;
}
__device__ __forceinline__ bool segments_meet(V3 n, V3 a, V3 b, V3 c, V3 e) {
  const double d1 = orient(n, c, e, a), d2 = orient(n, c, e, b), d3 = orient(n, a, b, c), d4 = orient(n, a, b, e);
  if (((d1 > 0 && d2 < 0) || (d1 < 0 && d2 > 0)) && ((d3 > 0 && d4 < 0) || (d3 < 0 && d4 > 0))) return true;
  return (d1 == 0 && on_segment(a, c, e)) || (d2 == 0 && on_segment(b, c, e)) || (d3 == 0 && on_segment(c, a, b)) ||
         (d4 == 0 && on_segment(e, a, b));
}
__device__ __forceinline__ bool inside(V3 n, V3 p, const V3* q) {
  return orient(n, q[0], q[1], p) >= 0 && orient(n, q[1], q[2], p) >= 0 && orient(n, q[2], q[0], p) >= 0;
}
// signed volumes proportional to the barycentric coordinates where the line a->b crosses the plane of q
__device__ __forceinline__ void volumes(V3 a, V3 b, const V3* q, double v[3]) {
  const V3 d = sub(b, a);
  v[0] = dot(d, cross(sub(q[1], a), sub(q[2], a)));
  v[1] = dot(d, cross(sub(q[2], a), sub(q[0], a)));
  v[2] = dot(d, cross(sub(q[0], a), sub(q[1], a)));
}
// closed segment [a, b] meets closed triangle q (normal n != 0)
__device__ __forceinline__ bool segment_meets_triangle(V3 a, V3 b, const V3* q, V3 n) {
  const double da = dot(n, sub(a, q[0])), db = dot(n, sub(b, q[0]));
  if ((da > 0 && db > 0) || (da < 0 && db < 0)) return false;
  if (da == 0 && db == 0)
    return inside(n, a, q) || inside(n, b, q) || segments_meet(n, a, b, q[0], q[1]) ||
           segments_meet(n, a, b, q[1], q[2]) || segments_meet(n, a, b, q[2], q[0]);
  double v[3];
  volumes(a, b, q, v);
  return (v[0] >= 0 && v[1] >= 0 && v[2] >= 0) || (v[0] <= 0 && v[1] <= 0 && v[2] <= 0);
}
// s = 1: the edge of p opposite its shared vertex p[i], moved halfway to it, pierces the open interior of q
__device__ __forceinline__ bool halfway_pierces(const V3* p, int i, const V3* q, V3 n) {
  const V3 m1 = midpoint(p[i], p[(i + 1) % 3]), m2 = midpoint(p[i], p[(i + 2) % 3]);
  const double da = dot(n, sub(m1, q[0])), db = dot(n, sub(m2, q[0]));
  if (!((da > 0 && db < 0) || (da < 0 && db > 0))) return false;
  double v[3];
  volumes(m1, m2, q, v);
  return (v[0] > 0 && v[1] > 0 && v[2] > 0) || (v[0] < 0 && v[1] < 0 && v[2] < 0);
}

__device__ __forceinline__ V3 vertex(const float* P, int v) {
  return {(double)__ldg(P + 3 * (size_t)v), (double)__ldg(P + 3 * (size_t)v + 1), (double)__ldg(P + 3 * (size_t)v + 2)};
}

// the specification's decision for faces f < g of one mesh
__device__ __noinline__ bool pair_intersects(const float* __restrict__ P, const int32_t* __restrict__ F, int f, int g) {
  int a[3], b[3];
  V3 p[3], q[3];
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    a[k] = __ldg(F + 3 * f + k);
    b[k] = __ldg(F + 3 * g + k);
  }
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    p[k] = vertex(P, a[k]);
    q[k] = vertex(P, b[k]);
  }
  const V3 nf = cross(sub(p[1], p[0]), sub(p[2], p[0])), ng = cross(sub(q[1], q[0]), sub(q[2], q[0]));
  if ((nf.x == 0 && nf.y == 0 && nf.z == 0) || (ng.x == 0 && ng.y == 0 && ng.z == 0)) return false;  // zero area
  int s = 0, i = -1, j = -1;
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    const bool in_g = a[k] == b[0] || a[k] == b[1] || a[k] == b[2];
    const bool in_f = b[k] == a[0] || b[k] == a[1] || b[k] == a[2];
    s += in_g;
    if (in_g && i < 0) i = k;
    if (in_f && j < 0) j = k;
  }
  if (s == 3) return true;
  if (s == 2) return false;
  if (s == 1) return halfway_pierces(p, i, q, ng) || halfway_pierces(q, j, p, nf);
  for (int k = 0; k < 3; ++k)
    if (segment_meets_triangle(p[k], p[(k + 1) % 3], q, ng)) return true;
  for (int k = 0; k < 3; ++k)
    if (segment_meets_triangle(q[k], q[(k + 1) % 3], p, nf)) return true;
  return false;
}

struct Grid {
  float lo[3], inv;
  int dim[3];
};

__device__ __forceinline__ int cell_of(const Grid& G, int axis, float x) {
  if (G.dim[axis] == 1) return 0;
  const float t = floorf((x - G.lo[axis]) * G.inv);  // monotone in x
  return (int)fminf(fmaxf(t, 0.f), (float)(G.dim[axis] - 1));
}

// block-wide reductions (fixed order; every value involved is exact: min / max / integer sums)
template <class T, class Op>
__device__ T block_reduce(T v, Op op, T* scratch) {
  for (int o = 16; o > 0; o >>= 1) v = op(v, __shfl_xor_sync(0xffffffffu, v, o));
  __syncthreads();
  if ((threadIdx.x & 31) == 0) scratch[threadIdx.x >> 5] = v;
  __syncthreads();
  T r = scratch[0];
  for (int w = 1; w < NWARP; ++w) r = op(r, scratch[w]);
  return r;
}

__global__ void __launch_bounds__(THREADS, 1)
    selfisect_kernel(const float* __restrict__ verts, int64_t B, int V, const int32_t* __restrict__ F, int nF,
                     float4* __restrict__ ws, int32_t* __restrict__ counts, uint8_t* __restrict__ sel) {
  extern __shared__ uint4 smem_raw[];
  uint32_t* cend = reinterpret_cast<uint32_t*>(smem_raw);  // [CMAX] per-cell counts -> starts -> ends
  uint32_t* bits = cend + CMAX;                              // [FMAX/32] selected faces
  uint16_t* ent = reinterpret_cast<uint16_t*>(bits + FMAX / 32);  // [ECAP] face ids grouped by cell
  __shared__ float red_f[NWARP];
  __shared__ long long red_i[NWARP];
  __shared__ uint32_t warp_tot[NWARP];
  __shared__ Grid G;
  __shared__ int s_ncell;
  const int tid = threadIdx.x;
  const int nwords = (nF + 31) / 32;
  float4* box = ws + (size_t)blockIdx.x * 2 * nF;  // [nF] x {lo, hi}

  for (int64_t b = blockIdx.x; b < B; b += gridDim.x) {
    const float* P = verts + (size_t)b * V * 3;
    // ---- 1. face AABBs, mesh bounds, finiteness
    float mn[3] = {INFINITY, INFINITY, INFINITY}, mx[3] = {-INFINITY, -INFINITY, -INFINITY};
    int bad = 0;
    for (int f = tid; f < nF; f += THREADS) {
      float lo[3] = {INFINITY, INFINITY, INFINITY}, hi[3] = {-INFINITY, -INFINITY, -INFINITY};
      for (int k = 0; k < 3; ++k) {
        const int v = __ldg(F + 3 * f + k);
        for (int c = 0; c < 3; ++c) {
          const float x = __ldg(P + 3 * (size_t)v + c);
          bad |= !isfinite(x);
          lo[c] = fminf(lo[c], x);
          hi[c] = fmaxf(hi[c], x);
        }
      }
      box[2 * f] = make_float4(lo[0], lo[1], lo[2], 0.f);
      box[2 * f + 1] = make_float4(hi[0], hi[1], hi[2], 0.f);
      for (int c = 0; c < 3; ++c) {
        mn[c] = fminf(mn[c], lo[c]);
        mx[c] = fmaxf(mx[c], hi[c]);
      }
    }
    for (int w = tid; w < nwords; w += THREADS) bits[w] = 0u;
    auto fmin_op = [](float x, float y) { return fminf(x, y); };
    auto fmax_op = [](float x, float y) { return fmaxf(x, y); };
    auto add_op = [](long long x, long long y) { return x + y; };
    for (int c = 0; c < 3; ++c) {
      mn[c] = block_reduce(mn[c], fmin_op, red_f);
      mx[c] = block_reduce(mx[c], fmax_op, red_f);
    }
    bad = (int)block_reduce((long long)bad, add_op, red_i);
    if (bad) {  // a face references a non-finite vertex: SI is NaN, nothing is selected
      if (tid == 0) counts[b] = -1;
      if (sel)
        for (int f = tid; f < nF; f += THREADS) sel[(size_t)b * nF + f] = 0;
      __syncthreads();
      continue;
    }
    // ---- 2. uniform grid: cubic cells of side h, coarsened until the (cell, face) entries fit
    float h = 0.f;
    if (tid == 0) {
      const float e[3] = {mx[0] - mn[0], mx[1] - mn[1], mx[2] - mn[2]};
      const float emax = fmaxf(e[0], fmaxf(e[1], e[2]));
      if (isfinite(emax) && emax > 0.f) {
        const float floor_e = emax / 256.f;  // flat meshes: a zero extent must not collapse the cell volume
        h = cbrtf(fmaxf(e[0], floor_e) / CMAX * fmaxf(e[1], floor_e) * fmaxf(e[2], floor_e));
        h = fmaxf(h, emax / MAX_DIM);
      }
    }
    for (int attempt = 0;; ++attempt) {
      if (tid == 0) {
        const float e[3] = {mx[0] - mn[0], mx[1] - mn[1], mx[2] - mn[2]};
        for (;;) {
          long long n = 1;
          for (int c = 0; c < 3; ++c) {
            G.lo[c] = mn[c];
            const float d = h > 0.f ? ceilf(e[c] / h) : 1.f;
            G.dim[c] = (h > 0.f && isfinite(e[c])) ? (int)fminf(fmaxf(d, 1.f), (float)MAX_DIM) : 1;
            n *= G.dim[c];
          }
          if (n <= CMAX) {
            s_ncell = (int)n;
            break;
          }
          h *= 1.25f;
        }
        G.inv = h > 0.f ? 1.f / h : 0.f;
      }
      __syncthreads();
      const int C = s_ncell;
      for (int c = tid; c < C; c += THREADS) cend[c] = 0u;
      __syncthreads();
      long long E = 0;
      for (int f = tid; f < nF; f += THREADS) {
        const float4 lo = box[2 * f], hi = box[2 * f + 1];
        const int x0 = cell_of(G, 0, lo.x), x1 = cell_of(G, 0, hi.x), y0 = cell_of(G, 1, lo.y),
                  y1 = cell_of(G, 1, hi.y), z0 = cell_of(G, 2, lo.z), z1 = cell_of(G, 2, hi.z);
        E += (long long)(x1 - x0 + 1) * (y1 - y0 + 1) * (z1 - z0 + 1);
        for (int z = z0; z <= z1; ++z)
          for (int y = y0; y <= y1; ++y)
            for (int x = x0; x <= x1; ++x) atomicAdd(&cend[(z * G.dim[1] + y) * G.dim[0] + x], 1u);
      }
      E = block_reduce(E, add_op, red_i);
      if (E <= ECAP) break;
      // a single cell holds nF <= FMAX < ECAP entries: doubling h reaches it after a bounded number of attempts
      if (tid == 0) h = (h > 0.f && G.dim[0] * G.dim[1] * G.dim[2] > 1) ? h * 2.f : 0.f;
      __syncthreads();
    }
    const int C = s_ncell;
    // exclusive scan of the cell counts (each thread owns a contiguous run of cells)
    {
      const int per = (C + THREADS - 1) / THREADS, c0 = min(tid * per, C), c1 = min(c0 + per, C);
      uint32_t sum = 0;
      for (int c = c0; c < c1; ++c) sum += cend[c];
      uint32_t incl = sum;
      const int lane = tid & 31;
      for (int o = 1; o < 32; o <<= 1) {
        const uint32_t t = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += t;
      }
      if (lane == 31) warp_tot[tid >> 5] = incl;
      __syncthreads();
      uint32_t run = incl - sum;
      for (int w = 0; w < (tid >> 5); ++w) run += warp_tot[w];
      for (int c = c0; c < c1; ++c) {
        const uint32_t t = cend[c];
        cend[c] = run;
        run += t;
      }
    }
    __syncthreads();
    for (int f = tid; f < nF; f += THREADS) {  // fill: cend[c] advances from the start to the end of cell c
      const float4 lo = box[2 * f], hi = box[2 * f + 1];
      const int x0 = cell_of(G, 0, lo.x), x1 = cell_of(G, 0, hi.x), y0 = cell_of(G, 1, lo.y), y1 = cell_of(G, 1, hi.y),
                z0 = cell_of(G, 2, lo.z), z1 = cell_of(G, 2, hi.z);
      for (int z = z0; z <= z1; ++z)
        for (int y = y0; y <= y1; ++y)
          for (int x = x0; x <= x1; ++x) ent[atomicAdd(&cend[(z * G.dim[1] + y) * G.dim[0] + x], 1u)] = (uint16_t)f;
    }
    __syncthreads();
    // ---- 3./4. pairs within each cell, each tested in the cell of its AABB overlap's lower corner
    const int E = (int)cend[C - 1];
    for (int e = tid; e < E; e += THREADS) {
      int lo_c = 0, hi_c = C - 1;  // first cell whose end exceeds e
      while (lo_c < hi_c) {
        const int mid = (lo_c + hi_c) >> 1;
        if (cend[mid] > (uint32_t)e) hi_c = mid;
        else lo_c = mid + 1;
      }
      const int cell = lo_c, end = (int)cend[cell];
      const int cx = cell % G.dim[0], cy = (cell / G.dim[0]) % G.dim[1], cz = cell / (G.dim[0] * G.dim[1]);
      const int f = ent[e];
      const float4 flo = box[2 * f], fhi = box[2 * f + 1];
      for (int k = e + 1; k < end; ++k) {
        const int g = ent[k];
        const float4 glo = box[2 * g], ghi = box[2 * g + 1];
        if (!(flo.x <= ghi.x && glo.x <= fhi.x && flo.y <= ghi.y && glo.y <= fhi.y && flo.z <= ghi.z &&
              glo.z <= fhi.z))
          continue;
        if (cell_of(G, 0, fmaxf(flo.x, glo.x)) != cx || cell_of(G, 1, fmaxf(flo.y, glo.y)) != cy ||
            cell_of(G, 2, fmaxf(flo.z, glo.z)) != cz)
          continue;
        const uint32_t bf = 1u << (f & 31), bg = 1u << (g & 31);
        if ((bits[f >> 5] & bf) && (bits[g >> 5] & bg)) continue;  // both already selected: the outcome cannot change
        if (pair_intersects(P, F, min(f, g), max(f, g))) {
          atomicOr(&bits[f >> 5], bf);
          atomicOr(&bits[g >> 5], bg);
        }
      }
    }
    __syncthreads();
    // ---- 5. count and per-face output
    long long cnt = 0;
    for (int w = tid; w < nwords; w += THREADS) cnt += __popc(bits[w]);
    cnt = block_reduce(cnt, add_op, red_i);
    if (tid == 0) counts[b] = (int32_t)cnt;
    if (sel)
      for (int f = tid; f < nF; f += THREADS) sel[(size_t)b * nF + f] = (uint8_t)((bits[f >> 5] >> (f & 31)) & 1u);
    __syncthreads();
  }
}

}  // namespace si
}  // namespace dpb

using namespace dpb;

extern "C" int dpb_selfisect_create(dpb_selfisect_t** out, const int32_t* faces, int n_faces, int n_vertices,
                                    int device) {
  if (!out || !faces) return fail(DPB_EINVAL, "dpb_selfisect_create: null argument");
  DPB_REQUIRE(n_faces > 0 && n_vertices > 0, "dpb_selfisect_create: need n_faces > 0 and n_vertices > 0");
  DPB_REQUIRE(n_vertices <= INT32_MAX / 3, "dpb_selfisect_create: too many vertices");
  for (int64_t i = 0; i < (int64_t)n_faces * 3; ++i)
    DPB_REQUIRE(faces[i] >= 0 && faces[i] < n_vertices, "dpb_selfisect_create: face vertex id out of range");
  if (n_faces > si::FMAX)
    return fail(DPB_EUNSUPPORTED, "dpb_selfisect_create: more than 32768 faces is not supported");
  DeviceGuard guard(device);
  cudaDeviceProp prop;
  DPB_CUDA_CHECK(cudaGetDeviceProperties(&prop, device));
  DPB_CUDA_CHECK(cudaFuncSetAttribute(si::selfisect_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)si::SMEM));
  dpb_selfisect* h = new dpb_selfisect();
  h->device = device;
  h->V = n_vertices;
  h->nF = n_faces;
  h->sm_count = prop.multiProcessorCount;
  cudaError_t e = cudaMalloc((void**)&h->faces, (size_t)n_faces * 3 * sizeof(int32_t));
  if (e == cudaSuccess) e = cudaMemcpy(h->faces, faces, (size_t)n_faces * 3 * sizeof(int32_t), cudaMemcpyHostToDevice);
  if (e != cudaSuccess) {
    if (h->faces) cudaFree(h->faces);
    delete h;
    return fail(DPB_ECUDA, std::string("dpb_selfisect_create: ") + cudaGetErrorString(e));
  }
  *out = h;
  return DPB_OK;
}

extern "C" int dpb_selfisect_destroy(dpb_selfisect_t* h) {
  if (!h) return DPB_OK;
  DeviceGuard guard(h->device);
  if (h->faces) cudaFree(h->faces);
  delete h;
  return DPB_OK;
}

static int64_t selfisect_ctas(const dpb_selfisect* h, int64_t B) { return std::min<int64_t>(B, h->sm_count); }

extern "C" size_t dpb_selfisect_workspace_bytes(dpb_selfisect_t* h, int64_t B) {
  if (!h || B <= 0) return 0;
  return (size_t)selfisect_ctas(h, B) * h->nF * 2 * sizeof(float4);
}

extern "C" int dpb_selfisect_run(dpb_selfisect_t* h, const float* vertices, int64_t B, int32_t* counts,
                                 uint8_t* selection, void* ws, size_t ws_bytes, void* stream) {
  if (!h || !vertices || !counts || B <= 0) return fail(DPB_EINVAL, "dpb_selfisect_run: bad argument");
  if (!ws || ws_bytes < dpb_selfisect_workspace_bytes(h, B))
    return fail(DPB_ENOMEM, "dpb_selfisect_run: workspace smaller than dpb_selfisect_workspace_bytes");
  DeviceGuard guard(h->device);
  si::selfisect_kernel<<<(unsigned)selfisect_ctas(h, B), si::THREADS, si::SMEM, (cudaStream_t)stream>>>(
      vertices, B, h->V, h->faces, h->nF, static_cast<float4*>(ws), counts, selection);
  DPB_CUDA_CHECK(cudaGetLastError());
  return DPB_OK;
}
