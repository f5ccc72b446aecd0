// tcgen05 blend engine for LBS:  v_posed[b, v, :] = v_template[v] + shapedirs[v] . beta_b + posedirs[:, v]^T . feat_b
// as ONE tensor-core GEMM with M = vertices (TMEM lane = vertex = epilogue thread, so the stores of a pose's
// vertices are coalesced), N = 64 poses, K = shape + pose-feature components.
//
// Precision: single-pass fp16 misses the 1e-5 m bound (measured 1.6e-5 m max on the SMPL-sized synthetic model),
// so both operands are split x = x_hi + x_lo (fp16 each) and the three significant products
// hi*hi + hi*lo + lo*hi are accumulated in fp32 (measured 4e-7 m).  The split is a data layout, not extra
// storage traffic: operands are stored once as [hi | lo] along K and the MMA issuer pairs K-steps.
//
//   warp 0  TMA producer: streams blend-basis slabs [128 vertices x 64 k] (A operand, L2 resident);
//           loads the pose group's operand [64 poses x K2] once per group (B operand, SMEM resident)
//   warp 1  tcgen05.mma issuer (M=128, N=64), accumulators D_x | D_y | D_z double-buffered in TMEM
//   warp 2  TMEM allocator
//   warps 4-7 epilogue: tcgen05.ld -> + v_template -> v_posed written into the vertex buffer
// The skinning itself (blend of the per-joint transforms and their application) runs in lbs_vertex_kernel
// (lbs.cu) in place on that buffer.  Reference semantics: smplx 0.1.28 lbs() (SURVEY.md App. A.6).
#include <cudaTypedefs.h>

#include <vector>

#include <cmath>

#include "lbs.h"
#include "ptx.cuh"

namespace dpb {

int make_tmap_2d(CUtensorMap* m, CUtensorMapDataType dt, const void* ptr, uint64_t inner, uint64_t rows,
                 uint32_t box_inner, uint32_t box_rows, size_t elem_bytes);  // score_tc.cu

namespace ltc {

constexpr int TILE_V = 128;   // vertices per block (MMA M)
constexpr int BK = 64;        // fp16 per 128-byte swizzle row
constexpr int A_SLAB = TILE_V * BK * 2;  // 16 KB
constexpr int NUM_THREADS = 384;   // 4 control warps + 8 epilogue warps (two per TMEM lane quarter)
constexpr int MAX_STAGES = 8;
constexpr int PAD_POSES = 128;     // operand rows are padded to whole pose groups of either size

constexpr int XP = 4;              // poses transposed per round through the per-warp staging buffer
constexpr int XSTAGE = XP * 96;    // floats per warp: 32 vertices x (x,y,z) x XP poses

// Lane l holds (x,y,z) of vertex v0+l for XP poses; memory wants, per pose, 96 consecutive floats.  Going through a
// per-warp shared buffer turns 3 stride-12-byte stores (13 sectors each) into 3 fully coalesced 128-byte stores.
__device__ __forceinline__ void warp_store_xyz(float* stage, const float (*xyz)[3], float* const* dst, int lane,
                                               int n_floats, int n_poses) {
#pragma unroll
  for (int i = 0; i < XP; ++i) {
    stage[i * 96 + 3 * lane + 0] = xyz[i][0];
    stage[i * 96 + 3 * lane + 1] = xyz[i][1];
    stage[i * 96 + 3 * lane + 2] = xyz[i][2];
  }
  __syncwarp();
#pragma unroll
  for (int i = 0; i < XP; ++i) {
    if (i < n_poses) {
#pragma unroll
      for (int k = 0; k < 3; ++k) {
        const int f = 32 * k + lane;
        if (f < n_floats) dst[i][f] = stage[i * 96 + f];
      }
    }
  }
  __syncwarp();
}
// inverse: per pose 96 consecutive floats in memory -> (x,y,z) of this lane's vertex
__device__ __forceinline__ void warp_load_xyz(float* stage, float (*xyz)[3], const float* const* src, int lane,
                                              int n_floats, int n_poses) {
#pragma unroll
  for (int i = 0; i < XP; ++i) {
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      const int f = 32 * k + lane;
      stage[i * 96 + f] = (i < n_poses && f < n_floats) ? src[i][f] : 0.f;
    }
  }
  __syncwarp();
#pragma unroll
  for (int i = 0; i < XP; ++i) {
    xyz[i][0] = stage[i * 96 + 3 * lane + 0];
    xyz[i][1] = stage[i * 96 + 3 * lane + 1];
    xyz[i][2] = stage[i * 96 + 3 * lane + 2];
  }
  __syncwarp();
}

struct KParams {
  int V, V_pad, n_vt;       // vertices, padded vertices, vertex tiles
  int ksteps_half;          // K16 steps of the hi (= lo) part: Kp / 16
  int n_slabs;              // 64-wide slabs of [hi | lo]: 2*Kp / 64
  int stages;
  int64_t B;
  int n_groups;             // ceil(B / NP)
  const float* v_template;  // [V,3]
  float* verts;             // [B,V,3]
};

// One block = (pose group of NP poses, vertex tile): D_x | D_y | D_z [128 vertices x NP poses] in one TMEM buffer
// (3*NP columns, double-buffered), so the epilogue has a vertex's three coordinates together and can write them
// as contiguous 12-byte records (transposed per warp through shared memory into fully coalesced lines).
// HALF / NSLABS: the blend K geometry at compile time (K16 steps of the hi part, 64-wide slabs of [hi | lo]) so that the
// issuer's slab loop unrolls and every operand descriptor is base + constant; 0 = take them from KParams.
template <int NP, int HALF = 0, int NSLABS = 0>
__global__ void __launch_bounds__(NUM_THREADS, 1)
lbs_blend_tc_kernel(const __grid_constant__ KParams p, const __grid_constant__ CUtensorMap tm_dirs,
                    const __grid_constant__ CUtensorMap tm_feat) {
  constexpr int B_SLAB = NP * BK * 2;
  constexpr uint32_t IDESC = ptx::umma_idesc_f16(TILE_V, NP, 0);
  // NP = 64: two TMEM buffers (2 x 192 columns).  NP = 128: one buffer (384 columns) -- the epilogue is short
  // (coalesced staged stores) and the N = 128 MMAs are long enough for the single issuing thread to keep up.
  constexpr int NBUF = (2 * 3 * NP <= 512) ? 2 : 1;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (ptx::smem_u32(smem_raw) & 1023u)) & 1023u);
  const uint32_t smem_base = ptx::smem_u32(smem);
  const uint32_t b_base = smem_base;                              // resident pose-group operand: n_slabs slabs
  const uint32_t a_base = smem_base + p.n_slabs * B_SLAB;         // ring of A slabs
  const uint32_t bar_base = a_base + p.stages * A_SLAB;
  auto full_bar = [&](uint32_t s) { return bar_base + 8u * s; };
  auto empty_bar = [&](uint32_t s) { return bar_base + 8u * (MAX_STAGES + s); };
  auto tfull_bar = [&](uint32_t b) { return bar_base + 8u * (2 * MAX_STAGES + b); };
  auto tempty_bar = [&](uint32_t b) { return bar_base + 8u * (2 * MAX_STAGES + 2 + b); };
  const uint32_t bfull_bar = bar_base + 8u * (2 * MAX_STAGES + 4);
  const uint32_t bempty_bar = bar_base + 8u * (2 * MAX_STAGES + 5);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + p.n_slabs * B_SLAB + p.stages * A_SLAB + (2 * MAX_STAGES + 6) * 8);
  float* xstage = reinterpret_cast<float*>(smem + p.n_slabs * B_SLAB + p.stages * A_SLAB + (2 * MAX_STAGES + 6) * 8 + 16);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 0) {
    for (int s = 0; s < p.stages; ++s) {
      ptx::mbar_init(full_bar(s), 1);
      ptx::mbar_init(empty_bar(s), 1);
    }
    for (int b = 0; b < 2; ++b) {
      ptx::mbar_init(tfull_bar(b), 1);
      ptx::mbar_init(tempty_bar(b), 8);
    }
    ptx::mbar_init(bfull_bar, 1);
    ptx::mbar_init(bempty_bar, 1);
    ptx::fence_barrier_init();
  }
  if (warp == 2) ptx::tmem_alloc(ptx::smem_u32(tmem_slot), 512);
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const int half = p.ksteps_half;

  // Warps 0 and 1 run their loops warp-wide; only the async instruction is issued by the elected lane
  // (ptx::elect_one), so descriptors and coordinates stay in uniform registers.
  if (warp == 0) {
    if (lane == 0) {
      ptx::prefetch_tmap(&tm_dirs);
      ptx::prefetch_tmap(&tm_feat);
    }
    __syncwarp();
    uint32_t stage = 0, phase = 0, gph = 0;
    for (int grp = blockIdx.x; grp < p.n_groups; grp += gridDim.x) {
      ptx::mbar_wait(bempty_bar, gph ^ 1);  // previous group's MMAs are done with the resident operand
      if (ptx::elect_one()) {
        ptx::mbar_arrive_expect_tx(bfull_bar, (uint32_t)p.n_slabs * B_SLAB);
        for (int i = 0; i < p.n_slabs; ++i) ptx::tma_load_2d(b_base + i * B_SLAB, &tm_feat, bfull_bar, i * BK, grp * NP);
      }
      gph ^= 1;
      for (int vt = 0; vt < p.n_vt; ++vt)
        for (int c = 0; c < 3; ++c)
          for (int i = 0; i < p.n_slabs; ++i) {
            ptx::mbar_wait(empty_bar(stage), phase ^ 1);
            if (ptx::elect_one()) {
              ptx::mbar_arrive_expect_tx(full_bar(stage), A_SLAB);
              ptx::tma_load_2d(a_base + stage * A_SLAB, &tm_dirs, full_bar(stage), i * BK, c * p.V_pad + vt * TILE_V);
            }
            if (++stage == (uint32_t)p.stages) { stage = 0; phase ^= 1; }
          }
    }
  } else if (warp == 1) {
    uint32_t stage = 0, phase = 0, gph = 0, unit = 0, tph = 0;
    const uint64_t adesc0 = ptx::umma_desc_sw128(a_base), bdesc0 = ptx::umma_desc_sw128(b_base);
    auto bdesc = [&](int step) { return bdesc0 + (uint64_t)((step >> 2) * (B_SLAB >> 4) + 2 * (step & 3)); };
    for (int grp = blockIdx.x; grp < p.n_groups; grp += gridDim.x) {
      ptx::mbar_wait(bfull_bar, gph);
      gph ^= 1;
      ptx::tc_fence_after();
      for (int vt = 0; vt < p.n_vt; ++vt) {
        const uint32_t buf = unit % NBUF;
        ptx::mbar_wait(tempty_bar(buf), ((tph >> buf) & 1) ^ 1);
        ptx::tc_fence_after();
#pragma unroll 1
        for (int c = 0; c < 3; ++c) {
          const uint32_t taddr = tmem_base + buf * (3 * NP) + c * NP;
          const int n_slabs = NSLABS ? NSLABS : p.n_slabs;
          const int khalf = HALF ? HALF : p.ksteps_half;
          auto slab = [&](int i) {
            ptx::mbar_wait(full_bar(stage), phase);
            ptx::tc_fence_after();
            const uint64_t adesc = adesc0 + (uint64_t)(stage * (A_SLAB >> 4));
            if (ptx::elect_one()) {
#pragma unroll
              for (int j = 0; j < BK / 16; ++j) {
                const int g = i * (BK / 16) + j;  // K16 step inside [hi | lo]
                if (g < khalf) {  // basis_hi x (feat_hi + feat_lo)
                  ptx::mma_f16_ss(taddr, adesc + 2 * j, bdesc(g), IDESC, g != 0 ? 1u : 0u);
                  ptx::mma_f16_ss(taddr, adesc + 2 * j, bdesc(khalf + g), IDESC, 1u);
                } else {         // basis_lo x feat_hi
                  ptx::mma_f16_ss(taddr, adesc + 2 * j, bdesc(g - khalf), IDESC, 1u);
                }
              }
              ptx::mma_commit(empty_bar(stage));
              if (c == 2 && i == n_slabs - 1) {
                ptx::mma_commit(tfull_bar(buf));
                if (vt == p.n_vt - 1) ptx::mma_commit(bempty_bar);
              }
            }
            if (++stage == (uint32_t)p.stages) { stage = 0; phase ^= 1; }
          };
          if (NSLABS) {
#pragma unroll
            for (int i = 0; i < NSLABS; ++i) slab(i);
          } else {
            for (int i = 0; i < n_slabs; ++i) slab(i);
          }
        }
        tph ^= 1u << buf;
        ++unit;
      }
    }
  } else if (warp >= 4) {
    const int q = warp & 3;
    const int hh = (warp - 4) >> 2;   // which half of the group's poses this warp stores
    const uint32_t lane_addr = (uint32_t)(q * 32) << 16;
    const size_t pstride = (size_t)p.V * 3;
    float* stage = xstage + (warp - 4) * XSTAGE;
    uint32_t unit = 0, tph = 0;
    for (int grp = blockIdx.x; grp < p.n_groups; grp += gridDim.x) {
      const int64_t bb = (int64_t)grp * NP + hh * (NP / 2);
      for (int vt = 0; vt < p.n_vt; ++vt) {
        const int v0 = vt * TILE_V + q * 32;          // first vertex of this warp's 32-vertex segment
        const int v = v0 + lane;
        const int n_floats = max(0, min(32, p.V - v0)) * 3;
        float vt3[3] = {0.f, 0.f, 0.f};   // v_template rides in the GEMM (K slot S+P, feature 1): nothing to add here
        if (p.v_template && v < p.V) { vt3[0] = p.v_template[v * 3]; vt3[1] = p.v_template[v * 3 + 1]; vt3[2] = p.v_template[v * 3 + 2]; }
        const uint32_t buf = unit % NBUF;
        ptx::mbar_wait(tfull_bar(buf), (tph >> buf) & 1);
        ptx::tc_fence_after();
#pragma unroll 1
        for (int k = 0; k < NP / 64; ++k) {          // 32 poses per pass
          uint32_t dx[32], dy[32], dz[32];
          const uint32_t t0 = tmem_base + lane_addr + buf * (3 * NP) + hh * (NP / 2) + k * 32;
          ptx::tmem_ld_32x32(t0, dx);
          ptx::tmem_ld_32x32(t0 + NP, dy);
          ptx::tmem_ld_32x32(t0 + 2 * NP, dz);
          ptx::tmem_ld_wait();
          if (k == NP / 64 - 1) {
            ptx::tc_fence_before();
            __syncwarp();
            if (lane == 0) ptx::mbar_arrive(tempty_bar(buf));
          }
          const int64_t b32 = bb + k * 32;
#pragma unroll
          for (int i0 = 0; i0 < 32; i0 += XP) {
            float xyz[XP][3];
            float* dst[XP];
#pragma unroll
            for (int i = 0; i < XP; ++i) {
              xyz[i][0] = __uint_as_float(dx[i0 + i]) + vt3[0];
              xyz[i][1] = __uint_as_float(dy[i0 + i]) + vt3[1];
              xyz[i][2] = __uint_as_float(dz[i0 + i]) + vt3[2];
              dst[i] = p.verts + (size_t)(b32 + i0 + i) * pstride + (size_t)v0 * 3;
            }
            const int64_t left = p.B - (b32 + i0);
            warp_store_xyz(stage, xyz, dst, lane, n_floats, left >= XP ? XP : (left > 0 ? (int)left : 0));
          }
        }
        tph ^= 1u << buf;
        ++unit;
      }
    }
  }
  __syncthreads();
  if (warp == 2) {
    ptx::tc_fence_after();
    ptx::tmem_dealloc(tmem_base, 512);
  }
}

// [betas | feat] -> fp16 [hi | lo] operand rows (zero padded); one thread per (pose, k)
__global__ void lbs_featop_kernel(const float* __restrict__ betas, const float* __restrict__ feat, int S, int P, int Pf,
                                  int Kp, __half* __restrict__ op, int64_t B, int64_t B_pad) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= B_pad * Kp) return;
  const int64_t b = i / Kp;
  const int k = (int)(i % Kp);
  float x = 0.f;
  if (b < B) {
    if (k < S) x = betas[b * S + k];
    else if (k < S + Pf) x = feat[b * P + (k - S)];   // the first Pf of the P pose features vary (const-tail variants)
    else if (k == S + Pf) x = 1.0f;     // the template slot
  }
  const __half hi = __float2half_rn(x);
  const __half lo = __float2half_rn(x - __half2float(hi));
  op[b * (2 * Kp) + k] = hi;
  op[b * (2 * Kp) + Kp + k] = lo;
}


// ------------------------------------------------------------------------------------------------------------
// Skinning on tensor cores:  T[v, (b,e)] = sum_j w[v,j] A[b,j,e]  (e = 12 entries of the 3x4 transform) as a GEMM
// with M = 128 vertices (lane = vertex = epilogue thread), N = 16 poses x 12 entries, K = joints; fp16 hi/lo
// 3-product split as in the blend.  The epilogue applies T to the blended vertex (read back from the vertex
// buffer, coalesced) and stores the skinned vertex in place.  CUDA-core skinning is shared-memory bound
// (4 x 48 B of transform per (pose, vertex) through LDS); here the blend of transforms costs 6 MMAs per 2048 pairs.
constexpr int SK_POSES = 16;               // poses per MMA (N = 192)
constexpr int SK_N = SK_POSES * 12;
constexpr int SK_GROUP = 64;               // poses whose transform operand stays resident: 4 chunks of 16 when one
                                           // K slab suffices (J <= 31), 2 chunks (32 poses) for SMPL-X's two slabs
constexpr int SK_WSTAGES = 3;
constexpr uint32_t SK_IDESC = ptx::umma_idesc_f16(TILE_V, SK_N, 0);

struct SkinParams {
  int V, n_vt, jsteps;      // jsteps: K16 steps of the hi (= lo) part = Jp/16
  int n_slabs;              // 64-wide slabs of [hi | lo] = 2*Jp/64
  int chunks;               // 16-pose chunks per resident pose group
  int64_t B;
  int n_groups;
  const float* transl;      // [B,3] or nullptr
  float* verts;             // [B,V,3] in: v_posed, out: skinned vertices (forward); in: vertex cotangents (adjoint)
  // adjoint mode (gvp16 != nullptr): g_vposed = T_R^T g, scaled per pose, as the fp16 [hi | lo] operand [B, 2*Rp] of the
  // transposed blend; gextra [B,n_need,3] (optional) adds the joint cotangents scattered onto the vertices they read
  __half* gvp16;
  int Rp, n_need;
  const float* scale;       // [B]
  const float* gextra;
  const int32_t* need_index;
};

__global__ void __launch_bounds__(NUM_THREADS, 1)
lbs_skin_tc_kernel(const __grid_constant__ SkinParams p, const __grid_constant__ CUtensorMap tm_w,
                   const __grid_constant__ CUtensorMap tm_s) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (ptx::smem_u32(smem_raw) & 1023u)) & 1023u);
  const uint32_t smem_base = ptx::smem_u32(smem);
  const int chunks = p.chunks;
  const int group = chunks * SK_POSES;
  const uint32_t s_slab = SK_N * BK * 2;                           // 24 KB: one chunk, one 64-wide slab
  const uint32_t s_bytes = chunks * p.n_slabs * s_slab;            // resident transform operand of the pose group
  const uint32_t w_bytes = p.n_slabs * A_SLAB;                     // one vertex tile of weights
  const uint32_t s_base = smem_base;
  const uint32_t w_base = smem_base + s_bytes;
  const uint32_t bar_base = w_base + SK_WSTAGES * w_bytes;
  auto wfull = [&](uint32_t s) { return bar_base + 8u * s; };
  auto wempty = [&](uint32_t s) { return bar_base + 8u * (SK_WSTAGES + s); };
  auto tfull_bar = [&](uint32_t b) { return bar_base + 8u * (2 * SK_WSTAGES + b); };
  auto tempty_bar = [&](uint32_t b) { return bar_base + 8u * (2 * SK_WSTAGES + 2 + b); };
  const uint32_t sfull = bar_base + 8u * (2 * SK_WSTAGES + 4);
  const uint32_t sempty = bar_base + 8u * (2 * SK_WSTAGES + 5);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + s_bytes + SK_WSTAGES * w_bytes + (2 * SK_WSTAGES + 6) * 8);
  float* xstage = reinterpret_cast<float*>(smem + s_bytes + SK_WSTAGES * w_bytes + (2 * SK_WSTAGES + 6) * 8 + 16);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 0) {
    for (int s = 0; s < SK_WSTAGES; ++s) { ptx::mbar_init(wfull(s), 1); ptx::mbar_init(wempty(s), 1); }
    for (int b = 0; b < 2; ++b) { ptx::mbar_init(tfull_bar(b), 1); ptx::mbar_init(tempty_bar(b), 8); }
    ptx::mbar_init(sfull, 1);
    ptx::mbar_init(sempty, 1);
    ptx::fence_barrier_init();
  }
  if (warp == 2) ptx::tmem_alloc(ptx::smem_u32(tmem_slot), 512);
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp < 4) {
  ptx::setmaxnreg_dec<56>();   // warpgroup 0 (producer, issuer, two idle warps) gives registers to the epilogue
  if (warp == 0) {   // warp-wide loops, elected lane issues (see lbs_blend_tc_kernel)
    uint32_t stage = 0, phase = 0, gph = 0;
    for (int grp = blockIdx.x; grp < p.n_groups; grp += gridDim.x) {
      ptx::mbar_wait(sempty, gph ^ 1);
      if (ptx::elect_one()) {
        ptx::mbar_arrive_expect_tx(sfull, s_bytes);
        for (int c = 0; c < chunks; ++c)
          for (int i = 0; i < p.n_slabs; ++i)
            ptx::tma_load_2d(s_base + (c * p.n_slabs + i) * s_slab, &tm_s, sfull, i * BK,
                             (grp * group + c * SK_POSES) * 12);
      }
      gph ^= 1;
      for (int vt = 0; vt < p.n_vt; ++vt) {
        ptx::mbar_wait(wempty(stage), phase ^ 1);
        if (ptx::elect_one()) {
          ptx::mbar_arrive_expect_tx(wfull(stage), w_bytes);
          for (int i = 0; i < p.n_slabs; ++i)
            ptx::tma_load_2d(w_base + stage * w_bytes + i * A_SLAB, &tm_w, wfull(stage), i * BK, vt * TILE_V);
        }
        if (++stage == SK_WSTAGES) { stage = 0; phase ^= 1; }
      }
    }
  } else if (warp == 1) {
    uint32_t stage = 0, phase = 0, gph = 0, blk = 0, tph = 0;
    const int js = p.jsteps;
    for (int grp = blockIdx.x; grp < p.n_groups; grp += gridDim.x) {
      ptx::mbar_wait(sfull, gph);
      gph ^= 1;
      for (int vt = 0; vt < p.n_vt; ++vt) {
        ptx::mbar_wait(wfull(stage), phase);
        ptx::tc_fence_after();
        const uint32_t wa = w_base + stage * w_bytes;
        auto wdesc = [&](int step) { return ptx::umma_desc_sw128(wa + (step >> 2) * A_SLAB) + 2 * (step & 3); };
        for (int c = 0; c < chunks; ++c) {
          const uint32_t buf = blk & 1;
          ptx::mbar_wait(tempty_bar(buf), ((tph >> buf) & 1) ^ 1);
          ptx::tc_fence_after();
          const uint32_t taddr = tmem_base + buf * 256;
          const uint32_t sa = s_base + c * p.n_slabs * s_slab;
          auto sdesc = [&](int step) { return ptx::umma_desc_sw128(sa + (step >> 2) * s_slab) + 2 * (step & 3); };
          if (ptx::elect_one()) {
            for (int g = 0; g < js; ++g) {   // w_hi x (A_hi + A_lo), then w_lo x A_hi
              ptx::mma_f16_ss(taddr, wdesc(g), sdesc(g), SK_IDESC, g ? 1u : 0u);
              ptx::mma_f16_ss(taddr, wdesc(g), sdesc(js + g), SK_IDESC, 1u);
              ptx::mma_f16_ss(taddr, wdesc(js + g), sdesc(g), SK_IDESC, 1u);
            }
            ptx::mma_commit(tfull_bar(buf));
            if (c == chunks - 1) {
              ptx::mma_commit(wempty(stage));
              if (vt == p.n_vt - 1) ptx::mma_commit(sempty);
            }
          }
          tph ^= 1u << buf;
          ++blk;
        }
        if (++stage == SK_WSTAGES) { stage = 0; phase ^= 1; }
      }
    }
  }
  } else {
    // Epilogue: warp (q, h8) applies the blended transforms of 8 poses to its 32 vertices, in place.  The blended
    // vertices come from HBM (the blend kernel wrote 5.4 GB of them): each thread keeps the next PF blocks' 24 floats each
    // in flight while it works on the current block, otherwise the loads are latency-bound (measured: the first
    // FMUL after them held 28 % of the kernel's stall samples).
    ptx::setmaxnreg_inc<224>();
    const int q = warp & 3;
    const int h8 = (warp - 4) >> 2;   // warps 4-7: poses 0-7 of the chunk, warps 8-11: poses 8-15
    const uint32_t lane_addr = (uint32_t)(q * 32) << 16;
    const size_t pstride = (size_t)p.V * 3;
    uint32_t blk = 0, tph = 0;
    struct Blk { int grp, vt, c; };
    auto advance = [&](Blk& b) {
      if (++b.c == chunks) { b.c = 0; if (++b.vt == p.n_vt) { b.vt = 0; b.grp += (int)gridDim.x; } }
    };
    auto locate = [&](const Blk& b, bool& vok, int64_t& bb) -> float* {
      const int v = b.vt * TILE_V + q * 32 + lane;
      vok = v < p.V;
      bb = ((int64_t)b.grp * group + b.c * SK_POSES) + h8 * 8;
      return p.verts + ((size_t)(vok && bb < p.B ? bb : 0) * p.V + (vok ? v : 0)) * 3;
    };
    auto fetch = [&](const Blk& b, float (&vp)[8][3]) {
      bool vok; int64_t bb;
      const float* o = locate(b, vok, bb);
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const float* s = o + (size_t)((vok && bb + i < p.B) ? i : 0) * pstride;
        vp[i][0] = s[0]; vp[i][1] = s[1]; vp[i][2] = s[2];
      }
      if (p.gvp16 && p.gextra && vok) {   // adjoint: joint cotangents of the vertices the extra joints / landmarks read
        const int qn = p.need_index[b.vt * TILE_V + q * 32 + lane];
        if (qn >= 0) {
#pragma unroll
          for (int i = 0; i < 8; ++i)
            if (bb + i < p.B) {
              const float* ge = p.gextra + ((size_t)(bb + i) * p.n_need + qn) * 3;
              vp[i][0] += ge[0]; vp[i][1] += ge[1]; vp[i][2] += ge[2];
            }
        }
      }
    };
    constexpr int PF = 2;                 // blocks in flight beyond the current one (3 measured no faster)
    float vq[PF + 1][8][3];               // vq[0] = current block, vq[d] = d blocks ahead
    Blk cur{(int)blockIdx.x, 0, 0};
    Blk ahead = cur;                      // the block PF - 1 ahead of `cur` (fetched before the loop)
    if (cur.grp < p.n_groups) fetch(cur, vq[0]);
#pragma unroll
    for (int d = 1; d < PF; ++d) {
      advance(ahead);
      if (ahead.grp < p.n_groups) fetch(ahead, vq[d]);
    }
    while (cur.grp < p.n_groups) {
      advance(ahead);
      if (ahead.grp < p.n_groups) fetch(ahead, vq[PF]);
      float (&vp)[8][3] = vq[0];
      bool vok; int64_t bb;
      float* o = locate(cur, vok, bb);
      const bool full = vok && (bb + 8 <= p.B);
      const uint32_t buf = blk & 1;
      ptx::mbar_wait(tfull_bar(buf), (tph >> buf) & 1);
      ptx::tc_fence_after();
      uint32_t t[96];
      const uint32_t t0 = tmem_base + lane_addr + buf * 256 + h8 * 96;
      ptx::tmem_ld_32x32(t0, t);
      ptx::tmem_ld_32x32(t0 + 32, t + 32);
      ptx::tmem_ld_32x32(t0 + 64, t + 64);
      ptx::tmem_ld_wait();
      ptx::tc_fence_before();
      __syncwarp();
      if (lane == 0) ptx::mbar_arrive(tempty_bar(buf));
      if (p.gvp16) {
        // skinning adjoint: g_vposed = T_R^T g, scaled into fp16's normal range, fp16 [hi | lo] halves of row (pose)
        const int v = cur.vt * TILE_V + q * 32 + lane;
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          if (full || (vok && bb + i < p.B)) {
            const float* T = reinterpret_cast<const float*>(t) + i * 12;
            const float sc = p.scale[bb + i];
            const float gx = vp[i][0] * sc, gy = vp[i][1] * sc, gz = vp[i][2] * sc;
            const float o3[3] = {T[0] * gx + T[3] * gy + T[6] * gz, T[1] * gx + T[4] * gy + T[7] * gz,
                                 T[2] * gx + T[5] * gy + T[8] * gz};
            __half* oh = p.gvp16 + (size_t)(bb + i) * 2 * p.Rp + (size_t)v * 3;
#pragma unroll
            for (int c = 0; c < 3; ++c) {
              const __half hi = __float2half_rn(o3[c]);
              oh[c] = hi;
              oh[p.Rp + c] = __float2half_rn(o3[c] - __half2float(hi));
            }
          }
        }
      } else
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        if (full || (vok && bb + i < p.B)) {
          const float* T = reinterpret_cast<const float*>(t) + i * 12;
          const float x = vp[i][0], y = vp[i][1], z = vp[i][2];
          float tx = 0.f, ty = 0.f, tz = 0.f;
          if (p.transl) {
            const float* tr = p.transl + (bb + i) * 3;
            tx = tr[0]; ty = tr[1]; tz = tr[2];
          }
          float* w = o + (size_t)i * pstride;
          w[0] = T[0] * x + T[1] * y + T[2] * z + T[9] + tx;
          w[1] = T[3] * x + T[4] * y + T[5] * z + T[10] + ty;
          w[2] = T[6] * x + T[7] * y + T[8] * z + T[11] + tz;
        }
      }
#pragma unroll
      for (int d = 0; d < PF; ++d)
#pragma unroll
        for (int i = 0; i < 8; ++i)
#pragma unroll
          for (int k = 0; k < 3; ++k) vq[d][i][k] = vq[d + 1][i][k];
      tph ^= 1u << buf;
      ++blk;
      advance(cur);
    }
  }
  __syncthreads();
  if (warp == 2) {
    ptx::tc_fence_after();
    ptx::tmem_dealloc(tmem_base, 512);
  }
}

// per-pose transforms A[b,j,12] -> operand rows (b*12 + e) = [A[b,:,e] hi (Jp) | lo (Jp)] fp16
// If J < Jp the spare joint slot J carries the translation: its weight is 1 for every vertex (lbs_tc_prepare) and
// its "transform" is [0 | transl], so T_t already includes + transl and the epilogue does not add it.
// One warp per pose: the pose's transforms A[b] (J x 12 floats, contiguous) are read once, coalesced; the 12 operand rows
// [hi | lo] (12 x 2 Jp halves, contiguous in `op`) are assembled in shared memory and leave as 16-byte vectors.  (The
// thread-per-element version issued two 2-byte stores per element and re-read every sector of A twelve times.)
__global__ void __launch_bounds__(128) lbs_skinop_kernel(const float* __restrict__ A, const float* __restrict__ transl, int J,
                                                         int Jp, __half* __restrict__ op, int64_t B, int64_t B_pad) {
  __shared__ __align__(16) __half stage[4][12 * 128];      // 2 * Jp <= 128
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int64_t b = (int64_t)blockIdx.x * 4 + w;
  if (b >= B_pad) return;                                   // warp-uniform
  __half* ss = stage[w];
  const int n_el = 12 * Jp;
  if (b < B) {
    for (int i = lane; i < 12 * Jp; i += 32) {              // zero-fill, then the valid entries below overwrite
      const int e = i / Jp, j = i - e * Jp;
      float x = 0.f;
      if (j == J && e >= 9 && transl) x = transl[b * 3 + (e - 9)];
      const __half hi = __float2half_rn(x);
      ss[e * 2 * Jp + j] = hi;
      ss[e * 2 * Jp + Jp + j] = __float2half_rn(x - __half2float(hi));
    }
    __syncwarp();
    const float* a = A + b * J * 12;
    for (int i = lane; i < J * 12; i += 32) {               // contiguous read of the pose's transforms
      const int j = i / 12, e = i - j * 12;
      const float x = a[i];
      const __half hi = __float2half_rn(x);
      ss[e * 2 * Jp + j] = hi;
      ss[e * 2 * Jp + Jp + j] = __float2half_rn(x - __half2float(hi));
    }
  } else {
    for (int i = lane; i < 2 * n_el; i += 32) ss[i] = __float2half_rn(0.f);
  }
  __syncwarp();
  const uint4* src = reinterpret_cast<const uint4*>(ss);
  uint4* dst = reinterpret_cast<uint4*>(op + (size_t)b * 12 * 2 * Jp);
  for (int i = lane; i < 3 * Jp; i += 32) dst[i] = src[i];  // 12 rows x 2 Jp halves = 3 Jp vectors of 16 bytes
}

}  // namespace ltc

int lbs_tc_prepare(dpb_lbs* h, const dpb_body_tensors* m) {
  h->tc_ready = false;
  const int V = h->V, S = h->S, P = h->P;
  const int Kp = (S + P + 1 + 31) / 32 * 32;   // hi (= lo) width incl. the template slot: multiple of 32 so that [hi | lo] is whole 64-wide slabs
  const int K2 = 2 * Kp;
  const int V_pad = (V + 2 * ltc::TILE_V - 1) / (2 * ltc::TILE_V) * (2 * ltc::TILE_V);   // whole tile PAIRS (CTA-pair kernels)
  const int n_slabs = K2 / ltc::BK;
  if ((size_t)n_slabs * (64 * ltc::BK * 2) + 2 * ltc::A_SLAB + 2048 > 232448) return DPB_OK;  // too wide: fp32 engine only
  // blend basis, vertex-major per coordinate: row (c*V_pad + v) = [shapedirs[v,c,:] | posedirs[:,3v+c]] as [hi | lo]
  std::vector<__half> basis((size_t)3 * V_pad * K2, __float2half_rn(0.f));
  for (int c = 0; c < 3; ++c)
    for (int v = 0; v < V; ++v) {
      __half* row = basis.data() + ((size_t)c * V_pad + v) * K2;
      for (int k = 0; k < S + P; ++k) {
        const float x = k < S ? m->shapedirs[((size_t)v * 3 + c) * S + k]
                              : m->posedirs[(size_t)(k - S) * V * 3 + (size_t)v * 3 + c];
        const __half hi = __float2half_rn(x);
        row[k] = hi;
        row[Kp + k] = __float2half_rn(x - __half2float(hi));
      }
      {   // template slot (the pose operand carries a 1 there)
        const float x = m->v_template[(size_t)v * 3 + c];
        const __half hi = __float2half_rn(x);
        row[S + P] = hi;
        row[Kp + S + P] = __float2half_rn(x - __half2float(hi));
      }
    }
  DPB_CUDA_CHECK(cudaMalloc((void**)&h->dirs16, basis.size() * sizeof(__half)));
  DPB_CUDA_CHECK(cudaMemcpy(h->dirs16, basis.data(), basis.size() * sizeof(__half), cudaMemcpyHostToDevice));
  int rc = make_tmap_2d(&h->tm_dirs, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, h->dirs16, K2, (uint64_t)3 * V_pad, ltc::BK,
                        ltc::TILE_V, 2);
  if (rc != DPB_OK) return rc;
  h->kext = K2;
  h->n_cols_pad = V_pad;
  // skinning-weight operand: row v = [w[v,:] hi (Jp) | lo (Jp)], Jp = joints padded to 32
  const int J = h->J, Jp = (J + 31) / 32 * 32;
  std::vector<__half> wop((size_t)V_pad * 2 * Jp, __float2half_rn(0.f));
  for (int v = 0; v < V; ++v)
    for (int j = 0; j < J; ++j) {
      const float x = m->lbs_weights[(size_t)v * J + j];
      const __half hi = __float2half_rn(x);
      wop[(size_t)v * 2 * Jp + j] = hi;
      wop[(size_t)v * 2 * Jp + Jp + j] = __float2half_rn(x - __half2float(hi));
    }
  if (J < Jp)
    for (int v = 0; v < V; ++v) wop[(size_t)v * 2 * Jp + J] = __float2half_rn(1.0f);   // translation slot
  DPB_CUDA_CHECK(cudaMalloc((void**)&h->wop16, wop.size() * sizeof(__half)));
  DPB_CUDA_CHECK(cudaMemcpy(h->wop16, wop.data(), wop.size() * sizeof(__half), cudaMemcpyHostToDevice));
  rc = make_tmap_2d(&h->tm_wop, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, h->wop16, 2 * Jp, (uint64_t)V_pad, ltc::BK,
                    ltc::TILE_V, 2);
  if (rc != DPB_OK) return rc;
  h->jp = Jp;
  h->tc_ready = true;
  return DPB_OK;
}

// Const-tail variant: joints n_var..J-1 always carry `tail_pose` (HOST [(J-n_var)*3]); their pose-blend contribution
// posedirs[tail features]^T . (R(tail) - I) is a constant per vertex and moves into the template slot.
int lbs_tc_make_tail(dpb_lbs* h, int n_var, const float* tail_pose) {
  const int V = h->V, S = h->S, P = h->P, J = h->J, V_pad = h->n_cols_pad;
  if (h->tailv.dirs16) { cudaFree(h->tailv.dirs16); h->tailv = LbsVariant(); }
  if (!h->tc_ready) return DPB_OK;
  const int Pf = 9 * (n_var - 1);
  const int Kp = (S + Pf + 1 + 31) / 32 * 32, K2 = 2 * Kp;
  std::vector<float> sd((size_t)V * 3 * S), pd((size_t)P * V * 3), vt((size_t)V * 3);
  DPB_CUDA_CHECK(cudaMemcpy(sd.data(), h->shapedirs, sd.size() * 4, cudaMemcpyDeviceToHost));
  DPB_CUDA_CHECK(cudaMemcpy(pd.data(), h->posedirs, pd.size() * 4, cudaMemcpyDeviceToHost));
  DPB_CUDA_CHECK(cudaMemcpy(vt.data(), h->v_template, vt.size() * 4, cudaMemcpyDeviceToHost));
  // (R - I) of the tail joints with smplx's Rodrigues (angle = ||r + 1e-8||), in double
  std::vector<double> tf((size_t)(J - n_var) * 9);
  for (int j = n_var; j < J; ++j) {
    const float* r = tail_pose + (size_t)(j - n_var) * 3;
    const double bx = (double)r[0] + 1e-8, by = (double)r[1] + 1e-8, bz = (double)r[2] + 1e-8;
    const double ang = std::sqrt(bx * bx + by * by + bz * bz);
    const double x = r[0] / ang, y = r[1] / ang, z = r[2] / ang, s = std::sin(ang), oc = 1.0 - std::cos(ang);
    const double R[9] = {1 + oc * (-(z * z) - y * y), s * -z + oc * x * y, s * y + oc * x * z,
                         s * z + oc * x * y, 1 + oc * (-(z * z) - x * x), s * -x + oc * y * z,
                         s * -y + oc * x * z, s * x + oc * y * z, 1 + oc * (-(y * y) - x * x)};
    for (int e = 0; e < 9; ++e) tf[(size_t)(j - n_var) * 9 + e] = R[e] - ((e == 0 || e == 4 || e == 8) ? 1.0 : 0.0);
  }
  std::vector<double> tmpl((size_t)V * 3);
  for (size_t i = 0; i < tmpl.size(); ++i) tmpl[i] = vt[i];
  for (int k = Pf; k < P; ++k) {
    const double f = tf[(size_t)(k - Pf)];
    if (f == 0.0) continue;
    const float* row = pd.data() + (size_t)k * V * 3;
    for (size_t i = 0; i < tmpl.size(); ++i) tmpl[i] += f * row[i];
  }
  std::vector<__half> basis((size_t)3 * V_pad * K2, __float2half_rn(0.f));
  auto put = [&](__half* row, int k, float x) {
    const __half hi = __float2half_rn(x);
    row[k] = hi;
    row[Kp + k] = __float2half_rn(x - __half2float(hi));
  };
  for (int c = 0; c < 3; ++c)
    for (int v = 0; v < V; ++v) {
      __half* row = basis.data() + ((size_t)c * V_pad + v) * K2;
      for (int k = 0; k < S; ++k) put(row, k, sd[((size_t)v * 3 + c) * S + k]);
      for (int k = 0; k < Pf; ++k) put(row, S + k, pd[(size_t)k * V * 3 + (size_t)v * 3 + c]);
      put(row, S + Pf, (float)tmpl[(size_t)v * 3 + c]);
    }
  LbsVariant t;
  t.n_var = n_var; t.p_feat = Pf; t.kext = K2;
  DPB_CUDA_CHECK(cudaMalloc((void**)&t.dirs16, basis.size() * sizeof(__half)));
  DPB_CUDA_CHECK(cudaMemcpy(t.dirs16, basis.data(), basis.size() * sizeof(__half), cudaMemcpyHostToDevice));
  int rc = make_tmap_2d(&t.tm_dirs, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, t.dirs16, K2, (uint64_t)3 * V_pad, ltc::BK,
                        ltc::TILE_V, 2);
  if (rc != DPB_OK) { cudaFree(t.dirs16); return rc; }
  h->tailv = t;
  return DPB_OK;
}

void lbs_tc_release(dpb_lbs* h) {
  if (h->tailv.dirs16) cudaFree(h->tailv.dirs16);
  h->tailv = LbsVariant();
  if (h->dirs16) cudaFree(h->dirs16);
  if (h->wop16) cudaFree(h->wop16);
  h->dirs16 = nullptr;
  h->wop16 = nullptr;
  h->tc_ready = false;
}

size_t lbs_tc_ws_bytes(const dpb_lbs* h, int64_t B) {
  if (!h->tc_ready) return 0;
  const int64_t B_pad = (B + ltc::PAD_POSES - 1) / ltc::PAD_POSES * ltc::PAD_POSES;
  return align_up((size_t)B_pad * h->kext * sizeof(__half), 1024) +
         align_up((size_t)B_pad * 12 * 2 * h->jp * sizeof(__half), 1024) + 1024;
}

bool lbs_tc_skin_fits(const dpb_lbs* h) {
  const int n_slabs = 2 * h->jp / ltc::BK;
  const int chunks = n_slabs == 1 ? 4 : 2;
  const size_t smem = (size_t)chunks * n_slabs * ltc::SK_N * ltc::BK * 2 +
                      (size_t)ltc::SK_WSTAGES * n_slabs * ltc::A_SLAB + 8 * ltc::XSTAGE * 4 + 2048;
  return h->tc_ready && h->J < h->jp && smem <= 232448;
}

// skins verts[B,V,3] (holding v_posed) in place with the per-pose transforms A[B,J,12]
int lbs_tc_skin(dpb_lbs* h, const float* A, const float* transl, __half* skinop, float* verts, int64_t B,
                cudaStream_t st) {
  const int Jp = h->jp;
  const int64_t B_pad = (B + ltc::SK_GROUP - 1) / ltc::SK_GROUP * ltc::SK_GROUP;   // operand rows (64 | 32 both divide)
  {
    const int64_t n = B_pad * 12 * Jp;
    ltc::lbs_skinop_kernel<<<(unsigned)((B_pad + 3) / 4), 128, 0, st>>>(A, transl, h->J, Jp, skinop, B, B_pad);
    DPB_CUDA_CHECK(cudaGetLastError());
  }
  CUtensorMap tm_s;
  int rc = make_tmap_2d(&tm_s, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, skinop, 2 * Jp, (uint64_t)B_pad * 12, ltc::BK, ltc::SK_N, 2);
  if (rc != DPB_OK) return rc;
  ltc::SkinParams p{};
  p.V = h->V;
  p.n_vt = h->n_cols_pad / ltc::TILE_V;
  p.jsteps = Jp / 16;
  p.n_slabs = 2 * Jp / ltc::BK;
  p.B = B;
  p.chunks = p.n_slabs == 1 ? 4 : 2;
  p.n_groups = (int)(B_pad / (p.chunks * ltc::SK_POSES));
  p.transl = h->J < Jp ? nullptr : transl;   // folded into the GEMM through the spare joint slot when there is one
  p.verts = verts;
  const size_t smem = (size_t)p.chunks * p.n_slabs * ltc::SK_N * ltc::BK * 2 +
                      (size_t)ltc::SK_WSTAGES * p.n_slabs * ltc::A_SLAB + (2 * ltc::SK_WSTAGES + 6) * 8 + 16 +
                      8 * ltc::XSTAGE * 4 + 1024;
  if (smem > 232448) return fail(DPB_EUNSUPPORTED, "lbs tc skin: transform operand does not fit shared memory");
  DPB_CUDA_CHECK(cudaFuncSetAttribute(ltc::lbs_skin_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  const int grid = p.n_groups < h->sm_count ? p.n_groups : h->sm_count;
  ltc::lbs_skin_tc_kernel<<<grid, ltc::NUM_THREADS, smem, st>>>(p, h->tm_wop, tm_s);
  DPB_CUDA_CHECK(cudaGetLastError());
  return DPB_OK;
}


// skinning adjoint, vertex side: gvp16 [B, 2*Rp] = fp16 [hi | lo] of scale[b] * T_R^T (g_verts + gextra) with the blended
// transforms T = W A recomputed on the tensor cores (the forward's kernel with an adjoint epilogue)
int lbs_tc_skin_adjoint(dpb_lbs* h, const float* A, __half* skinop, const float* g_verts, const float* gextra,
                        bool have_extra, const float* scale, __half* gvp16, int64_t B, cudaStream_t st) {
  const int Jp = h->jp;
  const int64_t B_pad = (B + ltc::SK_GROUP - 1) / ltc::SK_GROUP * ltc::SK_GROUP;
  {
    const int64_t n = B_pad * 12 * Jp;
    ltc::lbs_skinop_kernel<<<(unsigned)((B_pad + 3) / 4), 128, 0, st>>>(A, nullptr, h->J, Jp, skinop, B, B_pad);
    DPB_CUDA_CHECK(cudaGetLastError());
  }
  CUtensorMap tm_s;
  int rc = make_tmap_2d(&tm_s, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, skinop, 2 * Jp, (uint64_t)B_pad * 12, ltc::BK, ltc::SK_N, 2);
  if (rc != DPB_OK) return rc;
  ltc::SkinParams p{};
  p.V = h->V;
  p.n_vt = h->n_cols_pad / ltc::TILE_V;
  p.jsteps = Jp / 16;
  p.n_slabs = 2 * Jp / ltc::BK;
  p.B = B;
  p.chunks = p.n_slabs == 1 ? 4 : 2;
  p.n_groups = (int)(B_pad / (p.chunks * ltc::SK_POSES));
  p.transl = nullptr;
  p.verts = const_cast<float*>(g_verts);   // read-only in adjoint mode
  p.gvp16 = gvp16;
  p.Rp = h->bt_rp;
  p.n_need = h->n_need;
  p.scale = scale;
  p.gextra = have_extra ? gextra : nullptr;
  p.need_index = h->need_index;
  const size_t smem = (size_t)p.chunks * p.n_slabs * ltc::SK_N * ltc::BK * 2 +
                      (size_t)ltc::SK_WSTAGES * p.n_slabs * ltc::A_SLAB + (2 * ltc::SK_WSTAGES + 6) * 8 + 16 +
                      8 * ltc::XSTAGE * 4 + 1024;
  if (smem > 232448) return fail(DPB_EUNSUPPORTED, "lbs tc skin adjoint: transform operand does not fit shared memory");
  DPB_CUDA_CHECK(cudaFuncSetAttribute(ltc::lbs_skin_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  const int grid = p.n_groups < h->sm_count ? p.n_groups : h->sm_count;
  ltc::lbs_skin_tc_kernel<<<grid, ltc::NUM_THREADS, smem, st>>>(p, h->tm_wop, tm_s);
  DPB_CUDA_CHECK(cudaGetLastError());
  return DPB_OK;
}

// writes v_posed (template + shape blend + pose blend) into verts[B,V,3]
int lbs_tc_blend(dpb_lbs* h, const LbsVariant& var, const float* betas, const float* feat, __half* featop, float* verts,
                 int64_t B, cudaStream_t st) {
  const int K2 = var.kext, Kp = K2 / 2;
  const int64_t B_pad = (B + ltc::PAD_POSES - 1) / ltc::PAD_POSES * ltc::PAD_POSES;
  {
    const int64_t n = B_pad * Kp;
    ltc::lbs_featop_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(betas, feat, h->S, h->P, var.p_feat, Kp, featop, B, B_pad);
    DPB_CUDA_CHECK(cudaGetLastError());
  }
  const int n_slabs = K2 / ltc::BK;
  const size_t bars = (2 * ltc::MAX_STAGES + 6) * 8 + 16 + 8 * ltc::XSTAGE * 4 + 1024;
  // 128-pose groups when the group's operand leaves room for >= 4 ring stages (SMPL), else 64 (SMPL-X)
  const int np = ((size_t)n_slabs * 128 * ltc::BK * 2 + 4 * ltc::A_SLAB + bars <= 232448) ? 128 : 64;
  CUtensorMap tm_feat;
  int rc = make_tmap_2d(&tm_feat, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, featop, K2, (uint64_t)B_pad, ltc::BK, np, 2);
  if (rc != DPB_OK) return rc;
  ltc::KParams p{};
  p.V = h->V;
  p.V_pad = h->n_cols_pad;
  p.n_vt = h->n_cols_pad / ltc::TILE_V;
  p.ksteps_half = Kp / 16;
  p.n_slabs = n_slabs;
  p.B = B;
  p.n_groups = (int)((B + np - 1) / np);
  p.v_template = nullptr;   // folded into the GEMM
  p.verts = verts;
  const size_t fixed = (size_t)n_slabs * np * ltc::BK * 2 + bars;
  int stages = (int)((232448 - fixed) / ltc::A_SLAB);
  if (stages > ltc::MAX_STAGES) stages = ltc::MAX_STAGES;
  if (stages < 2) return fail(DPB_EUNSUPPORTED, "lbs tc: not enough shared memory for the operand ring");
  p.stages = stages;
  const size_t smem = fixed + (size_t)stages * ltc::A_SLAB;
  const int grid = p.n_groups < h->sm_count ? p.n_groups : h->sm_count;
  // instantiations with compile-time K geometry for the two body models, run-time geometry otherwise
  void (*kern)(ltc::KParams, CUtensorMap, CUtensorMap) = nullptr;
  if (np == 128) kern = (K2 == 448) ? ltc::lbs_blend_tc_kernel<128, 14, 7> : ltc::lbs_blend_tc_kernel<128>;
  else kern = (K2 == 1024) ? ltc::lbs_blend_tc_kernel<64, 32, 16> : ltc::lbs_blend_tc_kernel<64>;
  DPB_CUDA_CHECK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  kern<<<grid, ltc::NUM_THREADS, smem, st>>>(p, var.tm_dirs, tm_feat);
  DPB_CUDA_CHECK(cudaGetLastError());
  return DPB_OK;
}

}  // namespace dpb
