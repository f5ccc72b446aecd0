// tcgen05 engine of the score network: ONE persistent, warp-specialised kernel that runs every
// layer of every sampler step for a 128-row tile of poses.
//
//   warp 0      TMA producer, weight (B-operand) tiles   [N x 64] fp16, SWIZZLE_128B
//   warp 1      tcgen05.mma issuer (one thread), fp32 accumulators in TMEM (2 x 256 columns)
//   warp 2      TMEM allocator, then TMA producer of activation (A-operand) tiles [128 x 64]
//   warps 4-11  epilogue: tcgen05.ld 32x32b -> +time bias -> GroupNorm(32 ch, thread-local stats)
//               -> SiLU (-> +residual) -> fp16 -> per-CTA activation scratch (L2 resident);
//               last layer: Euler-Maruyama update / imputation / Philox noise (sampler),
//               scaled output (forward) or loss + closed-form gradient (prior loss)
//
// Numerics: fp16 operands with fp32 accumulation for the four 1024x1024 layers and post_dense;
// the 63-wide input layer uses a bf16 hi/lo split of x and W_pre expressed as a K-extension
// ([x_hi | x_lo | x_hi] . [W_hi | W_hi | W_lo]^T, K = 192) so it keeps ~16 mantissa bits and the
// fp32 range of x.  Math follows ScoreModelFC.forward (reference model.py:141-196), the EM update
// sampling.py:182-188 and imputation :413-422; identical formulas / Philox addressing as sampler.cu.
#include <cudaTypedefs.h>

#include <cstdlib>
#include <vector>

#include "ptx.cuh"
#include "score.h"

namespace dpb {
constexpr int PC_MAX_STEPS = 4096;   // sampler steps the fused predictor-corrector mode keeps norm sums for

namespace tc {

constexpr int TILE_M = 128;
constexpr int BLOCK_K = 64;  // 64 x 2 B = one 128-byte swizzle row
constexpr int CHUNK_N = 256;
constexpr bool TWO_SM = true;   // CTA pair: one tcgen05.mma.cta_group::2 (M = 256) per weight tile; each CTA keeps
                                // its own 128 rows of A and HALF of the weight tile, so weight ingest per CTA halves
#ifdef DPB_TC_STAGES   // timing experiments: ring depth (with DPB_TC_TINY_STG the staging area shrinks so that six stages fit;
constexpr int STAGES = DPB_TC_STAGES;   // only the operand-pipeline-only debug mode is meaningful then)
#else
constexpr int STAGES = TWO_SM ? 4 : 3;   // measured: the operand pipeline alone runs equally fast with 4, 5 or 6 stages
#endif   // the operand ring is latency bound: utilisation ~ STAGES*512/(L+512), L ~ 2.2k cycles
constexpr int NSUB = 1;      // row tiles in flight per CTA: one tile's epilogue overlaps the other tile's MMAs
constexpr int CLUSTER = 2;   // CTAs (different row tiles) that share every weight tile through TMA multicast
constexpr int A_BYTES = TILE_M * BLOCK_K * 2;   // 16 KB
constexpr int B_BYTES = CHUNK_N * BLOCK_K * 2 / (TWO_SM ? 2 : 1);  // this CTA's share of the weight tile
constexpr int STAGE_BYTES = A_BYTES + B_BYTES;
constexpr int NUM_THREADS = 640;   // 4 single-lane role warps + 16 epilogue warps
constexpr int EPI_THREADS = 512;
constexpr int ROLE_REGS = 32;      // setmaxnreg: 640 threads start at 96 registers; the role warpgroup gives, the
constexpr int EPI_REGS = 112;      // epilogue warpgroups take ((96 - 32) * 128 >= (112 - 96) * 512)
static_assert(2 * H / 4 == EPI_THREADS, "parameter staging assumes one float4 of gamma|beta per epilogue thread");
constexpr int PAR_BYTES = 2 * 3 * H * 4;   // [time bias | gamma | beta] x 1024 floats, double-buffered across layers
constexpr int STG_BYTES = TILE_M * 128;          // one [128 rows x 64 fp16] SWIZZLE_128B box of outgoing activations
constexpr int STG_BUFS = 2;                      // staging boxes per column half: box (hf, gp) of a chunk has its own buffer, so
                                                 // the LAST chunk of a layer stays in shared memory and feeds the next layer's
                                                 // first chunk directly (DIRECT_K0..), without the L2 round trip
constexpr int DIRECT_K0 = H / BLOCK_K - CHUNK_N / BLOCK_K;   // first K slab that is a column box of the previous layer's last chunk
static_assert(NSUB == 1 && STG_BUFS == 2 && CHUNK_N / BLOCK_K == 4 && STAGES >= 2, "the direct path assumes four boxes per chunk, one tile per CTA");
#ifdef DPB_TC_TINY_STG
constexpr int STG_TOTAL = 1024;
#else
constexpr int STG_TOTAL = 2 * STG_BUFS * STG_BYTES;
#endif
constexpr int NUM_BARS = 2 * STAGES + 4 + NSUB * 5 + 8;  // full, empty, tfull[2], tempty[2], xa, act[4], sfull[2][2], sempty[2][2]
constexpr int OFF_PAR = STAGES * STAGE_BYTES;
constexpr int OFF_STG = OFF_PAR + PAR_BYTES;     // 1024-aligned
constexpr int OFF_BAR = OFF_STG + STG_TOTAL;
constexpr int OFF_POSTB = (OFF_BAR + NUM_BARS * 8 + 16 + 15) / 16 * 16;   // post_dense bias (DP floats)
static_assert(OFF_POSTB % 16 == 0, "post_b is read with 128-bit loads");
static_assert(OFF_STG % 1024 == 0, "staging boxes must be 1024-byte aligned for SWIZZLE_128B");
constexpr int MMA_M = TWO_SM ? 2 * TILE_M : TILE_M;
constexpr uint32_t IDESC_F16_256 = ptx::umma_idesc_f16(MMA_M, CHUNK_N, 0);
constexpr uint32_t IDESC_BF16_256 = ptx::umma_idesc_f16(MMA_M, CHUNK_N, 1);
static_assert(!TWO_SM || CLUSTER == 2, "cta_group::2 needs clusters of exactly two CTAs");

// What depends on the pose width: the kernel is instantiated for the padded width PDP = 64 (63-D axis-angle network)
// and PDP = 128 (126-D rot6d network).
template <int PDP>
struct Width {
  static constexpr int D = pose_dim_of(PDP);
  static constexpr int XA_SLABS = PDP / BLOCK_K;   // 64-column slabs of x_hi (and of x_lo): 1 or 2
  static constexpr int XA_K = 3 * PDP;             // input-layer K-extension [x_hi | x_lo | x_hi]: 192 or 384
  static constexpr int TCOLS = PDP / 4;            // pose columns per epilogue thread in the prologue / tail (4 warps per row quarter)
  static constexpr int POST_B_BYTES = PDP * BLOCK_K * 2 / (TWO_SM ? 2 : 1);   // this CTA's share of a post_dense tile (N = PDP)
  static constexpr int OFF_PCROW = OFF_POSTB + PDP * 4;   // predictor-corrector mode: per-row squared norms [128][2]
  static constexpr int SMEM_BYTES = OFF_PCROW + TILE_M * 2 * 4 + 1024;   // + alignment slack
  static constexpr uint32_t IDESC_POST = ptx::umma_idesc_f16(MMA_M, PDP, 0);
  static_assert(SMEM_BYTES <= 232448, "exceeds the 227 KB per-CTA shared memory limit");
  // x occupies the A halves of the first 2 XA_SLABS ring stages during the input layer
  static_assert(2 * XA_SLABS <= STAGES, "the input-layer operand needs 2 * XA_SLABS ring stages");
  static_assert(TCOLS == 16 || TCOLS == 32, "the tail reads TCOLS accumulator columns with one tcgen05.ld");
};

struct KParams {
  int mode, n_steps, impute, noise_k, n_tiles;
  int debug;  // timing experiments only (DPB_TC_DEBUG): 1 = skip hidden-layer epilogue math, 2 = skip MMAs,
              // 4 / 8 = skip the activation / weight TMA loads, 16 = skip the activation TMA stores,
              // 64 = operand pipeline only (no epilogue, no activation dependencies; results are garbage),
              // 128 / 256 / 512 = skip the hidden layers' TMEM loads / staging stores / residual loads
  long long B;
  const float* x_in;
  float* x_io;
  const float* table;
  const float* coef;
  const float* gn;
  const float* post_b;
  const float* row_scale;
  float scale;
  float* out;
  const float* obs;
  const float* mask;
  const float* noise;
  unsigned long long seed, step_offset;
  float* traj;
  float* x_mean;
  float alpha, sd, inv_sigma_std, inv_div, wgt;
  const float* z;
  float* loss_out;
  float* grad_out;
  float* row_loss;
  __half* act_h;
  __half* act_t;
  int* flags;   // one hand-off flag per CTA (zeroed before the launch), see SegIter
  // predictor-corrector mode (Langevin corrector, sampling.py:282-302): n_steps counts SUB-steps, even = corrector, odd =
  // predictor of step (sub >> 1); every CTA owns one tile for the whole run (lock step) and the batch-global norms go
  // through pc_sums[step][2] and a counter barrier over the grid.  coef columns 5 / 6 = score scale / alpha of the step.
  int pc;
  float snr;
  float* pc_sums;
  int* pc_counter;
};

// ---- work distribution.  A "unit" is CLUSTER consecutive row tiles (one per CTA of a cluster) and a "chain" is
// one unit's n_steps sampler steps, which must run in order.  The chains are laid end to end and cut into one
// equal piece per cluster, so every cluster gets the same number of unit-steps (65536 rows on 148 SMs: 3.46
// chains each instead of 4 rounds with a quarter-full last wave).  A chain cut between clusters w-1 and w is
// run in two parts: cluster w starts its piece with the chain's FIRST steps, cluster w-1 ends its piece with
// the chain's LAST steps (the state x travels through x_io, ordered by a release/acquire flag).  A piece is at
// least one chain long, so part two never has to wait unless part one is late.
struct Seg {
  int unit, s0, s1;
  bool publish;   // first part of a cut chain: set flags[this cluster] when done
  bool acquire;   // second part of a cut chain: wait for flags[next cluster]
};
struct SegIter {
  long long pos, end;
  int S;
  __device__ SegIter(int worker, int n_workers, int n_units, int S_) : S(S_) {
    if (n_units <= n_workers) {
      pos = (long long)min(worker, n_units) * S;
      end = worker < n_units ? pos + S : pos;
    } else {
      const long long total = (long long)n_units * S;
      pos = total * worker / n_workers;
      end = total * (worker + 1) / n_workers;
    }
  }
  __device__ bool next(Seg& g) {
    if (pos >= end) return false;
    const int unit = (int)(pos / S);
    const int off = (int)(pos - (long long)unit * S);
    const long long chain_end = (long long)(unit + 1) * S;
    g.unit = unit; g.publish = false; g.acquire = false;
    if (off > 0) { g.s0 = 0; g.s1 = S - off; g.publish = true; pos = chain_end; }
    else if (chain_end > end) { g.s0 = S - (int)(end - pos); g.s1 = S; g.acquire = true; pos = end; }
    else { g.s0 = 0; g.s1 = S; pos = chain_end; }
    return true;
  }
};

// Wait-time accounting for timing experiments (build with DPB_BUILD_DEFINES=DPB_TC_PROFILE): every role sums
// the cycles it spends in each kind of wait; tc_launch prints the per-role means after the kernel.
// SiLU evaluation in the epilogue.  2 (default): y sigmoid(y) = h + h tanh(h) with h = y/2 and MUFU.TANH
// (tanh.approx.f32, documented relative error 2^-11, the rounding unit of the fp16 activations it feeds; the
// measured end-to-end error is unchanged at 4.5e-4) -- one MUFU per element.  0: y / (1 + 2^(-y log2 e)) with
// MUFU.EX2 + MUFU.RCP, two per element.
// Timing-experiment knobs (KParams::debug, set from DPB_TC_DEBUG) exist only in instrumented builds
// (DPB_BUILD_DEFINES=DPB_TC_PROFILE or DPB_TC_KNOBS); the product kernel compiles them out.
#if defined(DPB_TC_PROFILE) || defined(DPB_TC_KNOBS)
#define DBG(bit) ((p.debug & (bit)) != 0)
#else
#define DBG(bit) false
#endif

#ifndef DPB_SILU_MODE
#define DPB_SILU_MODE 2
#endif
#ifdef DPB_TC_PROFILE
__device__ long long g_prof[256 * 20 * 5];
#define PROF_DECL long long prof_acc[5] = {0, 0, 0, 0, 0}; const long long prof_t0 = clock64();
#define PROF_WAIT(k, ...) do { const long long _t = clock64(); __VA_ARGS__; prof_acc[k] += clock64() - _t; } while (0)
#define PROF_BEGIN(v) const long long v = clock64();
#define PROF_END(k, v) prof_acc[k] += clock64() - v;
#define PROF_FLUSH() do { if (lane == 0) { prof_acc[4] = clock64() - prof_t0; \
    for (int _k = 0; _k < 5; ++_k) g_prof[((size_t)blockIdx.x * 20 + warp) * 5 + _k] = prof_acc[_k]; } } while (0)
#else
#define PROF_DECL
#define PROF_WAIT(k, ...) do { __VA_ARGS__; } while (0)
#define PROF_BEGIN(v)
#define PROF_END(k, v)
#define PROF_FLUSH() do { } while (0)
#endif

// L2-only load: the scratch is written by TMA stores (async proxy), which do not update this SM's L1
__device__ __forceinline__ uint4 ld_global_v4(const uint4* p) {
  uint4 r;
  asm volatile("ld.global.cg.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p));
  return r;
}
// 256-bit variant (one full 32-byte sector per lane: the residual rows are 2 KB apart, so every lane opens its own line)
__device__ __forceinline__ void ld_global_v8(const uint4* p, uint4& a, uint4& b) {
  asm volatile("ld.global.cg.v8.u32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
               : "=r"(a.x), "=r"(a.y), "=r"(a.z), "=r"(a.w), "=r"(b.x), "=r"(b.y), "=r"(b.z), "=r"(b.w) : "l"(p));
}
__device__ __forceinline__ void st_shared_v4(uint32_t addr, uint4 v) {
  asm volatile("st.shared.v4.u32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}
__device__ __forceinline__ void st_global_v4(uint4* p, uint4 v) {
  asm volatile("st.global.v4.u32 [%0], {%1, %2, %3, %4};" ::"l"(p), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}

// ---- packed fp32x2 arithmetic (FADD2 / FMUL2 / FFMA2 on sm_100) and MUFU approximations
__device__ __forceinline__ float2 add2(float2 a, float2 b) {
  float2 d;
  asm("add.rn.f32x2 %0, %1, %2;" : "=l"(*reinterpret_cast<unsigned long long*>(&d))
      : "l"(*reinterpret_cast<unsigned long long*>(&a)), "l"(*reinterpret_cast<unsigned long long*>(&b)));
  return d;
}
__device__ __forceinline__ float2 mul2(float2 a, float2 b) {
  float2 d;
  asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(*reinterpret_cast<unsigned long long*>(&d))
      : "l"(*reinterpret_cast<unsigned long long*>(&a)), "l"(*reinterpret_cast<unsigned long long*>(&b)));
  return d;
}
__device__ __forceinline__ float2 fma2(float2 a, float2 b, float2 c) {
  float2 d;
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(*reinterpret_cast<unsigned long long*>(&d))
      : "l"(*reinterpret_cast<unsigned long long*>(&a)), "l"(*reinterpret_cast<unsigned long long*>(&b)),
        "l"(*reinterpret_cast<unsigned long long*>(&c)));
  return d;
}
__device__ __forceinline__ float ex2_approx(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ float tanh_approx(float x) {
  float y;
  asm("tanh.approx.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ float rcp_approx(float x) {
  float y;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

// One thread, one row, one GroupNorm group (32 consecutive channels):  acc + time bias -> GroupNorm -> SiLU
// (-> + residual) -> 32 fp16 values.  Reductions use four independent partial sums (short dependency chains);
// the elementwise math is packed two channels per instruction.
__device__ __forceinline__ void gn_silu_group(const uint32_t* vr, const float* tb, const float* gm, const float* bt,
                                              bool residual, const uint4* res, uint4* out) {
  float2 v[16];
  float2 s[4] = {{0.f, 0.f}, {0.f, 0.f}, {0.f, 0.f}, {0.f, 0.f}};
#pragma unroll
  for (int i = 0; i < 16; i += 2) {
    const float4 t4 = *reinterpret_cast<const float4*>(tb + 2 * i);
    v[i] = add2(make_float2(__uint_as_float(vr[2 * i]), __uint_as_float(vr[2 * i + 1])), make_float2(t4.x, t4.y));
    v[i + 1] = add2(make_float2(__uint_as_float(vr[2 * i + 2]), __uint_as_float(vr[2 * i + 3])), make_float2(t4.z, t4.w));
    s[(i >> 1) & 3] = add2(s[(i >> 1) & 3], add2(v[i], v[i + 1]));
  }
  const float2 st = add2(add2(s[0], s[1]), add2(s[2], s[3]));
  const float mean = (st.x + st.y) * (1.0f / GROUP);
  const float2 nm = make_float2(-mean, -mean);
  float2 q[4] = {{0.f, 0.f}, {0.f, 0.f}, {0.f, 0.f}, {0.f, 0.f}};
#pragma unroll
  for (int i = 0; i < 16; ++i) {
    v[i] = add2(v[i], nm);
    q[i & 3] = fma2(v[i], v[i], q[i & 3]);
  }
  const float2 qt = add2(add2(q[0], q[1]), add2(q[2], q[3]));
  const float rstd = rsqrtf((qt.x + qt.y) * (1.0f / GROUP) + GN_EPS);
#if DPB_SILU_MODE == 2
  const float2 r2 = make_float2(0.5f * rstd, 0.5f * rstd);   // h = y/2: the staged beta is already halved
#else
  const float2 r2 = make_float2(rstd, rstd);
  const float2 nl2e = make_float2(-1.4426950408889634f, -1.4426950408889634f);
  const float2 one = make_float2(1.0f, 1.0f);
#endif
  uint32_t pk[16];
#pragma unroll
  for (int i = 0; i < 16; i += 2) {
    const float4 g4 = *reinterpret_cast<const float4*>(gm + 2 * i);
    const float4 b4 = *reinterpret_cast<const float4*>(bt + 2 * i);
    float2 y0 = fma2(v[i], mul2(r2, make_float2(g4.x, g4.y)), make_float2(b4.x, b4.y));
    float2 y1 = fma2(v[i + 1], mul2(r2, make_float2(g4.z, g4.w)), make_float2(b4.z, b4.w));
#if DPB_SILU_MODE == 2
    // y0, y1 hold h = y/2 here: SiLU(y) = h + h tanh(h)
    y0 = fma2(y0, make_float2(tanh_approx(y0.x), tanh_approx(y0.y)), y0);
    y1 = fma2(y1, make_float2(tanh_approx(y1.x), tanh_approx(y1.y)), y1);
#else
    // SiLU: y / (1 + 2^(-y log2 e))
    float2 e0 = mul2(y0, nl2e), e1 = mul2(y1, nl2e);
    e0 = make_float2(ex2_approx(e0.x), ex2_approx(e0.y));
    e1 = make_float2(ex2_approx(e1.x), ex2_approx(e1.y));
    e0 = add2(e0, one);
    e1 = add2(e1, one);
    y0 = mul2(y0, make_float2(rcp_approx(e0.x), rcp_approx(e0.y)));
    y1 = mul2(y1, make_float2(rcp_approx(e1.x), rcp_approx(e1.y)));
#endif
    if (residual) {
      const uint32_t* rw = reinterpret_cast<const uint32_t*>(res);
      y0 = add2(y0, __half22float2(*reinterpret_cast<const __half2*>(&rw[i])));
      y1 = add2(y1, __half22float2(*reinterpret_cast<const __half2*>(&rw[i + 1])));
    }
    __half2 p0 = __floats2half2_rn(y0.x, y0.y), p1 = __floats2half2_rn(y1.x, y1.y);
    pk[i] = *reinterpret_cast<uint32_t*>(&p0);
    pk[i + 1] = *reinterpret_cast<uint32_t*>(&p1);
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) out[i] = make_uint4(pk[4 * i], pk[4 * i + 1], pk[4 * i + 2], pk[4 * i + 3]);
}

// K-slab visited at loop position k: the boxes of the previous layer's last chunk are produced in the order
// (hf0,gp0), (hf1,gp0), (hf0,gp1), (hf1,gp1) = slabs 12, 14, 13, 15, so positions 13 and 14 trade places
__device__ __forceinline__ int kslab(int layer, int k) { return (layer > 0 && (k == 13 || k == 14)) ? 27 - k : k; }
template <int PDP>
__device__ __forceinline__ int layer_nk(int layer) { return layer == 0 ? Width<PDP>::XA_K / BLOCK_K : H / BLOCK_K; }
__device__ __forceinline__ int layer_chunks(int layer) { return layer == 5 ? 1 : H / CHUNK_N; }

// First-layer operand.  x[TCOLS] (fp32, columns c0..c0+TCOLS-1 of row r) -> bf16 hi and lo parts, written straight into
// the A halves of the ring stages in the SWIZZLE_128B K-major layout the MMA reads ([128 rows x 64]: row pitch 128 B,
// 16-byte chunk j of row r stored at chunk j ^ (r & 7)).  x_hi column slab s (64 columns) goes to stage s, x_lo slab s
// to stage XA_SLABS + s: stages 0 | 1 at 64 columns, 0, 1 | 2, 3 at 128.  The first layer streams only weight tiles
// through the ring, so the A halves are free while it runs; the last third of [x_hi | x_lo | x_hi] reuses the hi tiles.
// The caller passes the A half of stage 0 (xa_base); the thread's TCOLS columns lie inside one slab.
// A half holding input-layer K slab ks (of 3 XA_SLABS), relative to ring stage 0
template <int PDP>
__device__ __forceinline__ uint32_t xa_stage_offset(int ks) {
  constexpr int NS = Width<PDP>::XA_SLABS;
  if constexpr (NS == 1) return ks == 1 ? STAGE_BYTES : 0;
  else return (uint32_t)(ks < 2 * NS ? ks : ks - 2 * NS) * STAGE_BYTES;
}

template <int PDP>
__device__ __forceinline__ void write_xa(uint32_t xa_base, int r, int c0, const float* x) {
  constexpr int TCOLS = Width<PDP>::TCOLS;
  uint32_t hi_base = xa_base, lo_base = xa_base + STAGE_BYTES;
  if constexpr (Width<PDP>::XA_SLABS > 1) {
    hi_base = xa_base + (uint32_t)(c0 / BLOCK_K) * STAGE_BYTES;
    lo_base = hi_base + (uint32_t)Width<PDP>::XA_SLABS * STAGE_BYTES;
    c0 %= BLOCK_K;
  }
  uint32_t hi[TCOLS / 2], lo[TCOLS / 2];
#pragma unroll
  for (int i = 0; i < TCOLS / 2; ++i) {
    __nv_bfloat16 h0 = __float2bfloat16_rn(x[2 * i]), h1 = __float2bfloat16_rn(x[2 * i + 1]);
    __nv_bfloat16 l0 = __float2bfloat16_rn(x[2 * i] - __bfloat162float(h0));
    __nv_bfloat16 l1 = __float2bfloat16_rn(x[2 * i + 1] - __bfloat162float(h1));
    hi[i] = (uint32_t)__bfloat16_as_ushort(h0) | ((uint32_t)__bfloat16_as_ushort(h1) << 16);
    lo[i] = (uint32_t)__bfloat16_as_ushort(l0) | ((uint32_t)__bfloat16_as_ushort(l1) << 16);
  }
#pragma unroll
  for (int i = 0; i < TCOLS / 8; ++i) {
    const uint32_t off = (uint32_t)r * 128u + ((uint32_t)((c0 / 8 + i) ^ (r & 7)) << 4);
    st_shared_v4(hi_base + off, make_uint4(hi[4 * i], hi[4 * i + 1], hi[4 * i + 2], hi[4 * i + 3]));
    st_shared_v4(lo_base + off, make_uint4(lo[4 * i], lo[4 * i + 1], lo[4 * i + 2], lo[4 * i + 3]));
  }
}

// Gaussian draws for this thread's TCOLS columns: caller-supplied plane or Philox (slot, step); the Philox
// addressing (row, step, slot, quad = column / 4) does not depend on how columns are split over threads
template <int PDP>
__device__ __forceinline__ void draw_cols(const float* plane, long long row, int c0, unsigned long long seed,
                                          uint32_t step, uint32_t slot, float* z) {
  constexpr int TCOLS = Width<PDP>::TCOLS, D = Width<PDP>::D;
  if (plane) {
#pragma unroll
    for (int i = 0; i < TCOLS; ++i) {
      int col = c0 + i;
      z[i] = col < D ? plane[row * D + col] : 0.f;
    }
  } else {
#pragma unroll
    for (int j = 0; j < TCOLS / 4; ++j)
      normal4(seed, (uint64_t)row, step, slot, (uint32_t)(c0 / 4 + j), z + 4 * j, (uint32_t)(PDP / 4));
  }
}

template <int PDP>
__global__ void __cluster_dims__(CLUSTER, 1, 1) __launch_bounds__(NUM_THREADS, 1)
score_tc_kernel(const __grid_constant__ KParams p,
                const __grid_constant__ CUtensorMap tm_h, const __grid_constant__ CUtensorMap tm_t,
                const __grid_constant__ CUtensorMap tm_pre, const __grid_constant__ CUtensorMap tm_w0,
                const __grid_constant__ CUtensorMap tm_w1, const __grid_constant__ CUtensorMap tm_w2,
                const __grid_constant__ CUtensorMap tm_w3, const __grid_constant__ CUtensorMap tm_post) {
  // the pose width of this instantiation (these hide the 63-D namespace constants D / DP)
  using Wd = Width<PDP>;
  constexpr int DP = PDP, D = Wd::D, TCOLS = Wd::TCOLS;
  extern __shared__ uint8_t smem_raw[];
  // 1024-byte alignment for SWIZZLE_128B; offset arithmetic on the __shared__ array keeps ld/st.shared
  uint8_t* smem = smem_raw + ((1024u - (ptx::smem_u32(smem_raw) & 1023u)) & 1023u);
  const uint32_t smem_base = ptx::smem_u32(smem);
  float* par_base = reinterpret_cast<float*>(smem + OFF_PAR);  // 2 x [tb | gamma | beta] x 1024
  const uint32_t stg_base = smem_base + OFF_STG;
  const uint32_t bar_base = smem_base + OFF_BAR;
  auto full_bar = [&](uint32_t s) { return bar_base + 8u * s; };
  auto empty_bar = [&](uint32_t s) { return bar_base + 8u * (STAGES + s); };
  auto tfull_bar = [&](uint32_t b) { return bar_base + 8u * (2 * STAGES + b); };
  auto tempty_bar = [&](uint32_t b) { return bar_base + 8u * (2 * STAGES + 2 + b); };
  auto xa_bar = [&](uint32_t sub) { return bar_base + 8u * (2 * STAGES + 4 + sub); };     // first-layer operand of tile `sub` ready
  auto act_bar = [&](uint32_t sub, uint32_t c) {                                          // column chunk c of a hidden layer ready
    return bar_base + 8u * (2 * STAGES + 4 + NSUB + sub * 4 + c);
  };
  auto sfull_bar = [&](uint32_t hf, uint32_t b) { return bar_base + 8u * (2 * STAGES + 4 + NSUB * 5 + hf * 2 + b); };
  auto sempty_bar = [&](uint32_t hf, uint32_t b) { return bar_base + 8u * (2 * STAGES + 4 + NSUB * 5 + 4 + hf * 2 + b); };
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + OFF_BAR + NUM_BARS * 8);
  float* postb = reinterpret_cast<float*>(smem + OFF_POSTB);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 0) {
    for (int s = 0; s < STAGES; ++s) {
      // TWO_SM: the leader's barrier collects the A and W producers of BOTH CTAs; one multicast commit frees both
      ptx::mbar_init(full_bar(s), TWO_SM ? 4 : 2);
      ptx::mbar_init(empty_bar(s), TWO_SM ? 1 : CLUSTER);
    }
    for (int b = 0; b < 2; ++b) {
      ptx::mbar_init(tfull_bar(b), 1);   // tcgen05.commit
      ptx::mbar_init(tempty_bar(b), TWO_SM ? 32 : 16);  // one lane of each epilogue warp (of both CTAs on the leader)
    }
    for (int sub = 0; sub < NSUB; ++sub) {
      ptx::mbar_init(xa_bar(sub), 16);
      for (int c = 0; c < 4; ++c) ptx::mbar_init(act_bar(sub, c), 1);  // the store warp, after the chunk's TMA stores completed
    }
    for (int hf = 0; hf < 2; ++hf)
      for (int b = 0; b < 2; ++b) {
        ptx::mbar_init(sfull_bar(hf, b), 8);   // the eight epilogue warps (row quarters x column groups) that fill one box
        ptx::mbar_init(sempty_bar(hf, b), 1);  // the store warp, once the TMA store has read the box
      }
    ptx::fence_barrier_init();
  }
  if (warp == 0 && lane == 0) {
    ptx::prefetch_tmap(&tm_pre); ptx::prefetch_tmap(&tm_w0); ptx::prefetch_tmap(&tm_w1);
    ptx::prefetch_tmap(&tm_w2); ptx::prefetch_tmap(&tm_w3); ptx::prefetch_tmap(&tm_post);
  }
  if (warp == 2) {
    if (lane == 0) { ptx::prefetch_tmap(&tm_h); ptx::prefetch_tmap(&tm_t); }
    __syncwarp();
    if (TWO_SM) ptx::tmem_alloc_2sm(ptx::smem_u32(tmem_slot), 512);
    else ptx::tmem_alloc(ptx::smem_u32(tmem_slot), 512);
  }
  if (threadIdx.x >= 128 && threadIdx.x < 128 + DP) postb[threadIdx.x - 128] = p.post_b[threadIdx.x - 128];
  ptx::tc_fence_before();
  __syncthreads();
  if (CLUSTER > 1) ptx::cluster_sync();  // peers' barriers are initialised before anyone multicasts / arrives remotely
  ptx::tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const int slot_row0 = blockIdx.x * NSUB * TILE_M;  // this CTA's rows in the scratch buffers (NSUB slots)
  const uint32_t crank = CLUSTER > 1 ? ptx::cluster_ctarank() : 0;
  constexpr uint16_t CMASK = (uint16_t)((1u << CLUSTER) - 1);
  // both CTAs of a cluster walk the same segment list (SegIter); CTA `crank` owns tile unit*CLUSTER + crank
  const int worker = (int)blockIdx.x / CLUSTER, n_workers = (int)gridDim.x / CLUSTER;
  const int n_units = (p.n_tiles + CLUSTER * NSUB - 1) / (CLUSTER * NSUB);
  Seg sg;
  PROF_DECL
  // the activation scratch is written and re-read once per layer and never needed in HBM: evict_last on its TMA
  // stores and loads keeps the boxes in L2 (DPB_TC_L2HINT=0 at build time restores unhinted copies, A/B)
#ifndef DPB_TC_L2HINT
#define DPB_TC_L2HINT 1
#endif
  const uint64_t pol_act = DPB_TC_L2HINT == 2 ? ptx::l2_policy_evict_first() : ptx::l2_policy_evict_last();

  // register budget: the four single-lane roles (warpgroup 0) give registers to the 256 epilogue threads
  if (warp < 4) {
  ptx::setmaxnreg_dec<ROLE_REGS>();
  if (warp == 0) {
    // ======================= weight producer =======================
    {
      uint32_t stage = 0, phase = 0;
      for (SegIter it(worker, n_workers, n_units, p.n_steps); it.next(sg);)
        for (int step = sg.s0; step < sg.s1; ++step)
          for (int layer = 0; layer < 6; ++layer) {
            const CUtensorMap* tm = layer == 0 ? &tm_pre : layer == 1 ? &tm_w0 : layer == 2 ? &tm_w1
                                  : layer == 3 ? &tm_w2 : layer == 4 ? &tm_w3 : &tm_post;
            const uint32_t bytes = layer == 5 ? Wd::POST_B_BYTES : B_BYTES;
            const int nk = layer_nk<PDP>(layer), nc = layer_chunks(layer);
            for (int chunk = 0; chunk < nc; ++chunk)
             for (int sub = 0; sub < NSUB; ++sub)
              for (int k = 0; k < nk; ++k) {
                PROF_WAIT(0, ptx::mbar_wait(empty_bar(stage), phase ^ 1));  // every CTA of the cluster has consumed this stage
                const int part_rows = (layer == 5 ? DP : CHUNK_N) / CLUSTER;
                if (TWO_SM) {  // my half of the weight tile into MY shared memory, completion on the leader's barrier
                  const uint32_t lbar = ptx::mapa(full_bar(stage), 0);
                  if (ptx::elect_one()) {
                    if (DBG(8)) ptx::mbar_arrive_cluster(lbar);
                    else {
                      ptx::mbar_arrive_expect_tx_cluster(lbar, bytes);
                      ptx::tma_load_2d_2sm(smem_base + stage * STAGE_BYTES + A_BYTES, tm, lbar, kslab(layer, k) * BLOCK_K,
                                           chunk * CHUNK_N + crank * part_rows);
                    }
                  }
                  if (++stage == STAGES) { stage = 0; phase ^= 1; }
                  continue;
                }
                const uint32_t dst = smem_base + stage * STAGE_BYTES + A_BYTES + crank * part_rows * (BLOCK_K * 2);
                if (ptx::elect_one()) {
                  ptx::mbar_arrive_expect_tx(full_bar(stage), bytes);  // whole tile: own part + the peers' multicasts
                  if (CLUSTER > 1)
                    ptx::tma_load_2d_mcast(dst, tm, full_bar(stage), kslab(layer, k) * BLOCK_K,
                                           chunk * CHUNK_N + crank * part_rows, CMASK);
                  else
                    ptx::tma_load_2d(dst, tm, full_bar(stage), kslab(layer, k) * BLOCK_K, chunk * CHUNK_N);
                }
                if (++stage == STAGES) { stage = 0; phase ^= 1; }
              }
          }
    }
  } else if (warp == 1) {
    // ======================= MMA issuer =======================
    if (!TWO_SM || crank == 0) {   // cta_group::2: the pair's leader issues for both CTAs (warp-wide loop, elected lane issues)
      uint32_t stage = 0, phase = 0, chunk_ctr = 0, tph = 0;
      for (SegIter it(worker, n_workers, n_units, p.n_steps); it.next(sg);)
        for (int step = sg.s0; step < sg.s1; ++step)
          for (int layer = 0; layer < 6; ++layer) {
            const uint32_t idesc = layer == 0 ? IDESC_BF16_256 : layer == 5 ? Wd::IDESC_POST : IDESC_F16_256;
            const int nk = layer_nk<PDP>(layer), nc = layer_chunks(layer);
            for (int cs = 0; cs < nc * NSUB; ++cs) {   // (chunk, sub) pairs; chunk_ctr & 1 == sub
              const uint32_t buf = chunk_ctr & 1;
              if (!DBG(64)) PROF_WAIT(0, ptx::mbar_wait(tempty_bar(buf), ((tph >> buf) & 1) ^ 1));
              ptx::tc_fence_after();
              const uint32_t taddr = tmem_base + buf * CHUNK_N;
              for (int k = 0; k < nk; ++k) {
                PROF_WAIT(1, ptx::mbar_wait(full_bar(stage), phase));
                ptx::tc_fence_after();
                const uint32_t s_addr = smem_base + stage * STAGE_BYTES;
                const int ks = kslab(layer, k);
                // first chunk of a layer: the last four K slabs are still in the staging boxes of the previous layer
                const bool direct = layer > 0 && cs == 0 && ks >= DIRECT_K0 && !DBG(64);
                // first layer: x_hi | x_lo | x_hi, written by the epilogue into the A halves of ring stages
                // 0 .. 2 XA_SLABS - 1 (slab ks; the last third re-reads the x_hi stages)
                const uint32_t a_addr = layer == 0 ? smem_base + xa_stage_offset<PDP>(ks)
                                      : direct ? stg_base + (ks - DIRECT_K0) * STG_BYTES : s_addr;
                const uint64_t adesc = ptx::umma_desc_sw128(a_addr);
                const uint64_t bdesc = ptx::umma_desc_sw128(s_addr + A_BYTES);
                PROF_BEGIN(issue_t0)
                if (ptx::elect_one()) {
                  if (!DBG(2))
#pragma unroll
                  for (int kk = 0; kk < BLOCK_K / 16; ++kk)  // UMMA_K = 16: advance 32 B inside the swizzle row
                    if (TWO_SM) ptx::mma_f16_ss_2sm(taddr, adesc + 2 * kk, bdesc + 2 * kk, idesc, (k | kk) != 0 ? 1u : 0u);
                    else ptx::mma_f16_ss(taddr, adesc + 2 * kk, bdesc + 2 * kk, idesc, (k | kk) != 0 ? 1u : 0u);
                  if (TWO_SM) ptx::mma_commit_2sm_mcast(empty_bar(stage), CMASK);
                  else if (CLUSTER > 1) ptx::mma_commit_mcast(empty_bar(stage), CMASK);
                  else ptx::mma_commit(empty_bar(stage));
                  if (k == nk - 1) {   // the chunk's accumulator is complete once everything issued so far retires
                    if (TWO_SM) ptx::mma_commit_2sm_mcast(tfull_bar(buf), CMASK);
                    else ptx::mma_commit(tfull_bar(buf));
                  }
                }
                __syncwarp();
                PROF_END(2, issue_t0)
                if (++stage == STAGES) { stage = 0; phase ^= 1; }
              }
              tph ^= 1u << buf;
              ++chunk_ctr;
            }
          }
    }
  } else if (warp == 2) {
    // ======================= activation producer =======================
    {
      uint32_t stage = 0, phase = 0, xph = 0, aph = 0, cctr = 0;   // cctr: chunks so far (the MMA warp's chunk_ctr)
      for (SegIter it(worker, n_workers, n_units, p.n_steps); it.next(sg);)
        for (int step = sg.s0; step < sg.s1; ++step)
          for (int layer = 0; layer < 6; ++layer) {
            // layer input: x (shared memory, written by the epilogue) | H | T | H | T | H
            const CUtensorMap* tm = (layer == 2 || layer == 4) ? &tm_t : &tm_h;
            const int nk = layer_nk<PDP>(layer), nc = layer_chunks(layer);
            if (layer == 1 && !DBG(64)) {
              // the first layer's operand lives in the A halves of ring stages 0 .. 2 XA_SLABS - 1 (0 / 1, or 0 - 3 at
              // 128 columns): no activation tile may land in ANY stage before ALL first-layer MMAs have retired (= the
              // accumulator of its last chunk is complete).  This wait precedes the first load of the next layer, so it
              // covers every stage the operand occupies.
              const uint32_t n = cctr - 1;
              PROF_WAIT(1, ptx::mbar_wait(tfull_bar(n & 1), (n >> 1) & 1));
            }
            for (int chunk = 0; chunk < nc; ++chunk, ++cctr)
             for (int sub = 0; sub < NSUB; ++sub) {
              if (layer == 0 && chunk == 0 && !DBG(64)) PROF_WAIT(0, ptx::mbar_wait(xa_bar(sub), xph));  // prologue / previous step's tail wrote x
              for (int k = 0; k < nk; ++k) {
                // K-slabs 4c..4c+3 of this layer's input are column chunk c of the previous layer's output:
                // wait for exactly that chunk (first use only), so the next layer starts while the previous
                // layer's last chunks are still in the epilogue.  The slabs of the LAST chunk are not loaded at
                // all for this layer's first chunk: the MMA reads them from the staging boxes (box = slab - 12)
                // as soon as the epilogue has filled them; the later chunks fetch them from the scratch.
                const int ks = kslab(layer, k);
                const bool boxed = layer > 0 && chunk == 0 && ks >= DIRECT_K0 && !DBG(64);
                const bool direct = boxed || layer == 0;   // nothing to load: the MMA reads shared memory the epilogue wrote
                if (layer > 0 && !DBG(64)) {
                  if (boxed) {
                    const int kb = ks - DIRECT_K0;   // (hf, gp) = (kb >> 1, kb & 1); the last chunk's box phase is always odd
                    PROF_WAIT(1, ptx::mbar_wait(sfull_bar(kb >> 1, kb & 1), 1));
                  } else if ((chunk == 0 && (ks & 3) == 0) || (chunk == 1 && k == DIRECT_K0)) {
                    PROF_WAIT(1, ptx::mbar_wait(act_bar(sub, ks >> 2), aph));
                  }
                }
                PROF_WAIT(2, ptx::mbar_wait(empty_bar(stage), phase ^ 1));
                if (TWO_SM) {
                  const uint32_t lbar = ptx::mapa(full_bar(stage), 0);
                  if (ptx::elect_one()) {
                    if (DBG(4) || direct) ptx::mbar_arrive_cluster(lbar);
                    else {
                      ptx::mbar_arrive_expect_tx_cluster(lbar, A_BYTES);
                      if (DPB_TC_L2HINT)
                        ptx::tma_load_2d_2sm_hint(smem_base + stage * STAGE_BYTES, tm, lbar, ks * BLOCK_K,
                                                  slot_row0 + sub * TILE_M, pol_act);
                      else
                        ptx::tma_load_2d_2sm(smem_base + stage * STAGE_BYTES, tm, lbar, ks * BLOCK_K, slot_row0 + sub * TILE_M);
                    }
                  }
                } else if (ptx::elect_one()) {
                  if (direct) ptx::mbar_arrive(full_bar(stage));
                  else {
                    ptx::mbar_arrive_expect_tx(full_bar(stage), A_BYTES);
                    ptx::tma_load_2d(smem_base + stage * STAGE_BYTES, tm, full_bar(stage), ks * BLOCK_K,
                                     slot_row0 + sub * TILE_M);
                  }
                }
                if (++stage == STAGES) { stage = 0; phase ^= 1; }
              }
             }
            if (layer == 0) xph ^= 1;
            else aph ^= 1;
          }
    }
  } else if (warp == 3) {
    // ======================= activation store warp =======================
    // Epilogue warps stage each [128 x 64] fp16 box in shared memory (swizzled); this warp turns boxes into
    // TMA stores (full 128-byte lines into the L2-resident scratch) and publishes a column chunk to the
    // activation producer once its stores have completed.
    // Bulk async-groups are tracked per thread: elect_one() names the same lane every time, so commit / wait
    // pair up with the stores they follow.
    {
      uint32_t cnt0 = 0, cnt1 = 0;
      uint32_t last_bar = 0;      // sempty barrier of the most recent store that has not been handed back yet
      bool last_released = true;
      if (!DBG(64))
      for (SegIter it(worker, n_workers, n_units, p.n_steps); it.next(sg);)
        for (int step = sg.s0; step < sg.s1; ++step)
          for (int layer = 0; layer < 5; ++layer) {
            const CUtensorMap* tm = (layer == 0 || layer == 2 || layer == 4) ? &tm_h : &tm_t;
            for (int cs = 0; cs < (H / CHUNK_N) * NSUB; ++cs) {
              const int chunk = cs / NSUB, sub = cs % NSUB;
              for (int gp = 0; gp < 2; ++gp)
#pragma unroll
                for (int hf = 0; hf < 2; ++hf) {
                  const uint32_t c = hf ? cnt1 : cnt0;
                  const uint32_t b = c % STG_BUFS, ph = (c / STG_BUFS) & 1;
                  PROF_WAIT(0, ptx::mbar_wait(sfull_bar(hf, b), ph));
                  if (ptx::elect_one()) {
                    if (!DBG(16))
                    {
                      if (DPB_TC_L2HINT)
                        ptx::tma_store_2d_hint(tm, stg_base + (hf * STG_BUFS + b) * STG_BYTES,
                                               chunk * CHUNK_N + hf * 128 + gp * 64, slot_row0 + sub * TILE_M, pol_act);
                      else
                        ptx::tma_store_2d(tm, stg_base + (hf * STG_BUFS + b) * STG_BYTES,
                                          chunk * CHUNK_N + hf * 128 + gp * 64, slot_row0 + sub * TILE_M);
                    }
                    ptx::tma_store_commit();
                    if (!last_released) {  // the previous store has finished READING its box: hand that box back
                      PROF_WAIT(1, ptx::tma_store_wait_read<1>());
                      ptx::mbar_arrive(last_bar);
                    }
                  }
                  last_bar = sempty_bar(hf, b);
                  last_released = false;
                  if (hf) ++cnt1; else ++cnt0;
                }
              if (ptx::elect_one()) {
                PROF_WAIT(2, ptx::tma_store_wait<0>());  // this chunk's stores are complete (visible to the TMA loads that follow)
                ptx::mbar_arrive(last_bar);
                ptx::mbar_arrive(act_bar(sub, chunk));
              }
              last_released = true;
            }
          }
    }
  }
  } else {
    // ======================= epilogue (16 warps) =======================
    // Warp (q, hf, sg2): TMEM lane quarter q (rows 32q..32q+31), column half hf of the chunk, and within each of the
    // half's two 64-column boxes the 32-column GroupNorm group sg2.  Four warps per scheduler hide the MUFU / TMEM /
    // shared-memory latencies of the per-row chains that two warps per scheduler left exposed.
    ptx::setmaxnreg_inc<EPI_REGS>();
    const int q = warp & 3;
    const int hf = (warp - 4) >> 3;
    const int sg2 = ((warp - 4) >> 2) & 1;
    const int et = threadIdx.x - 128;
    const int r_in = q * 32 + lane;
    const int c0 = hf * (2 * TCOLS) + sg2 * TCOLS;   // first of this thread's TCOLS pose columns (prologue / tail)
    const uint32_t lane_addr = (uint32_t)(q * 32) << 16;
    uint32_t chunk_ctr = 0, tph = 0, scnt = 0;
    auto signal = [&](uint32_t bar) {  // generic-proxy shared-memory writes -> visible to the MMA (async proxy) reads
      ptx::fence_proxy_async_smem();
      __syncwarp();
      if (lane == 0) ptx::mbar_arrive(bar);
    };
    const uint32_t xa_base = smem_base;   // A half of ring stage 0 (write_xa places the slabs)
    auto tempty_arrive = [&](uint32_t buf) {
      ptx::tc_fence_before();
      __syncwarp();
      if (lane == 0) {
        if (TWO_SM) ptx::mbar_arrive_cluster(ptx::mapa(tempty_bar(buf), 0));
        else ptx::mbar_arrive(tempty_bar(buf));
      }
    };
    uint32_t pcnt = 0;             // hidden layers processed so far (parameter buffer = pcnt & 1)
    bool par_prefetched = false;
    auto stage_par = [&](int step_, int layer_, uint32_t slot) {
      const float4* tb = reinterpret_cast<const float4*>(p.table + ((size_t)(p.pc ? step_ >> 1 : step_) * NL + layer_) * H);
      const float4* gn = reinterpret_cast<const float4*>(p.gn + (size_t)(layer_ * 2) * H);  // gamma | beta (pre-halved)
      const uint32_t dst = ptx::smem_u32(par_base) + slot * (3 * H * 4);
      if (et < H / 4) ptx::cp_async_16(dst + et * 16, tb + et);
      ptx::cp_async_16(dst + (H / 4 + et) * 16, gn + et);   // 2 * H / 4 == EPI_THREADS float4
      ptx::cp_async_commit();
    };
    float xs[NSUB][TCOLS];   // sampler state of this thread's (row, TCOLS columns), carried in registers across the steps
    if (!DBG(64))
    for (SegIter it(worker, n_workers, n_units, p.n_steps); it.next(sg);) {
      const long long tile0 = ((long long)sg.unit * CLUSTER + crank) * NSUB;
      if (sg.acquire) {  // the chain's first steps ran on the next cluster: wait until its x_io rows are published
        if (et == 0) {
          const int* f = p.flags + (size_t)(worker + 1) * CLUSTER + crank;
          while (ptx::ld_acquire_gpu(f) == 0) __nanosleep(200);
        }
        ptx::named_bar_sync(1, EPI_THREADS);
      }
      // ---------------- tile prologue: first-layer operand of the segment's first step
#pragma unroll
      for (int sub = 0; sub < NSUB; ++sub) {
        const long long row = (tile0 + sub) * TILE_M + r_in;
        const bool valid = row < p.B;
        float x[TCOLS];
#pragma unroll
        for (int i = 0; i < TCOLS; ++i) x[i] = 0.f;
        if (valid) {
          if (p.mode == 1) {
#pragma unroll
            for (int i = 0; i < TCOLS; ++i) {
              int col = c0 + i;
              if (col < D) x[i] = __ldcg(p.x_io + row * D + col);
            }
            if (p.impute && sg.s0 == 0 && !p.pc) {  // imputation that follows the (none) corrector of step 0, sampling.py:459
              float zc[TCOLS];
              draw_cols<PDP>(p.noise ? p.noise : nullptr, row, c0, p.seed, (uint32_t)p.step_offset, 0, zc);
              const float al = p.coef[3], sd = p.coef[4];
#pragma unroll
              for (int i = 0; i < TCOLS; ++i) {
                int col = c0 + i;
                if (col < D) {
                  float m = p.mask[row * D + col];
                  x[i] = x[i] * (1.0f - m) + (al * p.obs[row * D + col] + zc[i] * sd) * m;
                }
              }
            }
          } else if (p.mode == 0) {
#pragma unroll
            for (int i = 0; i < TCOLS; ++i) {
              int col = c0 + i;
              if (col < D) x[i] = p.x_in[row * D + col];
            }
          } else {  // prior loss: x_t = alpha x0 + std z
            float z[TCOLS];
            draw_cols<PDP>(p.z, row, c0, p.seed, (uint32_t)p.step_offset, 3, z);
#pragma unroll
            for (int i = 0; i < TCOLS; ++i) {
              int col = c0 + i;
              if (col < D) x[i] = p.alpha * p.x_in[row * D + col] + p.sd * z[i];
            }
          }
        }
        write_xa<PDP>(xa_base, r_in, c0, x);
        signal(xa_bar(sub));
#pragma unroll
        for (int i = 0; i < TCOLS; ++i) xs[sub][i] = x[i];
      }
      for (int step = sg.s0; step < sg.s1; ++step) {
        // ---------------- hidden layers 0..4
        for (int layer = 0; layer < 5; ++layer) {
          // layer parameters (time bias of this step, gamma, beta/2) are double-buffered in shared memory: the next
          // layer's set is copied with cp.async while this layer runs, so a layer boundary costs one barrier and no
          // exposed global-memory latency
          if (!par_prefetched) stage_par(step, layer, pcnt & 1);
          ptx::cp_async_wait_all();
          ptx::named_bar_sync(1, EPI_THREADS);  // all copies of this set have landed; everyone left the previous layer
          par_prefetched = false;
          if (layer < 4) { stage_par(step, layer + 1, (pcnt + 1) & 1); par_prefetched = true; }
          else if (step + 1 < sg.s1) { stage_par(step + 1, 0, (pcnt + 1) & 1); par_prefetched = true; }
          const float* par = par_base + (size_t)(pcnt & 1) * 3 * H;
          ++pcnt;
          const bool to_h = (layer == 0 || layer == 2 || layer == 4);
          const bool residual = (layer == 2 || layer == 4);
#pragma unroll 1
          for (int cs = 0; cs < (H / CHUNK_N) * NSUB; ++cs) {
            const int chunk = cs / NSUB, sub = cs % NSUB;
            __half* drow = (to_h ? p.act_h : p.act_t) + (size_t)(slot_row0 + sub * TILE_M + r_in) * H;
            const uint32_t buf = chunk_ctr & 1;
            // residual stream: this thread's 2 x 32 old values of the chunk are requested BEFORE the accumulator
            // wait (they were stored two layers ago), so their L2 latency hides behind it
            uint4 rres[2][4];
            if (residual && !DBG(512)) {
#pragma unroll
              for (int gp = 0; gp < 2; ++gp) {
                const uint4* rp = reinterpret_cast<const uint4*>(drow + chunk * CHUNK_N + (hf * 4 + gp * 2 + sg2) * 32);
                ld_global_v8(rp, rres[gp][0], rres[gp][1]);
                ld_global_v8(rp + 2, rres[gp][2], rres[gp][3]);
              }
            }
#ifdef DPB_TC_PROFILE_TAIL
            ptx::mbar_wait(tfull_bar(buf), (tph >> buf) & 1);
#else
            PROF_WAIT(0, ptx::mbar_wait(tfull_bar(buf), (tph >> buf) & 1));
#endif
            ptx::tc_fence_after();
#pragma unroll
            for (int gp = 0; gp < 2; ++gp) {
              const int g = hf * 4 + gp * 2 + sg2;           // my 32-column group of the chunk
              const int col0 = chunk * CHUNK_N + g * 32;
              uint32_t vr[32];
              if (DBG(128)) {
#pragma unroll
                for (int i = 0; i < 32; ++i) vr[i] = 0;
              } else {
                ptx::tmem_ld_32x32(tmem_base + lane_addr + buf * CHUNK_N + g * 32, vr);
              }
              const uint4* r0 = rres[gp];
              ptx::tmem_ld_wait();
              if (gp == 1) tempty_arrive(buf);  // last TMEM read of this warp for the buffer: hand it back to the MMA warp
              uint4 o[4];
              if (DBG(1)) {
#pragma unroll
                for (int i = 0; i < 4; ++i) o[i] = make_uint4(0, 0, 0, 0);
              } else {
#ifdef DPB_TC_PROFILE_TAIL
                gn_silu_group(vr, par + col0, par + H + col0, par + 2 * H + col0, residual, r0, o);
#else
                PROF_WAIT(2, gn_silu_group(vr, par + col0, par + H + col0, par + 2 * H + col0, residual, r0, o));
#endif
              }
              // stage this row's 32 fp16 (64 B, half of the 128-byte row) in the SWIZZLE_128B box (hf, gp); the
              // store warp ships the box with one TMA store (full lines, asynchronous) -- no per-row global stores
              const uint32_t sb = scnt % STG_BUFS;
#ifdef DPB_TC_PROFILE_TAIL
              ptx::mbar_wait(sempty_bar(hf, sb), ((scnt / STG_BUFS) & 1) ^ 1);
#else
              PROF_WAIT(1, ptx::mbar_wait(sempty_bar(hf, sb), ((scnt / STG_BUFS) & 1) ^ 1));
#endif
              const uint32_t rbase = stg_base + (hf * STG_BUFS + sb) * STG_BYTES + r_in * 128;
#pragma unroll
              for (int j = 0; j < 4; ++j)
                if (!DBG(256)) st_shared_v4(rbase + (((sg2 * 4 + j) ^ (r_in & 7)) << 4), o[j]);
              ptx::fence_proxy_async_smem();
              __syncwarp();
              if (lane == 0) ptx::mbar_arrive(sfull_bar(hf, sb));
              ++scnt;
            }
            tph ^= 1u << buf;
            ++chunk_ctr;
          }
        }
        // ---------------- post_dense + mode-specific tail
#pragma unroll
        for (int sub = 0; sub < NSUB; ++sub) {
          const long long row = (tile0 + sub) * TILE_M + r_in;
          const bool valid = row < p.B;
          const uint32_t buf = chunk_ctr & 1;
          // everything of the sampler update that does not depend on the network output is prepared BEFORE the
          // accumulator wait: this step's coefficients and its Gaussian draws (Philox + Box-Muller)
          const bool last = (step + 1 == p.n_steps);
          const int lstep = p.pc ? (step >> 1) : step;           // the sampler step this sub-step belongs to
          const bool corr = p.pc && !(step & 1);                 // corrector sub-step (its score evaluation just ran)
          const float* cf = p.coef + (size_t)lstep * DPB_COEF_STRIDE;
          const uint32_t gstep = (uint32_t)(p.step_offset + (unsigned long long)lstep);
          const size_t plane = (size_t)p.B * D;
          float ca = 0.f, cb = 0.f, cc = 0.f, al = 0.f, sd = 0.f;
          // given noise: [n, K, B, D] planes of the predictor; with the corrector [n, K + 1, B, D], its draw first
          const float* nzc = p.noise ? p.noise + (size_t)lstep * (p.noise_k + (p.pc ? 1 : 0)) * plane : nullptr;
          const float* nz = (nzc && p.pc) ? nzc + plane : nzc;
          float zp[TCOLS];
#pragma unroll
          for (int i = 0; i < TCOLS; ++i) zp[i] = 0.f;
          if (p.mode == 1 && valid) {
            ca = cf[0]; cb = cf[1]; cc = cf[2]; al = cf[3]; sd = cf[4];
            if (corr) draw_cols<PDP>(nzc, row, c0, p.seed, gstep, 4, zp);          // the Langevin draw (Philox slot 4)
            else draw_cols<PDP>(nz ? nz + (p.noise_k == 3 ? plane : 0) : nullptr, row, c0, p.seed, gstep, 1, zp);
          }
          if (p.mode == 1) {  // pin the draws above the wait (the compiler would otherwise sink them below it)
#pragma unroll
            for (int i = 0; i < TCOLS; ++i) asm volatile("" ::"f"(zp[i]));
          }
          ptx::mbar_wait(tfull_bar(buf), (tph >> buf) & 1);
          PROF_BEGIN(tail_t0)
          ptx::tc_fence_after();
          uint32_t vr[TCOLS];
          if constexpr (TCOLS == 32) ptx::tmem_ld_32x32(tmem_base + lane_addr + buf * CHUNK_N + c0, vr);
          else ptx::tmem_ld_32x16(tmem_base + lane_addr + buf * CHUNK_N + c0, vr);
          ptx::tmem_ld_wait();
          tempty_arrive(buf);
#ifdef DPB_TC_PROFILE_TAIL
          prof_acc[0] += clock64() - tail_t0;
#endif
          tph ^= 1u << buf;
          ++chunk_ctr;
          float raw[TCOLS];
#pragma unroll
          for (int i = 0; i < TCOLS; i += 4) {
            const float4 pb = *reinterpret_cast<const float4*>(postb + c0 + i);
            raw[i] = __uint_as_float(vr[i]) + pb.x; raw[i + 1] = __uint_as_float(vr[i + 1]) + pb.y;
            raw[i + 2] = __uint_as_float(vr[i + 2]) + pb.z; raw[i + 3] = __uint_as_float(vr[i + 3]) + pb.w;
          }
          if (p.mode == 0) {
            if (valid) {
              const float sc = p.row_scale ? p.row_scale[row] : p.scale;
#pragma unroll
              for (int i = 0; i < TCOLS; ++i) {
                int col = c0 + i;
                if (col < D) p.out[row * D + col] = raw[i] * sc;
              }
            }
          } else if (p.mode == 1 && corr && DBG(8192)) {     // timing experiment: corrector sub-step without its tail
            float x[TCOLS];
#pragma unroll
            for (int i = 0; i < TCOLS; ++i) x[i] = xs[sub][i] + 1e-9f * raw[i];
            write_xa<PDP>(xa_base, r_in, c0, x);
            signal(xa_bar(sub));
          } else if (p.mode == 1 && corr) {
            // ---- Langevin corrector (sampling.py:282-302): grad = score, batch-global mean norms, x += step grad + sqrt(2 step) z
            float* rowsq = reinterpret_cast<float*>(smem + Wd::OFF_PCROW);
            float gsq = 0.f, zsq = 0.f;
            float grad[TCOLS];
#pragma unroll
            for (int i = 0; i < TCOLS; ++i) {
              grad[i] = (valid && c0 + i < D) ? raw[i] * cf[5] : 0.f;
              gsq = fmaf(grad[i], grad[i], gsq);
              if (valid && c0 + i < D) zsq = fmaf(zp[i], zp[i], zsq);
            }
            if (c0 == 0) { rowsq[2 * r_in] = 0.f; rowsq[2 * r_in + 1] = 0.f; }
            ptx::named_bar_sync(1, EPI_THREADS);
            atomicAdd(rowsq + 2 * r_in, gsq);
            atomicAdd(rowsq + 2 * r_in + 1, zsq);
            ptx::named_bar_sync(1, EPI_THREADS);
            if (c0 == 0) {                                   // one warp per row quarter: sum of the rows' norms
              float ng = valid ? sqrtf(rowsq[2 * r_in]) : 0.f, nzz = valid ? sqrtf(rowsq[2 * r_in + 1]) : 0.f;
              for (int o = 16; o > 0; o >>= 1) {
                ng += __shfl_xor_sync(0xffffffffu, ng, o);
                nzz += __shfl_xor_sync(0xffffffffu, nzz, o);
              }
              if (lane == 0) {
                atomicAdd(p.pc_sums + 2 * lstep, ng);
                atomicAdd(p.pc_sums + 2 * lstep + 1, nzz);
              }
            }
            // grid barrier: every CTA has added its rows (lock step: all CTAs run the same sub-step sequence)
            if (!DBG(1024)) __threadfence();
            ptx::named_bar_sync(1, EPI_THREADS);
            if (et == 0 && !DBG(2048)) {
              atomicAdd(p.pc_counter, 1);
              const int target = (lstep + 1) * (int)gridDim.x;
              while (ptx::ld_acquire_gpu(p.pc_counter) < target) {
              }
              __threadfence();
            }
            ptx::named_bar_sync(1, EPI_THREADS);
            const float sum_g = DBG(4096) ? 1.f : __ldcg(p.pc_sums + 2 * lstep), sum_z = DBG(4096) ? 1.f : __ldcg(p.pc_sums + 2 * lstep + 1);
            const float rr = p.snr * sum_z / sum_g;          // both means share the divisor (sampling.py:296-298)
            const float stp = rr * rr * 2.0f * cf[6];
            const float sq = sqrtf(stp * 2.0f);
            float x[TCOLS];
#pragma unroll
            for (int i = 0; i < TCOLS; ++i) x[i] = valid ? (xs[sub][i] + stp * grad[i]) + sq * zp[i] : 0.f;
            if (valid && p.impute) {                         // imputation after the corrector (sampling.py:459, 413-422)
              float zc[TCOLS];
              draw_cols<PDP>(nz, row, c0, p.seed, gstep, 0, zc);
#pragma unroll
              for (int i = 0; i < TCOLS; ++i) {
                int col = c0 + i;
                if (col < D) {
                  float m = p.mask[row * D + col];
                  x[i] = x[i] * (1.0f - m) + (al * p.obs[row * D + col] + zc[i] * sd) * m;
                }
              }
            }
#pragma unroll
            for (int i = 0; i < TCOLS; ++i) xs[sub][i] = x[i];
            write_xa<PDP>(xa_base, r_in, c0, x);             // the predictor sub-step always follows
            signal(xa_bar(sub));
          } else if (p.mode == 1) {
            float x[TCOLS];
#pragma unroll
            for (int i = 0; i < TCOLS; ++i) x[i] = 0.f;
            if (valid) {
#pragma unroll
              for (int i = 0; i < TCOLS; ++i) {
                int col = c0 + i;
                if (col < D) {
                  float xm = ca * xs[sub][i] + cb * raw[i];  // sampling.py:185-186 in affine form
                  x[i] = xm + cc * zp[i];
                  if (last && p.x_mean) p.x_mean[row * D + col] = xm;
                }
              }
              // (between steps without a trajectory the imputed columns are overwritten by the next step's pre-imputation
              //  before anything reads them: the draw is skipped, results are identical)
              if (p.impute && (last || p.traj || p.pc)) {
                float zi[TCOLS];
                draw_cols<PDP>(nz ? nz + 2 * plane : nullptr, row, c0, p.seed, gstep, 2, zi);
#pragma unroll
                for (int i = 0; i < TCOLS; ++i) {
                  int col = c0 + i;
                  if (col < D) {
                    float m = p.mask[row * D + col];
                    x[i] = x[i] * (1.0f - m) + (al * p.obs[row * D + col] + zi[i] * sd) * m;
                  }
                }
              }
              if (p.traj) {
#pragma unroll
                for (int i = 0; i < TCOLS; ++i) {
                  int col = c0 + i;
                  if (col < D) p.traj[((size_t)lstep * p.B + row) * D + col] = x[i];
                }
              }
              if (!last && p.impute && !p.pc) {  // imputation in the corrector slot of the NEXT step precedes its score eval
                float zc[TCOLS];
                const float* nz1 = p.noise ? p.noise + (size_t)(step + 1) * p.noise_k * plane : nullptr;
                draw_cols<PDP>(nz1, row, c0, p.seed, gstep + 1, 0, zc);
                const float al1 = cf[DPB_COEF_STRIDE + 3], sd1 = cf[DPB_COEF_STRIDE + 4];
#pragma unroll
                for (int i = 0; i < TCOLS; ++i) {
                  int col = c0 + i;
                  if (col < D) {
                    float m = p.mask[row * D + col];
                    x[i] = x[i] * (1.0f - m) + (al1 * p.obs[row * D + col] + zc[i] * sd1) * m;
                  }
                }
              }
              if (step + 1 == sg.s1) {  // end of the segment: the state leaves the registers
#pragma unroll
                for (int i = 0; i < TCOLS; ++i) {
                  int col = c0 + i;
                  if (col < D) p.x_io[row * D + col] = x[i];
                }
              }
            }
#pragma unroll
            for (int i = 0; i < TCOLS; ++i) xs[sub][i] = x[i];
            if (step + 1 < sg.s1) {  // (a segment that stops mid-chain leaves x in x_io for the cluster that continues)
#ifdef DPB_TC_PROFILE_TAIL
              PROF_WAIT(2, write_xa<PDP>(xa_base, r_in, c0, x));
              PROF_WAIT(1, signal(xa_bar(sub)));
#else
              write_xa<PDP>(xa_base, r_in, c0, x);
              signal(xa_bar(sub));
#endif
            }
          } else {  // prior loss
            float acc = 0.f;
            if (valid) {
              float z[TCOLS];
              draw_cols<PDP>(p.z, row, c0, p.seed, (uint32_t)p.step_offset, 3, z);
              float racc = 0.f;
#pragma unroll
              for (int i = 0; i < TCOLS; ++i) {
                int col = c0 + i;
                if (col < D) {
                  float x0 = p.x_in[row * D + col];
                  float xt = p.alpha * x0 + p.sd * z[i];
                  float score = -raw[i] * p.inv_sigma_std;
                  float x0h = (xt + (p.sd * p.sd) * score) / p.alpha;
                  float d = x0 - x0h;
                  racc = fmaf(p.wgt * d, d, racc);
                  if (p.grad_out) p.grad_out[row * D + col] = 2.0f * p.wgt * d * p.inv_div;
                }
              }
              acc = racc;
              if (p.row_loss) atomicAdd(p.row_loss + row, acc);
            }
            for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
            if (lane == 0) atomicAdd(p.loss_out, acc * p.inv_div);
          }
          PROF_END(3, tail_t0)
        }
      }
      if (sg.publish) {  // first part of a cut chain: x_io rows of this tile are final for step s1
        __threadfence();
        ptx::named_bar_sync(1, EPI_THREADS);
        if (et == 0) ptx::st_release_gpu(p.flags + (size_t)worker * CLUSTER + crank, 1);
      }
    }
  }
  PROF_FLUSH();
  __syncthreads();
  if (CLUSTER > 1) ptx::cluster_sync();  // no CTA leaves while a peer may still multicast into it / arrive on its barriers
  if (warp == 2) {
    ptx::tc_fence_after();
    if (TWO_SM) ptx::tmem_dealloc_2sm(tmem_base, 512);
    else ptx::tmem_dealloc(tmem_base, 512);
  }
}

}  // namespace tc

// ------------------------------------------------------------------ host side
static PFN_cuTensorMapEncodeTiled_v12000 encode_fn() {
  static PFN_cuTensorMapEncodeTiled_v12000 fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<PFN_cuTensorMapEncodeTiled_v12000>(p);
  }
  return fn;
}

// 2-D row-major [rows, inner] 16-bit tensor, box {box_inner, box_rows}, 128-byte swizzle
int make_tmap_2d(CUtensorMap* m, CUtensorMapDataType dt, const void* ptr, uint64_t inner, uint64_t rows,
                 uint32_t box_inner, uint32_t box_rows, size_t elem_bytes) {
  auto enc = encode_fn();
  if (!enc) return fail(DPB_ECUDA, "cuTensorMapEncodeTiled is unavailable from the driver");
  cuuint64_t dims[2] = {inner, rows};
  cuuint64_t strides[1] = {inner * elem_bytes};
  cuuint32_t box[2] = {box_inner, box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = enc(m, dt, 2, const_cast<void*>(ptr), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                   CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail(DPB_ECUDA, "cuTensorMapEncodeTiled failed with code " + std::to_string((int)r));
  return DPB_OK;
}

int tc_prepare(dpb_score* h, const dpb_score_weights* w) {
  h->tc_ready = false;
  const int hd = h->pose_dim, hdp = h->pose_dp, xa_k = 3 * hdp;
  // fp16 copies of the square layers and post_dense (zero rows D..DP-1), bf16 hi/hi/lo split of pre_dense
  std::vector<__half> buf((size_t)H * H);
  for (int l = 0; l < 4; ++l) {
    for (size_t i = 0; i < (size_t)H * H; ++i) buf[i] = __float2half_rn(w->blk_w[l][i]);
    DPB_CUDA_CHECK(cudaMalloc((void**)&h->w16[l], buf.size() * sizeof(__half)));
    DPB_CUDA_CHECK(cudaMemcpy(h->w16[l], buf.data(), buf.size() * sizeof(__half), cudaMemcpyHostToDevice));
  }
  std::vector<__half> post((size_t)hdp * H, __float2half_rn(0.f));
  for (size_t i = 0; i < (size_t)hd * H; ++i) post[i] = __float2half_rn(w->post_w[i]);
  DPB_CUDA_CHECK(cudaMalloc((void**)&h->post16, post.size() * sizeof(__half)));
  DPB_CUDA_CHECK(cudaMemcpy(h->post16, post.data(), post.size() * sizeof(__half), cudaMemcpyHostToDevice));
  std::vector<__nv_bfloat16> pre((size_t)H * xa_k, __float2bfloat16_rn(0.f));
  for (int o = 0; o < H; ++o)
    for (int k = 0; k < hd; ++k) {
      float v = w->pre_w[(size_t)o * hd + k];
      __nv_bfloat16 hi = __float2bfloat16_rn(v);
      __nv_bfloat16 lo = __float2bfloat16_rn(v - __bfloat162float(hi));
      pre[(size_t)o * xa_k + k] = hi;             // pairs with x_hi
      pre[(size_t)o * xa_k + hdp + k] = hi;       // pairs with x_lo
      pre[(size_t)o * xa_k + 2 * hdp + k] = lo;   // pairs with x_hi
    }
  DPB_CUDA_CHECK(cudaMalloc((void**)&h->pre_split, pre.size() * sizeof(__nv_bfloat16)));
  DPB_CUDA_CHECK(cudaMemcpy(h->pre_split, pre.data(), pre.size() * sizeof(__nv_bfloat16), cudaMemcpyHostToDevice));
  // per-CTA activation scratch (one 128-row slot per SM)
  h->tc_slots = h->sm_count * tc::NSUB;
  const size_t rows = (size_t)h->tc_slots * tc::TILE_M;
  DPB_CUDA_CHECK(cudaMalloc((void**)&h->act_h, 2 * rows * H * sizeof(__half)));
  h->act_t = h->act_h + rows * H;
  DPB_CUDA_CHECK(cudaMemset(h->act_h, 0, 2 * rows * H * sizeof(__half)));
  // The scratch is written and re-read once per layer and never needed in HBM.  A persisting-L2 carve-out with an
  // access-policy window on the launch measured slower (profiles/r2_sampler_l2_policy.md: 565 vs 535 ms), so L2 is
  // left to the hardware policy plus evict_last hints on the scratch traffic.
  {  // gamma | beta of the five GroupNorms as the epilogue stages them (beta halved for the tanh-form SiLU)
    std::vector<float> gn((size_t)NL * 2 * H);
    DPB_CUDA_CHECK(cudaMemcpy(gn.data(), h->gn_packed, gn.size() * sizeof(float), cudaMemcpyDeviceToHost));
#if DPB_SILU_MODE == 2
    for (int l = 0; l < NL; ++l)
      for (int c = 0; c < H; ++c) gn[((size_t)l * 2 + 1) * H + c] *= 0.5f;
#endif
    DPB_CUDA_CHECK(cudaMalloc((void**)&h->gn_tc, gn.size() * sizeof(float)));
    DPB_CUDA_CHECK(cudaMemcpy(h->gn_tc, gn.data(), gn.size() * sizeof(float), cudaMemcpyHostToDevice));
  }
  DPB_CUDA_CHECK(cudaMalloc((void**)&h->tc_flags, sizeof(int) * h->tc_slots));
  DPB_CUDA_CHECK(cudaMemset(h->tc_flags, 0, sizeof(int) * h->tc_slots));
  int rc = DPB_OK;
  for (int l = 0; l < 4 && rc == DPB_OK; ++l)
    rc = make_tmap_2d(&h->tm_w[l], CU_TENSOR_MAP_DATA_TYPE_FLOAT16, h->w16[l], H, H, tc::BLOCK_K,
                      tc::CHUNK_N / tc::CLUSTER, 2);
  if (rc == DPB_OK) rc = make_tmap_2d(&h->tm_post, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, h->post16, H, hdp, tc::BLOCK_K,
                                    hdp / tc::CLUSTER, 2);
  if (rc == DPB_OK)
    rc = make_tmap_2d(&h->tm_pre, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, h->pre_split, xa_k, H, tc::BLOCK_K,
                      tc::CHUNK_N / tc::CLUSTER, 2);
  if (rc == DPB_OK)
    rc = make_tmap_2d(&h->tm_act_h, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, h->act_h, H, rows, tc::BLOCK_K, tc::TILE_M, 2);
  if (rc == DPB_OK)
    rc = make_tmap_2d(&h->tm_act_t, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, h->act_t, H, rows, tc::BLOCK_K, tc::TILE_M, 2);
  if (rc != DPB_OK) return rc;
  if (hdp == DP128)
    DPB_CUDA_CHECK(cudaFuncSetAttribute(tc::score_tc_kernel<DP128>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                        tc::Width<DP128>::SMEM_BYTES));
  else
    DPB_CUDA_CHECK(cudaFuncSetAttribute(tc::score_tc_kernel<DP>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                        tc::Width<DP>::SMEM_BYTES));
  DPB_CUDA_CHECK(cudaMalloc((void**)&h->pc_buf, (2 * PC_MAX_STEPS + 4) * sizeof(float)));
  h->tc_ready = true;
  return DPB_OK;
}

// the fused predictor-corrector mode needs every CTA to own one tile for the whole run (grid-wide norms per step)
bool tc_pc_possible(const dpb_score* h, int64_t B, int n_steps) {
  if (!h->tc_ready || !h->pc_buf || n_steps > PC_MAX_STEPS) return false;
  const int64_t n_tiles = (B + tc::TILE_M - 1) / tc::TILE_M;
  const int64_t max_grid = (h->tc_slots / tc::NSUB) / tc::CLUSTER * tc::CLUSTER;
  return (n_tiles + tc::CLUSTER - 1) / tc::CLUSTER * tc::CLUSTER <= max_grid;
}

void tc_release(dpb_score* h) {
  void* ptrs[] = {h->w16[0], h->w16[1], h->w16[2], h->w16[3], h->post16, h->pre_split, h->act_h, h->tc_flags, h->gn_tc, h->pc_buf};
  for (void* p : ptrs)
    if (p) cudaFree(p);
  h->tc_ready = false;
}

int tc_launch(dpb_score* h, const TcJob& j, cudaStream_t st) {
  tc::KParams p{};
  p.mode = j.mode;
  p.n_steps = j.pc ? 2 * j.n_steps : j.n_steps;
  p.pc = j.pc;
  p.snr = j.snr;
  p.pc_sums = h->pc_buf;
  p.pc_counter = reinterpret_cast<int*>(h->pc_buf + 2 * PC_MAX_STEPS);
  if (j.pc) DPB_CUDA_CHECK(cudaMemsetAsync(h->pc_buf, 0, (2 * PC_MAX_STEPS + 4) * sizeof(float), st));
  p.impute = j.impute;
  p.noise_k = j.noise_k;
  p.B = j.B;
  p.n_tiles = (int)((j.B + tc::TILE_M - 1) / tc::TILE_M);
  p.x_in = j.x_in; p.x_io = j.x_io; p.table = j.table; p.coef = j.coef;
  p.gn = h->gn_tc; p.post_b = h->post_b;
  p.row_scale = j.row_scale; p.scale = j.scale; p.out = j.out;
  p.obs = j.obs; p.mask = j.mask; p.noise = j.noise;
  p.seed = j.seed; p.step_offset = j.step_offset; p.traj = j.traj; p.x_mean = j.x_mean;
  p.alpha = j.alpha; p.sd = j.std; p.inv_sigma_std = j.inv_sigma_std;
  p.inv_div = j.divisor > 0.f ? 1.0f / j.divisor : 0.f;
  p.wgt = j.scale;  // prior loss: api.cu passes the weight through `scale`
  p.z = j.z; p.loss_out = j.loss_out; p.grad_out = j.grad_out; p.row_loss = j.row_loss;
  p.act_h = h->act_h; p.act_t = h->act_t;
  p.flags = h->tc_flags;
#if defined(DPB_TC_PROFILE) || defined(DPB_TC_KNOBS)
  {
    const char* dbg = getenv("DPB_TC_DEBUG");
    p.debug = dbg ? atoi(dbg) : 0;
  }
#endif
  if (j.mode == 2 && j.row_loss) DPB_CUDA_CHECK(cudaMemsetAsync(j.row_loss, 0, sizeof(float) * j.B, st));
  // grid: a multiple of the cluster size, at most one CTA per scratch slot
  const int n_groups = (p.n_tiles + tc::NSUB - 1) / tc::NSUB;
  int grid = (n_groups + tc::CLUSTER - 1) / tc::CLUSTER * tc::CLUSTER;
  const int max_grid = (h->tc_slots / tc::NSUB) / tc::CLUSTER * tc::CLUSTER;
  if (grid > max_grid) grid = max_grid;
  if (j.n_steps > 1) DPB_CUDA_CHECK(cudaMemsetAsync(h->tc_flags, 0, sizeof(int) * h->tc_slots, st));
  {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)grid);
    cfg.blockDim = dim3(tc::NUM_THREADS);
    cfg.dynamicSmemBytes = h->pose_dp == DP128 ? tc::Width<DP128>::SMEM_BYTES : tc::Width<DP>::SMEM_BYTES;
    cfg.stream = st;
    if (h->pose_dp == DP128)
      DPB_CUDA_CHECK(cudaLaunchKernelEx(&cfg, tc::score_tc_kernel<DP128>, p, h->tm_act_h, h->tm_act_t, h->tm_pre,
                                        h->tm_w[0], h->tm_w[1], h->tm_w[2], h->tm_w[3], h->tm_post));
    else
      DPB_CUDA_CHECK(cudaLaunchKernelEx(&cfg, tc::score_tc_kernel<DP>, p, h->tm_act_h, h->tm_act_t, h->tm_pre, h->tm_w[0],
                                        h->tm_w[1], h->tm_w[2], h->tm_w[3], h->tm_post));
  }
  DPB_CUDA_CHECK(cudaGetLastError());
#ifdef DPB_TC_PROFILE
  {
    cudaStreamSynchronize(st);
    std::vector<long long> hp((size_t)grid * 20 * 5);
    cudaMemcpyFromSymbol(hp.data(), tc::g_prof, hp.size() * sizeof(long long));
    static const char* names[5] = {"W-producer", "MMA", "A-producer", "store", "epi"};
    double acc[5][5] = {};
    int cnt[5] = {};
    for (int b = 0; b < grid; ++b)
      for (int w = 0; w < 20; ++w) {
        if (w == 1 && (b & 1)) continue;  // the MMA warp of the non-leader CTA is idle
        const int r = w < 4 ? w : 4;
        for (int k = 0; k < 5; ++k) acc[r][k] += (double)hp[((size_t)b * 20 + w) * 5 + k];
        ++cnt[r];
      }
    for (int r = 0; r < 5; ++r)
      fprintf(stderr, "[tc-prof] %-10s total %.0f  wait0 %.3f wait1 %.3f wait2 %.3f wait3 %.3f (fractions of total)\n",
              names[r], acc[r][4] / cnt[r], acc[r][0] / acc[r][4], acc[r][1] / acc[r][4], acc[r][2] / acc[r][4],
              acc[r][3] / acc[r][4]);
  }
#endif
  return DPB_OK;
}

}  // namespace dpb
