// Fused LBS forward, third generation: blend + skinning in ONE tcgen05 kernel on CTA pairs (cta_group::2) for SMPL and
// (with the constant hand / face tail folded away) SMPL-X.  Replaces smplx 0.1.28 lbs() as called from
// lib/body_model/body_model.py:75-88 and lib/body_model/smpl.py:67-78 (SURVEY.md App. A.6).
//
// What bounds this kernel family (profiles/r2_lbs_fused3_experiments.md): with every MMA, TMEM load and store removed,
// the TMA / barrier skeleton of an 80-pose-group kernel alone takes 1.5 ms for 65 536 SMPL poses -- 18.4 GB of operand
// tiles from L2 at the chip's ~12 TB/s TMA limit, 80 % of it the blend basis, which every CTA re-streams for every pose
// group (672 KB per tile pair and group).  MMAs add 0.4 ms and the 5.4 GB of vertex stores 1.0 ms on the same L2 fabric.
// The per-chunk issue chain that the second-generation kernel (lbs_fused2.cu) suffered from is NOT the limiter.  Changes:
//   * 128-pose groups: the basis bytes per pose drop by 1.6x (N = 128 blend MMAs); D_x | D_y | D_z take 384 TMEM columns,
//     leaving TWO 64-column T buffers (5 poses x 12 entries), one per issuing warp -- no cross-issuer protocol.
//   * buffer, stage and parities come from one running chunk counter with power-of-two arithmetic (no divisions, no
//     progress flags); 26 chunks per tile, the last one holds 3 poses.
//   * 16 epilogue warps in two sets (set = T buffer); the two warps of a set that share a TMEM lane quarter split a
//     chunk's poses 3 + 2, so a buffer is drained by 8 warps at once and released sooner.
//
//   warp 0  TMA: pose-group operand F (per group), blend-basis slabs (ring)        [both CTAs, own tile / own half]
//   warp 3  TMA: skinning weights (per tile, double buffered), transform chunks (ring)
//   warp 1  MMA issuer: blend + even chunks (T buffer 0, leader CTA);  warp 2  TMEM allocator + odd chunks (T buffer 1)
//   warps 4-19 epilogue: set = ((warp - 4) / 4) % 2 = T buffer, pose half = (warp - 4) / 8, TMEM lane quarter = warp % 4
#include <cudaTypedefs.h>

#include <cstdlib>

#include "lbs.h"
#include "ptx.cuh"

namespace dpb {

int make_tmap_2d(CUtensorMap* m, CUtensorMapDataType dt, const void* ptr, uint64_t inner, uint64_t rows,
                 uint32_t box_inner, uint32_t box_rows, size_t elem_bytes);  // score_tc.cu

namespace lt3 {

constexpr int TILE_V = 128;
constexpr int BK = 64;
constexpr int A_SLAB = TILE_V * BK * 2;        // 16 KB: [128 rows x 64 k] fp16, SWIZZLE_128B
constexpr int NP = 128;                        // poses per group = N of the blend MMAs
constexpr int CP = 5;                          // poses per skinning chunk
constexpr int NS = 64;                         // N of the skinning MMAs (CP * 12 = 60 used)
constexpr int NCH = (NP + CP - 1) / CP;        // 26 chunks per group (the last one holds 3 poses)
constexpr int NT = 2;                          // T buffers = issuing warps = epilogue warp sets
constexpr int NUM_THREADS = 128 + 16 * 32;     // 640
constexpr int F_SLAB = (NP / 2) * BK * 2;      // 8 KB: a CTA's half of the group's poses x 64 k
constexpr int S_SLAB = (NS / 2) * BK * 2;      // 4 KB: a CTA's half of the chunk's transform rows x 64 k
constexpr int T_COL0 = 3 * NP;                 // 384: first T column
// setmaxnreg moves registers inside the CTA's launch allocation (640 x 96): 128 * 64 + 512 * 104 = 61440
constexpr int ROLE_REGS = 64, EPI_REGS = 104;
static_assert(NCH % NT == 0, "a chunk's buffer is its running number modulo NT, tile after tile");
static_assert(T_COL0 + NT * NS <= 512 && F_SLAB % 1024 == 0 && S_SLAB % 1024 == 0, "TMEM / SWIZZLE_128B layout");
static_assert(NP % 16 == 0 && NS % 16 == 0, "cta_group::2 MMAs take N in steps of 16");

struct Params {
  int V, V_pad, n_tp;        // vertices, padded vertices, tile PAIRS
  int64_t B;
  long long n_items;         // pose groups x tile pairs
  float* verts;              // [B,V,3]
  int debug;                 // timing experiments only (DPB_LBS_DEBUG; results are garbage): 1 = epilogue loads T / D but
                             // skips math + stores, 2 = no blend MMAs, 4 = one skinning MMA per chunk, 8 = no TMEM loads;
                             // 16 / 32 keep the results: 16 = no L2::evict_last on basis / weight loads, 32 = plain
                             // (not st.global.cs) vertex stores
};

template <int JSLABS, int ASTAGES, int SSTAGES>
struct Smem {
  static constexpr int NSLABS_MAX = 7;
  static constexpr int OFF_F = 0;
  static constexpr int OFF_A = OFF_F + NSLABS_MAX * F_SLAB;                 // 57344 (1024-aligned)
  static constexpr int OFF_W = OFF_A + ASTAGES * A_SLAB;
  static constexpr int OFF_S = OFF_W + 2 * JSLABS * A_SLAB;
  static constexpr int OFF_BAR = OFF_S + SSTAGES * JSLABS * S_SLAB;
  static constexpr int NBARS = 2 * ASTAGES + 2 * SSTAGES + 4 + 2 + 2 + 2 * NT;
  static constexpr int BYTES = OFF_BAR + NBARS * 8 + 16 + 1024;             // + tmem slot + alignment slack
  static_assert(OFF_A % 1024 == 0 && OFF_W % 1024 == 0 && OFF_S % 1024 == 0, "operand tiles are 1024-byte aligned");
  static_assert(BYTES <= 232448, "exceeds the 227 KB per-CTA shared memory limit");
  static_assert((SSTAGES & (SSTAGES - 1)) == 0 && SSTAGES % NT == 0, "stage = running chunk number & (SSTAGES - 1)");
};

// KH16 = K16 steps of the hi half of the blend K, NSLABS = 64-wide slabs of [hi | lo]; JS = K16 steps of the hi half of
// the skinning K (joints + translation slot, padded), JSLABS = its 64-wide slabs.
template <int KH16, int NSLABS, int JS, int JSLABS, int ASTAGES, int SSTAGES>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(NUM_THREADS, 1)
lbs_fused3_kernel(const __grid_constant__ Params p, const __grid_constant__ CUtensorMap tm_dirs,
                  const __grid_constant__ CUtensorMap tm_feat, const __grid_constant__ CUtensorMap tm_w,
                  const __grid_constant__ CUtensorMap tm_s) {
  using L = Smem<JSLABS, ASTAGES, SSTAGES>;
  constexpr uint32_t IDESC_BLEND = ptx::umma_idesc_f16(2 * TILE_V, NP, 0);
  constexpr uint32_t IDESC_SKIN = ptx::umma_idesc_f16(2 * TILE_V, NS, 0);
  static_assert(NSLABS <= L::NSLABS_MAX && 2 * KH16 <= 4 * NSLABS && 2 * JS <= 4 * JSLABS, "K geometry");
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (ptx::smem_u32(smem_raw) & 1023u)) & 1023u);
  const uint32_t sb = ptx::smem_u32(smem);
  const uint32_t f_base = sb + L::OFF_F, a_base = sb + L::OFF_A, w_base = sb + L::OFF_W, s_base = sb + L::OFF_S;
  const uint32_t bar = sb + L::OFF_BAR;
  auto afull = [&](uint32_t s) { return bar + 8u * s; };
  auto aempty = [&](uint32_t s) { return bar + 8u * (ASTAGES + s); };
  auto sfull = [&](uint32_t s) { return bar + 8u * (2 * ASTAGES + s); };
  auto sempty = [&](uint32_t s) { return bar + 8u * (2 * ASTAGES + SSTAGES + s); };
  const uint32_t b2 = bar + 8u * (2 * ASTAGES + 2 * SSTAGES);
  auto wfull = [&](uint32_t b) { return b2 + 8u * b; };
  auto wempty = [&](uint32_t b) { return b2 + 8u * (2 + b); };
  const uint32_t ffull = b2 + 32, fempty = b2 + 40, dfull = b2 + 48, dempty = b2 + 56;
  auto tfull = [&](uint32_t b) { return b2 + 64 + 8u * b; };
  auto tempty = [&](uint32_t b) { return b2 + 64 + 8u * (NT + b); };
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + L::OFF_BAR + L::NBARS * 8);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 0) {
    // "full" barriers are waited on by the pair's leader only and collect one arrive.expect_tx from EACH CTA's
    // producer; "empty" / TMEM-full barriers exist in both CTAs and are signalled by multicast tcgen05.commit
    for (int s = 0; s < ASTAGES; ++s) { ptx::mbar_init(afull(s), 2); ptx::mbar_init(aempty(s), 1); }
    for (int s = 0; s < SSTAGES; ++s) { ptx::mbar_init(sfull(s), 2); ptx::mbar_init(sempty(s), 1); }
    for (int b = 0; b < 2; ++b) { ptx::mbar_init(wfull(b), 2); ptx::mbar_init(wempty(b), 2); }   // wempty: both issuers commit
    ptx::mbar_init(ffull, 2); ptx::mbar_init(fempty, 1);
    ptx::mbar_init(dfull, 1); ptx::mbar_init(dempty, 2 * 16);                // every epilogue warp of both CTAs
    for (int b = 0; b < NT; ++b) { ptx::mbar_init(tfull(b), 1); ptx::mbar_init(tempty(b), 2 * 16 / NT); }  // one set, both CTAs
    ptx::fence_barrier_init();
  }
  if (warp == 2) ptx::tmem_alloc_2sm(ptx::smem_u32(tmem_slot), 512);
  ptx::tc_fence_before();
  __syncthreads();
  ptx::cluster_sync();       // the peer's barriers are initialised before anyone arrives on them remotely
  ptx::tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const uint32_t crank = ptx::cluster_ctarank();
  constexpr uint16_t CMASK = 3;
  const long long worker = blockIdx.x >> 1, n_workers = gridDim.x >> 1;
  auto expect = [&](uint32_t fullbar, uint32_t bytes) { ptx::mbar_arrive_expect_tx_cluster(ptx::mapa(fullbar, 0), bytes); };
  auto load = [&](uint32_t dst, const CUtensorMap* tm, uint32_t fullbar, int c0, int c1) {
    ptx::tma_load_2d_2sm(dst, tm, ptx::mapa(fullbar, 0), c0, c1);
  };
  // operands every pose group re-reads (blend basis, skinning weights) load with L2::evict_last, the write-once vertices
  // leave with st.global.cs: 3.14 -> 3.06 ms per 65 536 SMPL poses, bit-identical (p.debug & 16 / & 32 switch them off, A/B)
  const bool keep_hint = (p.debug & 16) == 0;
  const uint64_t keep_pol = ptx::l2_policy_evict_last();
  auto load_keep = [&](uint32_t dst, const CUtensorMap* tm, uint32_t fullbar, int c0, int c1) {
    if (keep_hint) ptx::tma_load_2d_2sm_hint(dst, tm, ptx::mapa(fullbar, 0), c0, c1, keep_pol);
    else ptx::tma_load_2d_2sm(dst, tm, ptx::mapa(fullbar, 0), c0, c1);
  };
  const long long i0 = p.n_items * worker / n_workers, i1 = p.n_items * (worker + 1) / n_workers;
  const int n_my = (int)(i1 - i0);                 // items of this pair
  const int grp0 = (int)(i0 / p.n_tp), tp0 = (int)(i0 % p.n_tp);
  auto advance = [&](int& grp, int& tp) { if (++tp == p.n_tp) { tp = 0; ++grp; } };

  // chunks first, first + 2, ... of tile number tc (this worker's count): T[v, (pose, e)] = sum_j w[v,j] A[pose,j,e].
  // gc = running chunk number of this worker; buffer = gc % NT (= first: NCH is even), stage = gc % SSTAGES.
  auto skin_chunks = [&](uint32_t tc, uint32_t first) {
    const uint32_t wb = tc & 1;
    ptx::mbar_wait(wfull(wb), (tc >> 1) & 1);
    ptx::tc_fence_after();
    const uint64_t wdesc0 = ptx::umma_desc_sw128(w_base + wb * JSLABS * A_SLAB);
    const uint64_t sdesc0 = ptx::umma_desc_sw128(s_base);
    const uint32_t taddr = tmem_base + T_COL0 + first * NS;
    auto wdesc = [&](int step) { return wdesc0 + (uint64_t)((step >> 2) * (A_SLAB >> 4) + 2 * (step & 3)); };
#pragma unroll 1
    for (uint32_t ch = first; ch < NCH; ch += NT) {
      const uint32_t gc = tc * NCH + ch, sstage = gc & (SSTAGES - 1), use = gc / NT;
      ptx::mbar_wait(tempty(first), (use & 1) ^ 1u);              // the set has read this buffer's previous chunk
      ptx::mbar_wait(sfull(sstage), (gc / SSTAGES) & 1);
      ptx::tc_fence_after();
      const uint64_t sd = sdesc0 + (uint64_t)(sstage * (JSLABS * (S_SLAB >> 4)));
      auto sdesc = [&](int step) { return sd + (uint64_t)((step >> 2) * (S_SLAB >> 4) + 2 * (step & 3)); };
      if (ptx::elect_one()) {
#pragma unroll
        for (int g = 0; g < JS; ++g) {   // w_hi x (A_hi + A_lo), then w_lo x A_hi
          ptx::mma_f16_ss_2sm(taddr, wdesc(g), sdesc(g), IDESC_SKIN, g ? 1u : 0u);
          if (p.debug & 4) break;
          ptx::mma_f16_ss_2sm(taddr, wdesc(g), sdesc(JS + g), IDESC_SKIN, 1u);
          ptx::mma_f16_ss_2sm(taddr, wdesc(JS + g), sdesc(g), IDESC_SKIN, 1u);
        }
        ptx::mma_commit_2sm_mcast(sempty(sstage), CMASK);
        ptx::mma_commit_2sm_mcast(tfull(first), CMASK);
      }
      __syncwarp();
    }
    if (ptx::elect_one()) ptx::mma_commit_2sm_mcast(wempty(wb), CMASK);   // this issuer's MMAs on the tile's weights are done
    __syncwarp();
  };

  if (warp < 4) {
    ptx::setmaxnreg_dec<ROLE_REGS>();
    if (warp == 0) {
      // ---- pose-group operand + blend-basis slabs
      if (lane == 0) { ptx::prefetch_tmap(&tm_dirs); ptx::prefetch_tmap(&tm_feat); }
      __syncwarp();
      uint32_t stage = 0, phase = 0, fph = 0;
      int grp = grp0, tp = tp0;
      for (int it = 0; it < n_my; ++it, advance(grp, tp)) {
        const int tile = 2 * tp + (int)crank;
        if (it == 0 || tp == 0) {
          ptx::mbar_wait(fempty, fph ^ 1);   // the previous group's blends are done with the operand
          fph ^= 1;
          if (ptx::elect_one()) {
            expect(ffull, NSLABS * F_SLAB);
#pragma unroll
            for (int i = 0; i < NSLABS; ++i)
              load(f_base + i * F_SLAB, &tm_feat, ffull, i * BK, grp * NP + (int)crank * (NP / 2));
          }
          __syncwarp();
        }
        for (int c = 0; c < 3; ++c)
#pragma unroll
          for (int i = 0; i < NSLABS; ++i) {
            ptx::mbar_wait(aempty(stage), phase ^ 1);
            if (ptx::elect_one()) {
              expect(afull(stage), A_SLAB);
              load_keep(a_base + stage * A_SLAB, &tm_dirs, afull(stage), i * BK, c * p.V_pad + tile * TILE_V);
            }
            __syncwarp();
            if (++stage == ASTAGES) { stage = 0; phase ^= 1; }
          }
      }
    } else if (warp == 3) {
      // ---- skinning weights (per tile) + transform chunks
      if (lane == 0) { ptx::prefetch_tmap(&tm_w); ptx::prefetch_tmap(&tm_s); }
      __syncwarp();
      uint32_t tc = 0;
      int grp = grp0, tp = tp0;
      for (int it = 0; it < n_my; ++it, ++tc, advance(grp, tp)) {
        const int tile = 2 * tp + (int)crank;
        const uint32_t wb = tc & 1;
        ptx::mbar_wait(wempty(wb), ((tc >> 1) & 1) ^ 1);
        if (ptx::elect_one()) {
          expect(wfull(wb), JSLABS * A_SLAB);
#pragma unroll
          for (int i = 0; i < JSLABS; ++i)
            load_keep(w_base + (wb * JSLABS + i) * A_SLAB, &tm_w, wfull(wb), i * BK, tile * TILE_V);
        }
        __syncwarp();
        const int row0 = grp * NP * 12 + (int)crank * (NS / 2);
#pragma unroll 1
        for (uint32_t ch = 0; ch < NCH; ++ch) {
          const uint32_t gc = tc * NCH + ch, stage = gc & (SSTAGES - 1);
          ptx::mbar_wait(sempty(stage), ((gc / SSTAGES) & 1) ^ 1u);
          if (ptx::elect_one()) {
            expect(sfull(stage), JSLABS * S_SLAB);
#pragma unroll
            for (int i = 0; i < JSLABS; ++i)
              load(s_base + (stage * JSLABS + i) * S_SLAB, &tm_s, sfull(stage), i * BK, row0 + (int)ch * CP * 12);
          }
          __syncwarp();
        }
      }
    } else if (warp == 1 && crank == 0) {
      // ---- MMA issuer (the pair's leader issues for both CTAs; warp-wide loop, the elected lane issues)
      uint32_t astage = 0, aphase = 0, fph = 0, tc = 0;
      const uint64_t adesc0 = ptx::umma_desc_sw128(a_base), fdesc0 = ptx::umma_desc_sw128(f_base);
      auto fdesc = [&](int step) { return fdesc0 + (uint64_t)((step >> 2) * (F_SLAB >> 4) + 2 * (step & 3)); };
      int grp = grp0, tp = tp0;
      for (int it = 0; it < n_my; ++it, ++tc, advance(grp, tp)) {
        if (it == 0 || tp == 0) {
          ptx::mbar_wait(ffull, fph);
          fph ^= 1;
        }
        ptx::mbar_wait(dempty, (tc & 1) ^ 1);   // both CTAs' epilogues have read all of the previous tile's D
        ptx::tc_fence_after();
        const bool last_of_group = (it == n_my - 1) || (tp == p.n_tp - 1);
#pragma unroll 1
        for (int c = 0; c < 3; ++c) {
          const uint32_t taddr = tmem_base + c * NP;
#pragma unroll
          for (int i = 0; i < NSLABS; ++i) {
            ptx::mbar_wait(afull(astage), aphase);
            ptx::tc_fence_after();
            const uint64_t adesc = adesc0 + (uint64_t)(astage * (A_SLAB >> 4));
            if (ptx::elect_one()) {
#pragma unroll
              for (int j = 0; j < BK / 16; ++j) {
                const int g = i * (BK / 16) + j;   // K16 step inside [hi | lo], compile-time after unrolling
                if (p.debug & 2) continue;
                if (g < KH16) {                    // basis_hi x (feat_hi + feat_lo)
                  ptx::mma_f16_ss_2sm(taddr, adesc + 2 * j, fdesc(g), IDESC_BLEND, g != 0 ? 1u : 0u);
                  ptx::mma_f16_ss_2sm(taddr, adesc + 2 * j, fdesc(KH16 + g), IDESC_BLEND, 1u);
                } else if (g < 2 * KH16) {         // basis_lo x feat_hi
                  ptx::mma_f16_ss_2sm(taddr, adesc + 2 * j, fdesc(g - KH16), IDESC_BLEND, 1u);
                }
              }
              ptx::mma_commit_2sm_mcast(aempty(astage), CMASK);
              if (c == 2 && i == NSLABS - 1) {
                ptx::mma_commit_2sm_mcast(dfull, CMASK);
                if (last_of_group) ptx::mma_commit_2sm_mcast(fempty, CMASK);
              }
            }
            __syncwarp();
            if (++astage == ASTAGES) { astage = 0; aphase ^= 1; }
          }
        }
        skin_chunks(tc, 0u);
      }
    } else if (warp == 2 && crank == 0) {
      // ---- second skinning issuer (odd chunks, T buffer 1).  It waits for the tile's blend: the sets consume a tile's
      // chunks only after dfull, and an early chunk must not hold a transform stage the first issuer's chunks wait for.
      for (uint32_t tc = 0; tc < (uint32_t)n_my; ++tc) {
        ptx::mbar_wait(dfull, tc & 1);
        skin_chunks(tc, 1u);
      }
    }
  } else {
    // ---- epilogue: thread = vertex.  The chunk's T columns and (x,y,z) of D -> skinned vertex -> store.  The two warps
    // of a set on the same TMEM lane quarter take poses 0-2 / 3-4 of every chunk.
    ptx::setmaxnreg_inc<EPI_REGS>();
    const int q4 = warp & 3;
    const int set = ((warp - 4) >> 2) & 1, half = (warp - 4) >> 3;
    const int i_lo = half ? 3 : 0, n_i = half ? 2 : 3;           // this warp's poses within a chunk
    const uint32_t lane_addr = (uint32_t)(q4 * 32) << 16;
    const size_t pstride = (size_t)p.V * 3;
    const uint32_t l_tempty = ptx::mapa(tempty(set), 0), l_dempty = ptx::mapa(dempty, 0);
    const uint32_t my_tfull = tfull(set);
    const uint32_t t_addr = tmem_base + lane_addr + T_COL0 + set * NS + i_lo * 12;
    uint32_t tc = 0;
    int grp = grp0, tp = tp0;
    for (int it = 0; it < n_my; ++it, ++tc, advance(grp, tp)) {
      const int tile = 2 * tp + (int)crank;
      const int v = tile * TILE_V + q4 * 32 + lane;
      ptx::mbar_wait(dfull, tc & 1);
      ptx::tc_fence_after();
#pragma unroll 1
      for (int ch = set; ch < NCH; ch += NT) {
        const uint32_t use = (tc * NCH + ch) / NT;
        ptx::mbar_wait(my_tfull, use & 1);
        ptx::tc_fence_after();
        uint32_t t[36], d[3][4];
        const uint32_t d0 = tmem_base + lane_addr + ch * CP + i_lo;
        if (!(p.debug & 8)) {
          if (half == 0) {                       // poses 0-2: columns 0-35;  poses 3-4: columns 36-59 (warp-uniform)
            ptx::tmem_ld_32x32(t_addr, t);
            ptx::tmem_ld_32x4(t_addr + 32, t + 32);
          } else {
            ptx::tmem_ld_32x16(t_addr, t);
            ptx::tmem_ld_32x8(t_addr + 16, t + 16);
          }
          ptx::tmem_ld_32x4(d0, d[0]);
          ptx::tmem_ld_32x4(d0 + NP, d[1]);
          ptx::tmem_ld_32x4(d0 + 2 * NP, d[2]);
          ptx::tmem_ld_wait();
        } else {
#pragma unroll
          for (int i = 0; i < 36; ++i) t[i] = 0x3f800000u;
#pragma unroll
          for (int i = 0; i < 4; ++i) d[0][i] = d[1][i] = d[2][i] = 0x3f800000u + i;
        }
        ptx::tc_fence_before();
        __syncwarp();
        if (lane == 0) {
          ptx::mbar_arrive_cluster(l_tempty);
          if (ch + NT >= NCH) ptx::mbar_arrive_cluster(l_dempty);   // this warp's last read of the tile's D
        }
        const int64_t b0 = (int64_t)grp * NP + ch * CP + i_lo;
        int n_ok = min(n_i, NP - (ch * CP + i_lo));                   // poses of this warp inside the group ...
        if (b0 + n_ok > p.B) n_ok = (int)max((int64_t)0, p.B - b0);   // ... and inside the batch
        if (v < p.V && !(p.debug & 1)) {
          // each lane stores its vertex's 12 bytes; the warp's 32 records are one contiguous 384-byte run
          float* dst = p.verts + (size_t)b0 * pstride + (size_t)v * 3;
#pragma unroll
          for (int i = 0; i < 3; ++i) {
            const float* T = reinterpret_cast<const float*>(t) + i * 12;
            const float x = __uint_as_float(d[0][i]), y = __uint_as_float(d[1][i]), z = __uint_as_float(d[2][i]);
            const float ox = fmaf(T[0], x, fmaf(T[1], y, fmaf(T[2], z, T[9])));
            const float oy = fmaf(T[3], x, fmaf(T[4], y, fmaf(T[5], z, T[10])));
            const float oz = fmaf(T[6], x, fmaf(T[7], y, fmaf(T[8], z, T[11])));
            if (i < n_ok) {
              float* w = dst + (size_t)i * pstride;
              if (!(p.debug & 32)) { __stcs(w, ox); __stcs(w + 1, oy); __stcs(w + 2, oz); }   // streaming stores
              else { w[0] = ox; w[1] = oy; w[2] = oz; }
            }
          }
        }
      }
    }
  }
  ptx::tc_fence_before();
  __syncthreads();
  ptx::cluster_sync();       // no CTA leaves while the peer may still arrive on its barriers / read its operands
  if (warp == 2) {
    ptx::tc_fence_after();
    ptx::tmem_dealloc_2sm(tmem_base, 512);
  }
}

}  // namespace lt3

// One skinning K slab (jp = 32: SMPL).  Measured (profiles/r2_lbs_fused3_experiments.md): the 128-pose-group kernel
// wins there; lbs_fused2 wins for two slabs (jp = 64).
bool lbs_fused3_fits(const dpb_lbs* h, const LbsVariant& v) {
  if (!h->tc_ready || !v.dirs16) return false;
  if (v.kext != 448) return false;                      // instantiated for a 224-wide blend K (SMPL; SMPL-X const tail)
  if (h->J >= h->jp) return false;                      // needs the spare joint slot for the translation
  if (h->jp != 32) return false;
  if ((h->n_cols_pad / lt3::TILE_V) % 2) return false;  // whole tile pairs
  return true;
}

// verts[B,V,3] = skinned vertices.  featop [B_pad, kext] and skinop [B_pad*12, 2*jp] were written by the pose kernel.
int lbs_fused3(dpb_lbs* h, const LbsVariant& v, __half* featop, __half* skinop, float* verts, int64_t B,
               cudaStream_t st) {
  const int K2 = v.kext, Jp = h->jp;
  const int64_t B_pad = (B + 127) / 128 * 128;          // rows that physically exist (lbs_tc_ws_bytes); TMA zero-fills beyond
  CUtensorMap tm_feat, tm_s;
  int rc = make_tmap_2d(&tm_feat, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, featop, K2, (uint64_t)B_pad, lt3::BK, lt3::NP / 2, 2);
  if (rc == DPB_OK)
    rc = make_tmap_2d(&tm_s, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, skinop, 2 * Jp, (uint64_t)B_pad * 12, lt3::BK,
                      lt3::NS / 2, 2);
  if (rc != DPB_OK) return rc;
  lt3::Params p{};
  p.V = h->V;
  p.V_pad = h->n_cols_pad;
  p.n_tp = h->n_cols_pad / lt3::TILE_V / 2;
  p.B = B;
  p.n_items = (long long)((B + lt3::NP - 1) / lt3::NP) * p.n_tp;
  p.verts = verts;
  p.debug = getenv("DPB_LBS_DEBUG") ? atoi(getenv("DPB_LBS_DEBUG")) : 0;
  auto kern = lt3::lbs_fused3_kernel<14, 7, 2, 1, 6, 8>;   // F 56 KB + A 96 + W 32 + S 32
  const size_t smem = lt3::Smem<1, 6, 8>::BYTES;
  DPB_CUDA_CHECK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  int grid = h->sm_count & ~1;                                   // whole clusters of two
  const long long max_workers = p.n_items < 1 ? 1 : p.n_items;
  if (grid / 2 > max_workers) grid = (int)(2 * max_workers);
  kern<<<grid, lt3::NUM_THREADS, smem, st>>>(p, v.tm_dirs, tm_feat, h->tm_wop, tm_s);
  DPB_CUDA_CHECK(cudaGetLastError());
  return DPB_OK;
}

}  // namespace dpb
