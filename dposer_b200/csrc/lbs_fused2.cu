// Fused LBS forward, second generation: blend + skinning in ONE tcgen05 kernel on CTA PAIRS (cta_group::2), for
// SMPL and (with the constant hand / face tail folded away) SMPL-X.  Replaces smplx 0.1.28 lbs() as called from
// lib/body_model/body_model.py:75-88 and lib/body_model/smpl.py:67-78 (SURVEY.md App. A.6).
//
// Why a second kernel (profiles/r1_ncu_full_summary_final.md, the round-1 single-CTA fused kernel): tensor pipe 49 %
// active, the MMA warp waited 63 % of the time for a T buffer and the eight epilogue warps ran one dependent
// instruction every ~5 cycles.  The tensor work itself is fixed by the 3-product fp16 split (hi.hi + hi.lo + lo.hi),
// so the whole gap is overlap.  Changes:
//   * CTA pair, M = 256: each CTA keeps its own 128-vertex tile of the blend basis / skinning weights (A operands)
//     and only HALF of every pose-side B operand, so an N = 96 MMA fetches 32 + 12 cycles of shared memory for 48
//     cycles of math (N = 128 on one CTA: 32 + 32 for 64 -- the pipe and the epilogue's staging compete for the same
//     128 B/clk).  The pose operand of a group (48 rows) and a deep basis ring fit next to each other.
//   * 96 poses per group: D_x | D_y | D_z take 288 TMEM columns, leaving THREE 64-column T buffers (5 poses x 12
//     entries): the MMA -> epilogue -> MMA round trip (~650 cycles) is covered by two chunks in flight.
//   * 12 epilogue warps in three sets; a set owns every third chunk, so chunks are in their math / store tail
//     while the next ones are being loaded from TMEM.
//   * v_template rides in a spare K slot of the blend (feature = 1), the translation in the spare joint slot of the
//     skinning GEMM: the epilogue is 9 FFMA + 3 stores per (vertex, pose).
//   * work = (pose group, tile pair) items laid end to end and cut into equal contiguous pieces per CTA pair.
//
//   warp 0  TMA: pose-group operand F (per group), blend-basis slabs (ring)        [both CTAs, own tile / own half]
//   warp 3  TMA: skinning weights (per tile, double buffered), transform chunks (ring)
//   warp 1  MMA issuer (leader CTA only);   warp 2  TMEM allocator
//   warps 4-15 epilogue: set = (warp - 4) / 4, TMEM lane quarter = warp % 4, thread = vertex
#include <cudaTypedefs.h>

#include <cstdlib>

#include "lbs.h"
#include "ptx.cuh"

namespace dpb {

int make_tmap_2d(CUtensorMap* m, CUtensorMapDataType dt, const void* ptr, uint64_t inner, uint64_t rows,
                 uint32_t box_inner, uint32_t box_rows, size_t elem_bytes);  // score_tc.cu

namespace lt2 {

constexpr int TILE_V = 128;
constexpr int BK = 64;
constexpr int A_SLAB = TILE_V * BK * 2;        // 16 KB: [128 rows x 64 k] fp16, SWIZZLE_128B
constexpr int NP = 96;                         // poses per group = N of the blend MMAs
constexpr int CP = 5;                          // poses per skinning chunk
constexpr int NS = 64;                         // N of the skinning MMAs (CP * 12 = 60 used)
constexpr int NCH = (NP + CP - 1) / CP;        // 20 chunks per group (the last one holds a single pose)
constexpr int NT = 3;                          // T buffers
constexpr int NSETS = 3;                       // epilogue warp sets (12 warps: 84 TMEM values live per thread need ~150 registers)
constexpr int NUM_THREADS = 128 + NSETS * 128; // 512
// pose-side (B) operand tiles: each CTA of a pair (cta_group::2) holds half of the rows
constexpr int F_SLAB = NP / 2 * BK * 2;        // 6 KB: poses x 64 k
constexpr int S_SLAB = NS / 2 * BK * 2;        // 4 KB: transform rows x 64 k
constexpr int T_COL0 = 3 * NP;                 // 288: first T column
constexpr int ROLE_REGS = 72, EPI_REGS = 144;  // setmaxnreg: 128 * 72 + 384 * 144 <= 65536
static_assert(NCH >= NSETS, "every epilogue set handles at least one chunk per tile");
static_assert(T_COL0 + NT * NS <= 512 && F_SLAB % 1024 == 0 && S_SLAB % 1024 == 0, "TMEM / SWIZZLE_128B layout");

struct Params {
  int V, V_pad, n_tp;        // vertices, padded vertices, tile PAIRS (n_vt / 2)
  int64_t B;
  long long n_items;         // pose groups x tile pairs
  float* verts;              // [B,V,3]
  int debug;                 // timing experiments only (DPB_LBS_DEBUG): 1 = no stores, 2 = no TMEM load of T,
                             // 4 = no TMEM load of D, 16 = no skinning chunks, 32 = no blend (results are garbage)
};

template <int JSLABS, int ASTAGES, int SSTAGES, int WBUFS>
struct Smem {
  static constexpr int NSLABS_MAX = 7;
  static constexpr int OFF_F = 0;
  static constexpr int OFF_A = OFF_F + NSLABS_MAX * F_SLAB;                 // 43008 (1024-aligned)
  static constexpr int OFF_W = OFF_A + ASTAGES * A_SLAB;
  static constexpr int OFF_S = OFF_W + WBUFS * JSLABS * A_SLAB;
  static constexpr int OFF_BAR = OFF_S + SSTAGES * JSLABS * S_SLAB;
  static constexpr int NBARS = 2 * ASTAGES + 2 * SSTAGES + 4 + 2 + 2 + 2 * NT;
  static constexpr int BYTES = OFF_BAR + NBARS * 8 + 16 + 1024;             // + tmem slot + alignment slack
  static_assert(OFF_A % 1024 == 0 && OFF_W % 1024 == 0 && OFF_S % 1024 == 0, "operand tiles are 1024-byte aligned");
  static_assert(BYTES <= 232448, "exceeds the 227 KB per-CTA shared memory limit");
};

// KH16 = K16 steps of the hi half of the blend K, NSLABS = 64-wide slabs of [hi | lo]; JS = K16 steps of the hi half of
// the skinning K (joints + translation slot, padded), JSLABS = its 64-wide slabs.  Compile-time: the issuer's loops
// unroll and every descriptor is base + constant.  CTA pair with cta_group::2 MMAs: M = 256, pose-side operands split
// between the CTAs, the leader issues, barriers cross the pair.
template <int KH16, int NSLABS, int JS, int JSLABS, int ASTAGES, int SSTAGES, int WBUFS>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(NUM_THREADS, 1)
lbs_fused2_kernel(const __grid_constant__ Params p, const __grid_constant__ CUtensorMap tm_dirs,
                  const __grid_constant__ CUtensorMap tm_feat, const __grid_constant__ CUtensorMap tm_w,
                  const __grid_constant__ CUtensorMap tm_s) {
  using L = Smem<JSLABS, ASTAGES, SSTAGES, WBUFS>;
  constexpr uint32_t IDESC_BLEND = ptx::umma_idesc_f16(2 * TILE_V, NP, 0);
  constexpr uint32_t IDESC_SKIN = ptx::umma_idesc_f16(2 * TILE_V, NS, 0);
  constexpr int NC = 2;                          // CTAs that feed one MMA stream
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
  volatile uint32_t* issued = tmem_slot + 1;   // [2]: chunks (global count + 1) whose T-buffer wait each skin issuer has passed

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 0) {
    issued[0] = issued[1] = 0;
    // "full" barriers are waited on by the pair's leader only and collect one arrive.expect_tx from EACH CTA's
    // producer; "empty" / TMEM-full barriers exist in both CTAs and are signalled by multicast tcgen05.commit
    for (int s = 0; s < ASTAGES; ++s) { ptx::mbar_init(afull(s), NC); ptx::mbar_init(aempty(s), 1); }
    for (int s = 0; s < SSTAGES; ++s) { ptx::mbar_init(sfull(s), NC); ptx::mbar_init(sempty(s), 1); }
    for (int b = 0; b < 2; ++b) { ptx::mbar_init(wfull(b), NC); ptx::mbar_init(wempty(b), 2); }   // wempty: both skin issuers commit
    ptx::mbar_init(ffull, NC); ptx::mbar_init(fempty, 1);
    ptx::mbar_init(dfull, 1); ptx::mbar_init(dempty, NC * NSETS * 4);        // every epilogue warp (of both CTAs)
    for (int b = 0; b < NT; ++b) { ptx::mbar_init(tfull(b), 1); ptx::mbar_init(tempty(b), NC * 4); }  // one set (both CTAs)
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
  // both CTAs signal the leader's barriers; commits are multicast to the pair
  auto expect = [&](uint32_t fullbar, uint32_t bytes) { ptx::mbar_arrive_expect_tx_cluster(ptx::mapa(fullbar, 0), bytes); };
  auto load = [&](uint32_t dst, const CUtensorMap* tm, uint32_t fullbar, int c0, int c1) {
    ptx::tma_load_2d_2sm(dst, tm, ptx::mapa(fullbar, 0), c0, c1);
  };
  auto mma = [&](uint32_t taddr, uint64_t ad, uint64_t bd, uint32_t idesc, uint32_t acc) {
    ptx::mma_f16_ss_2sm(taddr, ad, bd, idesc, acc);
  };
  auto commit = [&](uint32_t b) { ptx::mma_commit_2sm_mcast(b, CMASK); };
  const long long i0 = p.n_items * worker / n_workers, i1 = p.n_items * (worker + 1) / n_workers;
  const int n_my = (int)(i1 - i0);                 // items of this pair
  const int grp0 = (int)(i0 / p.n_tp), tp0 = (int)(i0 % p.n_tp);
  // walk (group, tile pair) without a division per item
  auto advance = [&](int& grp, int& tp) { if (++tp == p.n_tp) { tp = 0; ++grp; } };

  // chunks first, first+2, ... of tile number tc (this worker's count): T[v, (pose, e)] = sum_j w[v,j] A[pose,j,e]
  auto skin_chunks = [&](uint32_t tc, int first) {
    const uint32_t wb = tc % WBUFS;
    ptx::mbar_wait(wfull(wb), (tc / WBUFS) & 1);
    ptx::tc_fence_after();
    const uint32_t wa = w_base + wb * JSLABS * A_SLAB;
    auto wdesc = [&](int step) { return ptx::umma_desc_sw128(wa + (step >> 2) * A_SLAB) + 2 * (step & 3); };
    const int nch = (p.debug & 16) ? 0 : NCH;
#pragma unroll 1
    for (int ch = first; ch < nch; ch += 2) {
      const uint32_t cc = tc * NCH + ch, buf = cc % NT, sstage = cc % SSTAGES;
      // A parity wait cannot tell "use k of the buffer drained" from "use k-2 drained": do not start waiting for this
      // use before the buffer's previous use (chunk cc - NT, the OTHER issuer's since NT is odd) got past its own wait.
      static_assert(NT % 2 == 1, "the buffer's previous use belongs to the other issuer");
      if (cc >= NT)
        while (issued[first ^ 1] < cc - NT + 1) {
        }
      ptx::mbar_wait(tempty(buf), ((cc / NT) & 1) ^ 1);
      if (lane == 0) issued[first] = cc + 1;
      ptx::mbar_wait(sfull(sstage), (cc / SSTAGES) & 1);
      ptx::tc_fence_after();
      const uint32_t taddr = tmem_base + T_COL0 + buf * NS;
      const uint32_t sa = s_base + sstage * JSLABS * S_SLAB;
      auto sdesc = [&](int step) { return ptx::umma_desc_sw128(sa + (step >> 2) * S_SLAB) + 2 * (step & 3); };
      if (ptx::elect_one()) {
#pragma unroll
        for (int g = 0; g < JS; ++g) {   // w_hi x (A_hi + A_lo), then w_lo x A_hi
          mma(taddr, wdesc(g), sdesc(g), IDESC_SKIN, g ? 1u : 0u);
          mma(taddr, wdesc(g), sdesc(JS + g), IDESC_SKIN, 1u);
          mma(taddr, wdesc(JS + g), sdesc(g), IDESC_SKIN, 1u);
        }
        commit(sempty(sstage));
        commit(tfull(buf));
      }
      __syncwarp();
    }
    if (ptx::elect_one()) commit(wempty(wb));   // this issuer's MMAs on the tile's weights are done
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
            for (int i = 0; i < NSLABS; ++i)
              load(f_base + i * F_SLAB, &tm_feat, ffull, i * BK, grp * NP + (int)crank * (NP / 2));
          }
        }
        for (int c = 0; c < ((p.debug & 32) ? 0 : 3); ++c)
          for (int i = 0; i < NSLABS; ++i) {
            ptx::mbar_wait(aempty(stage), phase ^ 1);
            if (ptx::elect_one()) {
              expect(afull(stage), A_SLAB);
              load(a_base + stage * A_SLAB, &tm_dirs, afull(stage), i * BK, c * p.V_pad + tile * TILE_V);
            }
            if (++stage == ASTAGES) { stage = 0; phase ^= 1; }
          }
      }
    } else if (warp == 3) {
      // ---- skinning weights (per tile) + transform chunks
      if (lane == 0) { ptx::prefetch_tmap(&tm_w); ptx::prefetch_tmap(&tm_s); }
      __syncwarp();
      uint32_t stage = 0, phase = 0, tc = 0;
      int grp = grp0, tp = tp0;
      for (int it = 0; it < n_my; ++it, ++tc, advance(grp, tp)) {
        const int tile = 2 * tp + (int)crank;
        const uint32_t wb = tc % WBUFS;
        ptx::mbar_wait(wempty(wb), ((tc / WBUFS) & 1) ^ 1);
        if (ptx::elect_one()) {
          expect(wfull(wb), JSLABS * A_SLAB);
          for (int i = 0; i < JSLABS; ++i)
            load(w_base + (wb * JSLABS + i) * A_SLAB, &tm_w, wfull(wb), i * BK, tile * TILE_V);
        }
        for (int ch = 0; ch < ((p.debug & 16) ? 0 : NCH); ++ch) {
          ptx::mbar_wait(sempty(stage), phase ^ 1);
          if (ptx::elect_one()) {
            expect(sfull(stage), JSLABS * S_SLAB);
            for (int i = 0; i < JSLABS; ++i)
              load(s_base + (stage * JSLABS + i) * S_SLAB, &tm_s, sfull(stage), i * BK,
                   (grp * NP + ch * CP) * 12 + (int)crank * (NS / 2));
          }
          if (++stage == SSTAGES) { stage = 0; phase ^= 1; }
        }
      }
    } else if (warp == 1 && crank == 0) {
      // ---- MMA issuer (the pair's leader issues for both CTAs; warp-wide loop, the elected lane issues)
      uint32_t astage = 0, aphase = 0, fph = 0, dph = 0, tc = 0;
      const uint64_t adesc0 = ptx::umma_desc_sw128(a_base), fdesc0 = ptx::umma_desc_sw128(f_base);
      auto fdesc = [&](int step) { return fdesc0 + (uint64_t)((step >> 2) * (F_SLAB >> 4) + 2 * (step & 3)); };
      int grp = grp0, tp = tp0;
      for (int it = 0; it < n_my; ++it, ++tc, advance(grp, tp)) {
        if (it == 0 || tp == 0) {
          ptx::mbar_wait(ffull, fph);
          fph ^= 1;
        }
        ptx::mbar_wait(dempty, dph ^ 1);   // both CTAs' epilogues have read all of the previous tile's D
        dph ^= 1;
        ptx::tc_fence_after();
        const bool last_of_group = (it == n_my - 1) || (tp == p.n_tp - 1);
        if (p.debug & 32) {
          if (ptx::elect_one()) {
            commit(dfull);
            if (last_of_group) commit(fempty);
          }
          __syncwarp();
        }
#pragma unroll 1
        for (int c = 0; c < ((p.debug & 32) ? 0 : 3); ++c) {
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
                if (g < KH16) {                    // basis_hi x (feat_hi + feat_lo)
                  mma(taddr, adesc + 2 * j, fdesc(g), IDESC_BLEND, g != 0 ? 1u : 0u);
                  mma(taddr, adesc + 2 * j, fdesc(KH16 + g), IDESC_BLEND, 1u);
                } else if (g < 2 * KH16) {         // basis_lo x feat_hi
                  mma(taddr, adesc + 2 * j, fdesc(g - KH16), IDESC_BLEND, 1u);
                }
              }
              commit(aempty(astage));
              if (c == 2 && i == NSLABS - 1) {
                commit(dfull);
                if (last_of_group) commit(fempty);
              }
            }
            __syncwarp();
            if (++astage == ASTAGES) { astage = 0; aphase ^= 1; }
          }
        }
        skin_chunks(tc, 0);   // even chunks of this tile (warp 2 issues the odd ones)
      }
    } else if (warp == 2 && crank == 0) {
      // ---- second skinning issuer: the odd chunks.  One issuing thread spends ~490 cycles per chunk on its serial
      // chain (two mbarrier waits at ~90 cycles each, fence, six MMAs, commits) for 192 cycles of tensor work
      // (measured with an empty epilogue); two warps alternate chunks so the chains overlap.
      // It must not start a tile's chunks before the tile's blend is complete: the epilogue consumes chunks in order
      // only after dfull, so a chunk issued early would sit in a T buffer that an EARLIER chunk (issued by warp 1
      // after the blend) needs -- a deadlock.
      for (uint32_t tc = 0; tc < (uint32_t)n_my; ++tc) {
        ptx::mbar_wait(dfull, tc & 1);
        skin_chunks(tc, 1);
      }
    }
  } else {
    // ---- epilogue: thread = vertex.  T (60 columns) and the chunk's 5 x (x,y,z) of D -> skinned vertex -> store
    ptx::setmaxnreg_inc<EPI_REGS>();
    const int q = warp & 3;
    const int set = (warp - 4) >> 2;
    const uint32_t lane_addr = (uint32_t)(q * 32) << 16;
    const size_t pstride = (size_t)p.V * 3;
    const uint32_t l_tempty0 = ptx::mapa(tempty(0), 0), l_dempty = ptx::mapa(dempty, 0);
    auto arrive = [&](uint32_t b) { ptx::mbar_arrive_cluster(b); };
    uint32_t dph = 0, tc = 0;
    int grp = grp0, tp = tp0;
    for (int it = 0; it < n_my; ++it, ++tc, advance(grp, tp)) {
      const int tile = 2 * tp + (int)crank;
      const int v0 = tile * TILE_V + q * 32;
      const int v = v0 + lane;
      // this set's chunks of the tile are set, set+3, ...: with NSETS == NT they all use T buffer (tc*NCH + set) % NT
      // shifted by nothing, and the barrier phase flips once per chunk
      uint32_t cc = tc * NCH + set;
      uint32_t buf = cc % NT, tph = (cc / NT) & 1;
      ptx::mbar_wait(dfull, dph);
      dph ^= 1;
      ptx::tc_fence_after();
      if (p.debug & 16) {
        __syncwarp();
        if (lane == 0) arrive(l_dempty);
      }
#pragma unroll 1
      for (int ch = set; ch < ((p.debug & 16) ? 0 : NCH); ch += NSETS) {
        ptx::mbar_wait(tfull(buf), tph);
        ptx::tc_fence_after();
        uint32_t t[64], dx[8], dy[8], dz[8];
        const uint32_t d0 = tmem_base + lane_addr + ch * CP;
        if (!(p.debug & 2)) ptx::tmem_ld_32x64(tmem_base + lane_addr + T_COL0 + buf * NS, t);
        else {
#pragma unroll
          for (int i = 0; i < 64; ++i) t[i] = 0x3f800000u;
        }
        if (!(p.debug & 4)) {
          ptx::tmem_ld_32x8(d0, dx);
          ptx::tmem_ld_32x8(d0 + NP, dy);
          ptx::tmem_ld_32x8(d0 + 2 * NP, dz);
        } else {
#pragma unroll
          for (int i = 0; i < 8; ++i) dx[i] = dy[i] = dz[i] = 0x3f800000u + i;
        }
        ptx::tmem_ld_wait();
        ptx::tc_fence_before();
        __syncwarp();
        if (lane == 0) {
          arrive(l_tempty0 + 8u * buf);
          if (ch + NSETS >= NCH) arrive(l_dempty);   // this warp's last read of the tile's D
        }
        static_assert(NSETS == NT, "a set keeps its T buffer within a tile: phase flips per chunk");
        tph ^= 1;
        const int64_t b0 = (int64_t)grp * NP + ch * CP;
        int n_ok = NP - ch * CP;                                        // poses of this chunk inside the group ...
        if (n_ok > CP) n_ok = CP;
        if (b0 + n_ok > p.B) n_ok = (int)max((int64_t)0, p.B - b0);     // ... and inside the batch
        // all CP poses first (independent FFMA chains), then the stores in one batch
        float o[CP][3];
        if (p.debug & 1) continue;
#pragma unroll
        for (int i = 0; i < CP; ++i) {
          const float* T = reinterpret_cast<const float*>(t) + i * 12;
          const float x = __uint_as_float(dx[i]), y = __uint_as_float(dy[i]), z = __uint_as_float(dz[i]);
          o[i][0] = fmaf(T[0], x, fmaf(T[1], y, fmaf(T[2], z, T[9])));
          o[i][1] = fmaf(T[3], x, fmaf(T[4], y, fmaf(T[5], z, T[10])));
          o[i][2] = fmaf(T[6], x, fmaf(T[7], y, fmaf(T[8], z, T[11])));
        }
        if (v < p.V) {
          // each lane stores its vertex's 12 bytes; the warp's 32 records are one contiguous 384-byte run
          float* dst = p.verts + (size_t)b0 * pstride + (size_t)v * 3;
#pragma unroll
          for (int i = 0; i < CP; ++i)
            if (i < n_ok) {
              float* w = dst + (size_t)i * pstride;
              w[0] = o[i][0];
              w[1] = o[i][1];
              w[2] = o[i][2];
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

}  // namespace lt2

// Two skinning K slabs (jp = 64: SMPL-X with the const tail).  Measured (profiles/r2_lbs_fused3_experiments.md): the
// 96-pose-group kernel wins there, its three T buffers hide the longer chunks; lbs_fused3 wins for one slab (jp = 32).
bool lbs_fused2_fits(const dpb_lbs* h, const LbsVariant& v) {
  if (!h->tc_ready || !v.dirs16) return false;
  if (v.kext != 448) return false;                      // instantiated for a 224-wide blend K (SMPL; SMPL-X const tail)
  if (h->J >= h->jp) return false;                      // needs the spare joint slot for the translation
  return h->jp == 64;
}

// verts[B,V,3] = skinned vertices.  featop [B_pad, kext] and skinop [B_pad*12, 2*jp] were written by the pose kernel.
int lbs_fused2(dpb_lbs* h, const LbsVariant& v, __half* featop, __half* skinop, float* verts, int64_t B,
               cudaStream_t st) {
  const int K2 = v.kext, Jp = h->jp;
  const int64_t B_pad = (B + 127) / 128 * 128;          // rows that physically exist (lbs_tc_ws_bytes); TMA zero-fills beyond
  CUtensorMap tm_feat, tm_s;
  int rc = make_tmap_2d(&tm_feat, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, featop, K2, (uint64_t)B_pad, lt2::BK, lt2::NP / 2, 2);
  if (rc == DPB_OK)
    rc = make_tmap_2d(&tm_s, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, skinop, 2 * Jp, (uint64_t)B_pad * 12, lt2::BK,
                      lt2::NS / 2, 2);
  if (rc != DPB_OK) return rc;
  lt2::Params p{};
  p.V = h->V;
  p.V_pad = h->n_cols_pad;
  p.n_tp = h->n_cols_pad / lt2::TILE_V / 2;
  p.B = B;
  p.n_items = (long long)((B + lt2::NP - 1) / lt2::NP) * p.n_tp;
  p.verts = verts;
  p.debug = getenv("DPB_LBS_DEBUG") ? atoi(getenv("DPB_LBS_DEBUG")) : 0;
  auto kern = lt2::lbs_fused2_kernel<14, 7, 4, 2, 4, 6, 1>;
  const size_t smem = lt2::Smem<2, 4, 6, 1>::BYTES;
  DPB_CUDA_CHECK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  int grid = h->sm_count & ~1;                                   // whole clusters of two
  const long long max_workers = p.n_items < 1 ? 1 : p.n_items;
  if (grid / 2 > max_workers) grid = (int)(2 * max_workers);
  kern<<<grid, lt2::NUM_THREADS, smem, st>>>(p, v.tm_dirs, tm_feat, h->tm_wop, tm_s);
  DPB_CUDA_CHECK(cudaGetLastError());
  return DPB_OK;
}

}  // namespace dpb
