// K1 for nucleotides (A = 4) on the FP64 tensor cores (DMMA m8n8k4): down pass, up pass +
// contraction.
//
// Contract: Bio++ DRHomogeneousTreeLikelihood::initialize (computeSubtreeLikelihoodPostfix /
// Prefix) + LegacySubstitutionMappingTools::computeSubstitutionVectors; reference call sites
// CoETools.cpp:209,358-359,395-397, AnalysisTools.cpp:592-611; SURVEY.md s3.3, s8 a1/a4.
// The first, thread-per-site design (now k1_map.cu, proteins only) was bound by shared-memory
// bandwidth and issue slots: every lane re-read every 4x4 table as warp-uniform broadcast loads
// (ncu r1f: LSU 66 %, FP64 pipe 21 %).  Here a warp owns 8*NG sites and ALL rate classes; lane =
// (site s = lane / 4, state q = lane % 4) holds ONE double per 4-vector, and every 4x4
// matrix-vector product of 8 sites is one DMMA.8x8x4 whose B operand (the table) is one double
// per lane:
//   MMA1/2  D_child (8 sites x 4) x [P | W]      -> lane (s, q): S[q] = (P D)[q], T[q] = (W D)[q]
//   U_a = G o S_b, U_b = G o S_a;   n_a += U_a . T_a  (per lane product, summed over classes
//   in registers, then over q with a two-stage transposing shuffle reduction per node)
//   MMA3/4  U (8 sites x 4) x P^T                -> lane (s, q): message to an inner child
// B fragments come precomputed in the op stream (schedule.cpp build_up_mma_stream /
// build_down_mma_stream), so a table costs 256 B of shared-memory reads per warp instead of 32
// broadcast rows.  Resolved tips are column picks from the raw 4x4 tables (conflict-free);
// ambiguity codes fall back to 0/1 mask partials through the DMMA.  Node bodies are specialised
// by what the two children are, so the C x NG independent DMMA chains of a node interleave.
// DMMA.8x8x4 runs at the FP64 pipe's full rate (tools/dmmabench: 37 TFLOP/s, 4 cycles per SM):
// ~2-3 DMMA per (node, class, 8 sites).
//
// Partials: [128-site chunk][slot][class][site][state] -- a lane reads / writes its double at
// consecutive addresses (256 B per DMMA A operand) and one TMA bulk copy moves a child's whole
// chunk (C * 4 KB) into the stage ring.  Measured on B200 at config 4 (517 k sites): down 4.2 ms
// (5.1 TB/s of stores), up 10.8 ms.
#include <algorithm>
#include <type_traits>
#include "device_utils.cuh"
#include "kernels.h"

namespace cmb {

namespace {

__device__ __forceinline__ void dmma(double& d0, double& d1, double a, double b) {
  asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%4,%5};"
               : "=d"(d0), "=d"(d1)
               : "d"(a), "d"(b), "d"(0.), "d"(0.));
}

struct UpMmaParams {
  const unsigned char* stream;                   // records, one per node
  const uint32_t *rec_off, *rec_bytes;
  const int4* refs;     // per node 2 x int4: (flags, ref_a, ref_b, tips_off), (ref_a2, ref_b2, blk_off, 0)
  uint32_t n_nodes, stage_bytes; // stage_bytes: largest packed stage (record | tip rows | chunks), 128-aligned
  int n_stages;         // ring depth
};
constexpr int kMaxStages = 8;
// Sites per CTA: a whole 128-site chunk of the partial layout, or a quarter of one when the batch is too small to
// give every SM a CTA (the observed alignment: 5000 sites = 40 chunks on 148 SMs; a narrow CTA walks the tree
// about five times faster because its two warps have the SM to themselves)
constexpr int kWideSG = kChunkSites, kNarrowSG = 32;

// what a child is, warp-uniform
enum : int { kInner = 0, kTip = 1, kCherry = 2 };

// Offsets (in doubles, from the end of the header) of a record's tables given what the two children are
// (schedule.cpp build_up_mma_stream): F1 / F3 fragments of the non-tip children, then per child the raw 4x4
// tables: tip P[C] W[C]; cherry P1[C] P2[C] W1[C] W2[C] (its two leaf edges).  Compile-time constants inside
// the specialised node bodies.
struct RecLayout { int F1a, F1b, F3a, F3b, Ra, Rb; };
__host__ __device__ constexpr RecLayout rec_layout(int C, int ka, int kb) {
  RecLayout r{};
  r.F1a = 0;
  r.F1b = r.F1a + (ka != 1 /* kTip */ ? C * 32 : 0);
  r.F3a = r.F1b + (kb != 1 ? C * 32 : 0);
  r.F3b = r.F3a + (ka != 1 ? C * 32 : 0);
  r.Ra = r.F3b + (kb != 1 ? C * 32 : 0);
  r.Rb = r.Ra + (ka == 1 ? 2 * C * 16 : ka == 2 /* kCherry */ ? 4 * C * 16 : 0);
  return r;
}

// entry `code` of row q of a raw 4x4 table (a resolved state), or the sum of the row's entries over the
// states an ambiguity code allows (MASK)
template <bool MASK>
__device__ __forceinline__ double pick(const double* row, uint32_t code) {
  if constexpr (!MASK) return row[code];
  else {
    double t = 0.;
#pragma unroll
    for (int y = 0; y < 4; y++) t += (code >> y) & 1u ? row[y] : 0.;
    return t;
  }
}

// The arithmetic of one node: straight-line code over the classes so the C x NG independent DMMA chains
// interleave.
//   inner child : D from the stage, (S, T) = DMMA(D, [P | W])
//   tip child   : S = P[q][state], T = W[q][state]   (column picks from the raw tables)
//   cherry child: D = P1[q][s1] * P2[q][s2], then as inner; its message M = DMMA(U, P^T) stays in registers
//                 and its two leaf branches are contracted here: n_1 += (M o P2 pick) . W1 pick, n_2 likewise
// acc: a, b, a1, a2, b1, b2 (the last four only for cherry children).  MASK: the codes are state masks
// (ambiguity somewhere in the warp's sites).  tab: first table of the record, blk: chunks, lane offsets applied.
template <int NG, int C, int SG, int KA, int KB, bool MASK>
__device__ __forceinline__ void node_body(const double* tab, const double* blk_a, const double* blk_b, int lane,
                                          const uint32_t (&sa)[NG], const uint32_t (&sa2)[NG], const uint32_t (&sb)[NG],
                                          const uint32_t (&sb2)[NG], double (&G)[C][NG], double (*push)[NG],
                                          const double (*pop)[NG], double (&acc)[6][NG]) {
  const int q = lane & 3;
  constexpr RecLayout L = rec_layout(C, KA, KB);
#pragma unroll
  for (int c = 0; c < C; c++) {
    double Sa[NG], Ta[NG], Sb[NG], Tb[NG];
    double p1a[NG], p2a[NG], p1b[NG], p2b[NG]; // leaf-edge picks of cherry children
    auto child = [&](auto kind, const double* F1, const double* blk, const double* R, const uint32_t (&s1)[NG],
                     const uint32_t (&s2)[NG], double (&S)[NG], double (&T)[NG], double (&p1)[NG], double (&p2)[NG]) {
      constexpr int K = decltype(kind)::value;
      if constexpr (K == kTip) {
#pragma unroll
        for (int g = 0; g < NG; g++) {
          S[g] = pick<MASK>(R + c * 16 + q * 4, s1[g]);
          T[g] = pick<MASK>(R + (C + c) * 16 + q * 4, s1[g]);
        }
      } else {
        double D[NG];
        if constexpr (K == kInner) {
#pragma unroll
          for (int g = 0; g < NG; g++) D[g] = blk[(size_t)c * (SG * 4) + g * 32];
        } else {
#pragma unroll
          for (int g = 0; g < NG; g++) {
            p1[g] = pick<MASK>(R + c * 16 + q * 4, s1[g]);
            p2[g] = pick<MASK>(R + (C + c) * 16 + q * 4, s2[g]);
            D[g] = p1[g] * p2[g];
          }
        }
        const double f = F1[c * 32 + lane];
#pragma unroll
        for (int g = 0; g < NG; g++) dmma(S[g], T[g], D[g], f);
      }
    };
    child(std::integral_constant<int, KA>(), tab + L.F1a, blk_a, tab + L.Ra, sa, sa2, Sa, Ta, p1a, p2a);
    child(std::integral_constant<int, KB>(), tab + L.F1b, blk_b, tab + L.Rb, sb, sb2, Sb, Tb, p1b, p2b);
    double Ua[NG], Ub[NG];
#pragma unroll
    for (int g = 0; g < NG; g++) {
      Ua[g] = G[c][g] * Sb[g];
      Ub[g] = G[c][g] * Sa[g];
      acc[0][g] = c == 0 ? Ua[g] * Ta[g] : fma(Ua[g], Ta[g], acc[0][g]);
      acc[1][g] = c == 0 ? Ub[g] * Tb[g] : fma(Ub[g], Tb[g], acc[1][g]);
    }
    double unused;
    // a cherry child's own node, inline: message through its edge, then its two leaf branches
    auto cherry = [&](const double* F3, const double* R, const uint32_t (&s1)[NG], const uint32_t (&s2)[NG],
                      const double (&U)[NG], const double (&p1)[NG], const double (&p2)[NG], double (&n1)[NG], double (&n2)[NG]) {
      const double f3 = F3[c * 32 + lane];
#pragma unroll
      for (int g = 0; g < NG; g++) {
        double M;
        dmma(M, unused, U[g], f3);
        const double w1 = pick<MASK>(R + (2 * C + c) * 16 + q * 4, s1[g]);
        const double w2 = pick<MASK>(R + (3 * C + c) * 16 + q * 4, s2[g]);
        const double u1 = M * p2[g], u2 = M * p1[g];
        n1[g] = c == 0 ? u1 * w1 : fma(u1, w1, n1[g]);
        n2[g] = c == 0 ? u2 * w2 : fma(u2, w2, n2[g]);
      }
    };
    if constexpr (KA == kCherry) cherry(tab + L.F3a, tab + L.Ra, sa, sa2, Ua, p1a, p2a, acc[2], acc[3]);
    if constexpr (KB == kCherry) cherry(tab + L.F3b, tab + L.Rb, sb, sb2, Ub, p1b, p2b, acc[4], acc[5]);
    if constexpr (KA == kInner) { // then b is inner too: b's message waits on the stack
      const double f3b = tab[L.F3b + c * 32 + lane];
#pragma unroll
      for (int g = 0; g < NG; g++) dmma(push[c][g], unused, Ub[g], f3b);
      const double f3a = tab[L.F3a + c * 32 + lane];
#pragma unroll
      for (int g = 0; g < NG; g++) dmma(G[c][g], unused, Ua[g], f3a);
    } else if constexpr (KB == kInner) {
      const double f3 = tab[L.F3b + c * 32 + lane];
#pragma unroll
      for (int g = 0; g < NG; g++) dmma(G[c][g], unused, Ub[g], f3);
    } else if (pop) {
#pragma unroll
      for (int g = 0; g < NG; g++) G[c][g] = pop[c][g];
    }
  }
}

// Per-lane constants of a consumer warp.
struct UpLane {
  int lane, q, lsite;      // lsite = wsite + s8: this lane's first site inside the CTA (group g adds 8 g)
  double* out;             // b.out + site0 + wsite + 8 (q & 1) + s8: the lane's store column after the quad reduction
  int64_t n_pad;
};

// One node of the walk, specialised by what the two children are: tip codes, arithmetic, release of the
// stage, then the sums over the four state lanes of a site and the stores.  STATES: the codes are resolved
// state indices (device-simulated alignments); otherwise they go through the code -> state-mask table and
// the warp takes the mask path when any of its sites is ambiguous.
template <int NG, int C, int SG, int KA, int KB, bool STATES>
__device__ __forceinline__ void node_step(const unsigned char* stage, int4 h0, const UpLane& ln, const uint32_t* cmask,
                                          double (&G)[C][NG], double (*stk)[C][NG], uint64_t* empty_bar) {
  constexpr uint32_t kBlock = C * SG * 32;
  const double* tab = reinterpret_cast<const double*>(stage + sizeof(UpMmaHdr));
  const unsigned char* ts = stage + h0.y + ln.lsite;   // tip code of (row, group g): ts[row * SG + 8 g]
  const double* blk_a = reinterpret_cast<const double*>(stage + h0.z) + ln.lsite * 4 + ln.q;
  const double* blk_b = blk_a + (KA == kInner ? kBlock / 8 : 0);
  double (*push)[NG] = stk[(h0.x >> 8) & 0xff];
  const int pop_level = (h0.x >> 16) & 0xff;
  const double (*pop)[NG] = (KA != kInner && KB != kInner && pop_level != 0xff) ? stk[pop_level] : nullptr;

  uint32_t sa[NG], sa2[NG], sb[NG], sb2[NG];
#pragma unroll
  for (int g = 0; g < NG; g++) {
    sa[g] = KA != kInner ? ts[8 * g] : 0;
    sa2[g] = KA == kCherry ? ts[2 * SG + 8 * g] : 0;
    sb[g] = KB != kInner ? ts[SG + 8 * g] : 0;
    sb2[g] = KB == kCherry ? ts[3 * SG + 8 * g] : 0;
  }
  double acc[6][NG];
  if constexpr (STATES || (KA == kInner && KB == kInner)) {
    node_body<NG, C, SG, KA, KB, false>(tab, blk_a, blk_b, ln.lane, sa, sa2, sb, sb2, G, push, pop, acc);
  } else {
    bool single = true;
#pragma unroll
    for (int g = 0; g < NG; g++) {
      sa[g] = KA != kInner ? cmask[sa[g]] : 1u;
      sa2[g] = KA == kCherry ? cmask[sa2[g]] : 1u;
      sb[g] = KB != kInner ? cmask[sb[g]] : 1u;
      sb2[g] = KB == kCherry ? cmask[sb2[g]] : 1u;
      single = single && __popc(sa[g]) == 1 && __popc(sa2[g]) == 1 && __popc(sb[g]) == 1 && __popc(sb2[g]) == 1;
    }
    if (__all_sync(0xffffffffu, single)) {
#pragma unroll
      for (int g = 0; g < NG; g++) {
        sa[g] = __ffs(sa[g]) - 1; sa2[g] = __ffs(sa2[g]) - 1;
        sb[g] = __ffs(sb[g]) - 1; sb2[g] = __ffs(sb2[g]) - 1;
      }
      node_body<NG, C, SG, KA, KB, false>(tab, blk_a, blk_b, ln.lane, sa, sa2, sb, sb2, G, push, pop, acc);
    } else {
      node_body<NG, C, SG, KA, KB, true>(tab, blk_a, blk_b, ln.lane, sa, sa2, sb, sb2, G, push, pop, acc);
    }
  }
  // output rows: lanes with q & 2 own the second branch of each pair (b, a2, b2)
  const int* hdr = reinterpret_cast<const int*>(stage);
  const int sel = (ln.q >> 1) & 1;
  const int ob0 = hdr[4 + sel];
  const int ob1 = KA == kCherry ? hdr[6 + sel] : -1;
  const int ob2 = KB == kCherry ? hdr[8 + sel] : -1;
  __syncwarp();
  if (ln.lane == 0) mbar_arrive(empty_bar);      // the stage has been read

  // ---- sum over the four state lanes of a site: 2 NG values per lane -> NG / 2 complete sums per lane
  //      (transposing reduction, 3 NG / 2 shuffles instead of 4 NG); lane q ends up with the items
  //      (branch = q >> 1, groups 2 j + (q & 1)).  1 / L is already in G (folded into the root message).
  constexpr int NJ = NG / 2;
  auto reduce_pair = [&](const double (&x)[NG], const double (&y)[NG], int ob) {
    double v[NG];
#pragma unroll
    for (int g = 0; g < NG; g++) {
      const double send = (ln.q & 2) ? x[g] : y[g];
      const double keep = (ln.q & 2) ? y[g] : x[g];
      v[g] = keep + __shfl_xor_sync(0xffffffffu, send, 2);
    }
#pragma unroll
    for (int j = 0; j < NJ; j++) {
      const double send = (ln.q & 1) ? v[2 * j] : v[2 * j + 1];
      const double keep = (ln.q & 1) ? v[2 * j + 1] : v[2 * j];
      const double t = keep + __shfl_xor_sync(0xffffffffu, send, 1);
      if (ob >= 0) ln.out[(size_t)ob * ln.n_pad + 16 * j] = t;
    }
  };
  reduce_pair(acc[0], acc[1], ob0);
  if constexpr (KA == kCherry) reduce_pair(acc[2], acc[3], ob1);
  if constexpr (KB == kCherry) reduce_pair(acc[4], acc[5], ob2);
}

// One node's copies into ring stage s: record, tip rows, partial chunks of the stored children (one lane).
template <int C, int SG>
__device__ __forceinline__ void up_issue_node(const MapModel& m, const MapBuffers& b, const UpMmaParams& up, int4 r0, int4 r1,
                                              uint32_t roff, uint32_t rnb, unsigned char* st, uint64_t* full, int64_t site0) {
  constexpr uint32_t kBlock = C * SG * 32;
  const int64_t n_pad = b.n_pad;
  const int64_t chunk = site0 / kChunkSites;
  const uint32_t flags = (uint32_t)r0.x;
  const int ref_a = r0.y, ref_b = r0.z, ref_a2 = r1.x, ref_b2 = r1.y;
  const uint32_t tips_off = (uint32_t)r0.w, blk_off = (uint32_t)r1.z;
  const bool tipa = flags & kUpTipA, tipb = flags & kUpTipB, cha = flags & kUpCherryA, chb = flags & kUpCherryB;
  const bool ina = !(tipa || cha), inb = !(tipb || chb);
  unsigned char* tp = st + tips_off;
  const uint32_t nrows = (tipa || cha) + (tipb || chb) + cha + chb;
  mbar_expect_tx(full, rnb + nrows * (uint32_t)SG + ((uint32_t)ina + (uint32_t)inb) * kBlock);
  tma_bulk_g2s(st, up.stream + roff, rnb, full);
  if (tipa || cha) tma_bulk_g2s(tp, b.tips + (size_t)ref_a * n_pad + site0, SG, full);
  if (tipb || chb) tma_bulk_g2s(tp + SG, b.tips + (size_t)ref_b * n_pad + site0, SG, full);
  if (cha) tma_bulk_g2s(tp + 2 * SG, b.tips + (size_t)ref_a2 * n_pad + site0, SG, full);
  if (chb) tma_bulk_g2s(tp + 3 * SG, b.tips + (size_t)ref_b2 * n_pad + site0, SG, full);
  // stored children, in order a then b, from blk_off: the whole chunk, or this CTA's sites of every class
  auto child = [&](unsigned char* dst, int slot) {
    const double* src = b.D + d_chunk(chunk, slot, m.n_slots, C);
    if constexpr (SG == kChunkSites) tma_bulk_g2s(dst, src, kBlock, full);
    else {
      const int sub = (int)(site0 % kChunkSites);
#pragma unroll
      for (int c = 0; c < C; c++) tma_bulk_g2s(dst + c * (SG * 32), src + (size_t)c * (kChunkSites * 4) + sub * 4, SG * 32, full);
    }
  };
  if (ina) child(st + blk_off, ref_a);
  if (inb) child(st + blk_off + (ina ? kBlock : 0), ref_b);
}

// Measured and left out (B200, config 4): folding the producer into the consumer warps (8 warps per CTA, 128
// registers: 36.3 ms per step against 34.4), L2 prefetch of the chunks 2..8 nodes ahead of their stage copy
// (33.3-35.6 against 33.1), producer wake-up by suspend-time hint or a 40 ns back-off instead of 200 ns (no change).
template <int NG, int C, int SG, int MINB, bool STATES>
__global__ void __launch_bounds__(32 * (SG / (8 * NG) + 1), MINB) k1_up_mma(MapModel m, MapBuffers b, UpMmaParams up) {
  extern __shared__ __align__(128) unsigned char smem[];
  constexpr int W = SG / (8 * NG);                 // consumer warps
  const uint32_t stage_bytes = up.stage_bytes;     // packed per node: record | tip rows (a, b, a2, b2) | chunks
  const int NSTG = up.n_stages;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int64_t site0 = (int64_t)blockIdx.x * SG;
  if (b.n_active && site0 >= (int64_t)__ldg(b.n_active)) return; // pattern-compressed batch: nothing behind the packed columns
  uint64_t* stg_full = reinterpret_cast<uint64_t*>(smem);
  uint64_t* stg_empty = stg_full + kMaxStages;
  unsigned char* stg_ring = smem + 128;

  __shared__ uint32_t cmask[STATES ? 1 : 256];
  if constexpr (!STATES)
    for (int i = threadIdx.x; i < 256; i += blockDim.x) cmask[i] = __ldg(m.code_mask + i);
  if (threadIdx.x == 0) {
    for (int i = 0; i < NSTG; i++) { mbar_init(&stg_full[i], 1); mbar_init(&stg_empty[i], W); }
    mbar_fence_init();
  }
  __syncthreads();

  if (warp == W) {
    // ---- producer: node n's record, tip rows and the partial chunks of its inner children go
    //      to stage n % NSTG; one mbarrier full / empty pair per stage.  The 32 lanes fetch the
    //      descriptors of 32 nodes at a time; lane 0 issues the copies.
    uint32_t s = 0, ph = 1;
    bool first = true;
    for (uint32_t n0 = 0; n0 < up.n_nodes; n0 += 32) {
      const uint32_t mine = min(n0 + lane, up.n_nodes - 1);
      const int4 r0 = __ldg(up.refs + 2 * mine), r1 = __ldg(up.refs + 2 * mine + 1);
      const uint32_t off = __ldg(up.rec_off + mine), nb = __ldg(up.rec_bytes + mine);
      const uint32_t cnt = min(32u, up.n_nodes - n0);
      for (uint32_t j = 0; j < cnt; j++) {
        int4 q0, q1;
        q0.x = __shfl_sync(0xffffffffu, r0.x, j); q0.y = __shfl_sync(0xffffffffu, r0.y, j);
        q0.z = __shfl_sync(0xffffffffu, r0.z, j); q0.w = __shfl_sync(0xffffffffu, r0.w, j);
        q1.x = __shfl_sync(0xffffffffu, r1.x, j); q1.y = __shfl_sync(0xffffffffu, r1.y, j);
        q1.z = __shfl_sync(0xffffffffu, r1.z, j); q1.w = 0;
        const uint32_t roff = __shfl_sync(0xffffffffu, off, j), rnb = __shfl_sync(0xffffffffu, nb, j);
        if (!first) mbar_wait_sleep(&stg_empty[s], ph, 200);
        if (lane == 0) up_issue_node<C, SG>(m, b, up, q0, q1, roff, rnb, stg_ring + (size_t)s * stage_bytes, &stg_full[s], site0);
        __syncwarp();
        if (++s == (uint32_t)NSTG) { s = 0; ph ^= 1; first = false; }
      }
    }
    return;
  }

  // ---- consumers
  UpLane ln;
  ln.lane = lane; ln.q = lane & 3;
  ln.lsite = warp * (8 * NG) + (lane >> 2);
  ln.n_pad = b.n_pad;
  ln.out = b.out + site0 + warp * (8 * NG) + 8 * (lane & 1) + (lane >> 2);
  double G[C][NG];
  double stk[kMaxStack][C][NG];
  {
    // root message pi, with 1 / L of the site folded in: every contraction below is linear in it, so the
    // stored values are n / L without a multiplication per output
    const double piq = __ldg(m.pi + ln.q);
#pragma unroll
    for (int g = 0; g < NG; g++) {
      const double gi = piq * b.invL[site0 + ln.lsite + 8 * g];
#pragma unroll
      for (int c = 0; c < C; c++) G[c][g] = gi;
    }
  }

  uint32_t cs = 0, cph = 0;
  for (uint32_t node = 0; node < up.n_nodes; node++) {
    mbar_wait(&stg_full[cs], cph);
    const unsigned char* stage = stg_ring + (size_t)cs * stage_bytes;
    const int4 h0 = *reinterpret_cast<const int4*>(stage); // kase | push level << 8 | pop level << 16, tips_off, blk_off, flags
    // smaller child first: an inner a implies an inner b, a cherry a implies a non-tip b
    switch (h0.x & 0xff) {
#define CMB_NODE(KA, KB) \
  case KA * 3 + KB: node_step<NG, C, SG, KA, KB, STATES>(stage, h0, ln, cmask, G, stk, &stg_empty[cs]); break;
      CMB_NODE(kInner, kInner) CMB_NODE(kTip, kInner) CMB_NODE(kTip, kTip) CMB_NODE(kTip, kCherry)
      CMB_NODE(kCherry, kInner) CMB_NODE(kCherry, kCherry)
#undef CMB_NODE
    }
    if (++cs == (uint32_t)NSTG) { cs = 0; cph ^= 1; }
  }
}

template <int NG, int C, int SG, int MINB, bool STATES>
bool try_up_mma(const MapModel& m, const MapBuffers& b, const DevStream& s, cudaStream_t st) {
  if (m.C != C) return false;
  int dev = 0, max_smem = 0;
  CMB_CUDA(cudaGetDevice(&dev));
  CMB_CUDA(cudaDeviceGetAttribute(&max_smem, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev));
  max_smem = max_smem / MINB - 1024 - 1024;      // 1 KB system reserve per CTA, 1 KB static (cmask)
  // largest packed stage at SG sites per CTA: nodes with k stored children need blk_off + k chunks
  size_t stage = 0;
  for (int k = 0; k < 3; k++)
    if (s.blk_off_max[k] || k == 0) stage = std::max(stage, (size_t)s.blk_off_max[k] + (size_t)k * C * SG * 32);
  stage = (stage + 127) & ~size_t(127);
  const size_t fixed = 128;
  if ((size_t)max_smem < fixed + 2 * stage) return false;
  UpMmaParams up;
  up.stream = s.bytes.as<unsigned char>();
  up.rec_off = s.off.as<uint32_t>();
  up.rec_bytes = s.nbytes.as<uint32_t>();
  up.refs = s.aux.as<int4>();
  up.n_nodes = s.n_records;
  up.stage_bytes = (uint32_t)stage;
  up.n_stages = (int)std::min<size_t>(kMaxStages, ((size_t)max_smem - fixed) / stage);
  // Shared memory is carved out of the 256 KB it shares with L1, and the consumers' message stack and
  // register spills live in local memory behind that L1: a third stage at C = 4 (2 x 111 KB of shared
  // memory, ~28 KB of L1) ran 41 ms per step instead of 33.  Keep a CTA's ring within 80 KB.
  constexpr size_t kRingBytes = 80 * 1024;
  if (MINB > 1) up.n_stages = (int)std::max<size_t>(2, std::min<size_t>(up.n_stages, kRingBytes / stage));
  const size_t smem = fixed + (size_t)up.n_stages * stage;
  constexpr int threads = 32 * (SG / (8 * NG) + 1);
  CMB_CUDA(cudaFuncSetAttribute(k1_up_mma<NG, C, SG, MINB, STATES>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  k1_up_mma<NG, C, SG, MINB, STATES><<<(unsigned)(b.n_pad / SG), threads, smem, st>>>(m, b, up);
  CMB_CUDA(cudaGetLastError());
  return true;
}

// batches that cannot give every SM a 128-site CTA run 32-site CTAs
bool narrow_batch(const MapBuffers& b) {
  static int sms = 0;
  if (!sms) {
    int dev = 0;
    CMB_CUDA(cudaGetDevice(&dev));
    CMB_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  }
  return b.n_pad / kWideSG < sms;
}

template <int C>
bool up_mma_for(const MapModel& m, const MapBuffers& b, const DevStream& s, cudaStream_t st) {
  if (m.C != C) return false;
  // B200, config 4 (517 k sites): 2 groups/warp x 2 CTAs/SM (16 consumer warps) 10.8 ms;
  // 4 groups/warp x 2 CTAs/SM (8 warps, 168 regs) 11.2 ms; 2 groups/warp x 1 CTA/SM 12.7 ms
  if (narrow_batch(b)) {
    if (m.states_only ? try_up_mma<2, C, kNarrowSG, 2, true>(m, b, s, st) : try_up_mma<2, C, kNarrowSG, 2, false>(m, b, s, st)) return true;
  }
  // device-simulated batches: 64-site CTAs, three per SM (12 consumer warps at 128 registers, a 3-stage ring each):
  // 26.6 ms per config-4 step against 27.7 for 128-site CTAs x 2
  if (m.states_only && try_up_mma<2, C, 64, 3, true>(m, b, s, st)) return true;
  if (m.states_only) return try_up_mma<2, C, kWideSG, 2, true>(m, b, s, st) || try_up_mma<2, C, kWideSG, 1, true>(m, b, s, st);
  return try_up_mma<2, C, kWideSG, 2, false>(m, b, s, st) || try_up_mma<2, C, kWideSG, 1, false>(m, b, s, st);
}

// ------------------------------------------------------------------------------ down
// Felsenstein post-order pass in the same lane mapping (lane = (site, state), warp = 8 NG
// sites x all classes).  A child's message through its edge, P D, is one DMMA per 8 sites
// (the second half of the B operand is unused) or, for a resolved tip, a column pick; the
// message of a larger sibling waits in a SHARED-MEMORY stack (depth <= log2 T, known from the
// schedule) instead of per-thread local memory; every stored partial leaves as one 256-byte
// row per (class, 8 sites).  The only global reads are the op stream and the tip rows, both
// through the producer warp's TMA ring.
struct DownMmaParams {
  const unsigned char* stream;
  const uint32_t *rec_off, *rec_bytes;
  const int4* refs;     // per node (flags, row_a, row_b, 0)
  uint32_t n_nodes, rec_cap;
  int n_stages;
};
constexpr int kDownStages = 8;

template <int NG, int C, int SG, int MINB, bool STATES>
__global__ void __launch_bounds__(32 * (SG / (8 * NG) + 1), MINB) k1_down_mma(MapModel m, MapBuffers b, DownMmaParams dp) {
  extern __shared__ __align__(128) unsigned char smem[];
  constexpr int W = SG / (8 * NG);
  constexpr uint32_t kEntry = C * SG * 32;         // one stack level of the CTA
  const uint32_t stage_bytes = dp.rec_cap + 2 * kWideSG;
  const int NSTG = dp.n_stages;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int64_t n_pad = b.n_pad;
  const int64_t site0 = (int64_t)blockIdx.x * SG;
  if (b.n_active && site0 >= (int64_t)__ldg(b.n_active)) return; // pattern-compressed batch
  uint64_t* stg_full = reinterpret_cast<uint64_t*>(smem);
  uint64_t* stg_empty = stg_full + kDownStages;
  unsigned char* stg_ring = smem + 128;
  double* stack = reinterpret_cast<double*>(stg_ring + (size_t)NSTG * stage_bytes);

  __shared__ uint32_t cmask[STATES ? 1 : 256];
  if constexpr (!STATES)
    for (int i = threadIdx.x; i < 256; i += blockDim.x) cmask[i] = __ldg(m.code_mask + i);
  if (threadIdx.x == 0) {
    for (int i = 0; i < NSTG; i++) { mbar_init(&stg_full[i], 1); mbar_init(&stg_empty[i], W); }
    mbar_fence_init();
  }
  __syncthreads();

  if (warp == W) {
    // ---- producer: record + the tip rows of node n into stage n % NSTG
    uint32_t s = 0, ph = 1;
    bool first = true;
    for (uint32_t n0 = 0; n0 < dp.n_nodes; n0 += 32) {
      const uint32_t mine = min(n0 + lane, dp.n_nodes - 1);
      const int4 r0 = __ldg(dp.refs + mine);
      const uint32_t off = __ldg(dp.rec_off + mine), nb = __ldg(dp.rec_bytes + mine);
      const uint32_t cnt = min(32u, dp.n_nodes - n0);
      for (uint32_t j = 0; j < cnt; j++) {
        const uint32_t flags = (uint32_t)__shfl_sync(0xffffffffu, r0.x, j);
        const int row_a = __shfl_sync(0xffffffffu, r0.y, j), row_b = __shfl_sync(0xffffffffu, r0.z, j);
        const uint32_t roff = __shfl_sync(0xffffffffu, off, j), rnb = __shfl_sync(0xffffffffu, nb, j);
        if (!first) mbar_wait_sleep(&stg_empty[s], ph, 200);
        if (lane == 0) {
          const bool tipa = flags & kDownTipA, tipb = flags & kDownTipB;
          unsigned char* st = stg_ring + (size_t)s * stage_bytes;
          mbar_expect_tx(&stg_full[s], rnb + ((uint32_t)tipa + (uint32_t)tipb) * (uint32_t)SG);
          tma_bulk_g2s(st, dp.stream + roff, rnb, &stg_full[s]);
          if (tipa) tma_bulk_g2s(st + dp.rec_cap, b.tips + (size_t)row_a * n_pad + site0, SG, &stg_full[s]);
          if (tipb) tma_bulk_g2s(st + dp.rec_cap + SG, b.tips + (size_t)row_b * n_pad + site0, SG, &stg_full[s]);
        }
        __syncwarp();
        if (++s == (uint32_t)NSTG) { s = 0; ph ^= 1; first = false; }
      }
    }
    return;
  }

  // ---- consumers
  const int q = lane & 3, s8 = lane >> 2;
  const int wsite = warp * (8 * NG);
  double cur[C][NG];
#pragma unroll
  for (int c = 0; c < C; c++)
#pragma unroll
    for (int g = 0; g < NG; g++) cur[c][g] = 0.;
  double* my_stack = stack + (size_t)wsite * 4 + lane; // + level * kEntry / 8 + c * SG * 4 + g * 32
  double* my_D = b.D + d_chunk(site0 / kChunkSites, 0, m.n_slots, C) + (size_t)(site0 % kChunkSites + wsite) * 4 + lane;
  const size_t slot_stride = (size_t)C * kChunkSites * 4;

  uint32_t cs = 0, cph = 0;
  for (uint32_t node = 0; node < dp.n_nodes; node++) {
    mbar_wait(&stg_full[cs], cph);
    const unsigned char* stage = stg_ring + (size_t)cs * stage_bytes;
    const int4 h = *reinterpret_cast<const int4*>(stage); // flags | pop level << 16 | push level << 24, rows, slot
    const uint32_t flags = (uint32_t)h.x;
    const bool tipa = flags & kDownTipA, tipb = flags & kDownTipB;
    const double* F = reinterpret_cast<const double*>(stage + 16);              // fragment of the running child
    const double* Ra = F + (tipa ? 0 : C * 32);                                  // raw P of tip a
    const double* Rb = Ra + (tipa ? C * 16 : 0);                                 // raw P of tip b
    const double* Fv = Rb + (tipb ? C * 16 : 0);                                 // fragment of v's own edge (push)
    const unsigned char* ts = stage + dp.rec_cap + wsite + s8;

    // message of a tip through its edge: lane q's component, all classes
    auto tip_message = [&](const unsigned char* codes, const double* R, double (&M)[C][NG]) {
      bool fast = true;
      uint32_t mk[NG];
#pragma unroll
      for (int g = 0; g < NG; g++) mk[g] = codes[8 * g];
      if constexpr (!STATES) {
        bool single = true;
#pragma unroll
        for (int g = 0; g < NG; g++) {
          mk[g] = cmask[mk[g]];
          single = single && __popc(mk[g]) == 1;
        }
        fast = __all_sync(0xffffffffu, single);
        if (fast) {
#pragma unroll
          for (int g = 0; g < NG; g++) mk[g] = __ffs(mk[g]) - 1;
        }
      }
      if (fast) {
#pragma unroll
        for (int c = 0; c < C; c++)
#pragma unroll
          for (int g = 0; g < NG; g++) M[c][g] = R[c * 16 + q * 4 + mk[g]];
      } else {
#pragma unroll
        for (int c = 0; c < C; c++)
#pragma unroll
          for (int g = 0; g < NG; g++) {
            double t = 0.;
#pragma unroll
            for (int y = 0; y < 4; y++) t += (mk[g] >> y) & 1u ? R[c * 16 + q * 4 + y] : 0.;
            M[c][g] = t;
          }
      }
    };
    auto edge_message = [&](const double* Fr, double (&M)[C][NG]) { // M = P cur, one DMMA per (class, 8 sites)
      double unused;
#pragma unroll
      for (int c = 0; c < C; c++) {
        const double f = Fr[c * 32 + lane];
#pragma unroll
        for (int g = 0; g < NG; g++) dmma(M[c][g], unused, cur[c][g], f);
      }
    };

    double Ma[C][NG], Mb[C][NG];
    if (tipa) {                       // cherry
      tip_message(ts, Ra, Ma);
      tip_message(ts + SG, Rb, Mb);
    } else if (tipb) {                // a's partial is the running one
      edge_message(F, Ma);
      tip_message(ts + SG, Rb, Mb);
    } else {                          // a's message waits on the stack, b's partial is the running one
      edge_message(F, Mb);
      const double* e = my_stack + (size_t)((flags >> 16) & 0xff) * (kEntry / 8);
#pragma unroll
      for (int c = 0; c < C; c++)
#pragma unroll
        for (int g = 0; g < NG; g++) Ma[c][g] = e[c * (SG * 4) + g * 32];
    }
#pragma unroll
    for (int c = 0; c < C; c++)
#pragma unroll
      for (int g = 0; g < NG; g++) cur[c][g] = Ma[c][g] * Mb[c][g];
    if (h.w >= 0) {
      double* d = my_D + (size_t)h.w * slot_stride;
#pragma unroll
      for (int c = 0; c < C; c++)
#pragma unroll
        for (int g = 0; g < NG; g++) d[c * (kChunkSites * 4) + g * 32] = cur[c][g];
    }
    if (flags & kDownPush) {
      double M[C][NG];
      edge_message(Fv, M);
      double* e = my_stack + (size_t)((flags >> 24) & 0xff) * (kEntry / 8);
#pragma unroll
      for (int c = 0; c < C; c++)
#pragma unroll
        for (int g = 0; g < NG; g++) e[c * (SG * 4) + g * 32] = M[c][g];
    }
    __syncwarp();
    if (lane == 0) mbar_arrive(&stg_empty[cs]);
    if (++cs == (uint32_t)NSTG) { cs = 0; cph ^= 1; }
  }
  // ---- root: class likelihood L_c = sum_x pi_x root[c][x]
  const double piq = __ldg(m.pi + q);
#pragma unroll
  for (int c = 0; c < C; c++)
#pragma unroll
    for (int g = 0; g < NG; g++) {
      double v = cur[c][g] * piq;
      v += __shfl_xor_sync(0xffffffffu, v, 1);
      v += __shfl_xor_sync(0xffffffffu, v, 2);
      if (q == 0) b.Lc[(size_t)c * n_pad + site0 + wsite + 8 * g + s8] = v;
    }
}

template <int NG, int C, int SG, int MINB, bool STATES>
bool try_down_mma(const MapModel& m, const MapBuffers& b, const DevStream& s, cudaStream_t st) {
  if (m.C != C) return false;
  int dev = 0, max_smem = 0;
  CMB_CUDA(cudaGetDevice(&dev));
  CMB_CUDA(cudaDeviceGetAttribute(&max_smem, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev));
  max_smem = max_smem / MINB - 1024 - 1024;      // 1 KB system reserve per CTA, 1 KB static (cmask)
  const size_t stage = (size_t)s.cap + 2 * (size_t)kWideSG, entry = (size_t)C * SG * 32;
  DownMmaParams dp;
  dp.stream = s.bytes.as<unsigned char>();
  dp.rec_off = s.off.as<uint32_t>();
  dp.rec_bytes = s.nbytes.as<uint32_t>();
  dp.refs = s.aux.as<int4>();
  dp.n_nodes = s.n_records;
  dp.rec_cap = s.cap;
  dp.n_stages = kDownStages;
  while (dp.n_stages > 2 && 128 + dp.n_stages * stage + entry > (size_t)max_smem) dp.n_stages /= 2;
  if (128 + dp.n_stages * stage > (size_t)max_smem) return false;
  // the whole message stack lives in shared memory (its levels are in the records: no run-time stack pointer)
  if (128 + dp.n_stages * stage + (size_t)s.stack_depth * entry > (size_t)max_smem) return false;
  const size_t smem = 128 + dp.n_stages * stage + (size_t)s.stack_depth * entry;
  constexpr int threads = 32 * (SG / (8 * NG) + 1);
  CMB_CUDA(cudaFuncSetAttribute(k1_down_mma<NG, C, SG, MINB, STATES>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  k1_down_mma<NG, C, SG, MINB, STATES><<<(unsigned)(b.n_pad / SG), threads, smem, st>>>(m, b, dp);
  CMB_CUDA(cudaGetLastError());
  return true;
}

template <int C>
bool down_mma_for(const MapModel& m, const MapBuffers& b, const DevStream& s, cudaStream_t st) {
  if (m.C != C) return false;
  if (m.states_only) {
    if (narrow_batch(b) && try_down_mma<2, C, kNarrowSG, 2, true>(m, b, s, st)) return true;
    return try_down_mma<2, C, kWideSG, 2, true>(m, b, s, st) || try_down_mma<2, C, kWideSG, 1, true>(m, b, s, st) ||
           try_down_mma<2, C, kNarrowSG, 1, true>(m, b, s, st);
  }
  if (narrow_batch(b) && try_down_mma<2, C, kNarrowSG, 2, false>(m, b, s, st)) return true;
  return try_down_mma<2, C, kWideSG, 2, false>(m, b, s, st) || try_down_mma<2, C, kWideSG, 1, false>(m, b, s, st) ||
         try_down_mma<2, C, kNarrowSG, 1, false>(m, b, s, st);
}

} // namespace

void launch_map_up_mma(const MapModel& m, const MapBuffers& b, const DevStream& s, cudaStream_t st) {
  if (m.A != 4) fail("internal: the tensor-core up pass is built for A = 4");
  if (b.n_pad % kWideSG) fail("internal: n_pad must be a multiple of %d", kWideSG);
  const bool done = up_mma_for<1>(m, b, s, st) || up_mma_for<2>(m, b, s, st) || up_mma_for<3>(m, b, s, st) ||
                    up_mma_for<4>(m, b, s, st) || up_mma_for<5>(m, b, s, st) || up_mma_for<6>(m, b, s, st) ||
                    up_mma_for<7>(m, b, s, st) || up_mma_for<8>(m, b, s, st);
  if (!done) fail("mapping up pass: no launch shape fits shared memory for A = 4, C = %d", m.C);
}

} // namespace cmb

namespace cmb {
void launch_map_down_mma(const MapModel& m, const MapBuffers& b, const DevStream& s, cudaStream_t st) {
  if (m.A != 4) fail("internal: the tensor-core down pass is built for A = 4");
  if (b.n_pad % kWideSG) fail("internal: n_pad must be a multiple of %d", kWideSG);
  const bool done = down_mma_for<1>(m, b, s, st) || down_mma_for<2>(m, b, s, st) || down_mma_for<3>(m, b, s, st) ||
                    down_mma_for<4>(m, b, s, st) || down_mma_for<5>(m, b, s, st) || down_mma_for<6>(m, b, s, st) ||
                    down_mma_for<7>(m, b, s, st) || down_mma_for<8>(m, b, s, st);
  if (!done) fail("mapping down pass: no launch shape fits shared memory for A = 4, C = %d", m.C);
}
} // namespace cmb
