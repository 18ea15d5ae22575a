// K1 for proteins (A = 20): per-site probabilistic substitution mapping on sm_100a, thread per
// site.  (Nucleotides, A = 4, run on the FP64 tensor-core kernels of k1_mma.cu; this file also
// holds the class-likelihood epilogue k1_finish and the [B][site] <-> [site][B] transpose.)
//
// Replaces DRHomogeneousTreeLikelihood::initialize (Felsenstein post-order + pre-order
// conditional likelihoods) followed by LegacySubstitutionMappingTools::
// computeSubstitutionVectors -- reference call sites CoETools.cpp:209,358-359,397 and
// AnalysisTools.cpp:592-611 (SURVEY.md s3.3, s8 a1/a2/a4/a5).
//
// Design (DESIGN.md "K1"):
//   * one warp per (32-site group, rate class): lane = site, so every table read is a
//     warp-uniform 128-bit shared load and every partial access is a coalesced 256-byte
//     row; the C class-warps of a site group sit in the same CTA and combine their
//     class terms through shared memory in a fixed order (deterministic, no atomics);
//   * the tree walk is a precompiled op stream (schedule.cpp) whose records carry the
//     branch transition matrices P_c(b) and reward matrices W_c(b) = p_c P o n; the CTA
//     streams it through shared memory with double-buffered TMA bulk copies;
//   * down pass: each inner node's partial is written to HBM exactly once
//     ([256-site block][slot][class*A+state][site], site contiguous -> coalesced); the message
//     of the larger child waits on a <= log2(T)-deep per-thread stack; two CTAs per SM at 128
//     registers (a register cache of the stack top costs 2 x 20 doubles and halves occupancy);
//   * up pass: each partial is read exactly once; both children of a node are expanded
//     together, the contraction sum_x Up[x] sum_y W[x][y] D[y] is fused, and the vector
//     entry is written as out[branch][site] (site contiguous); producer warps stream tables and
//     partials through shared-memory rings; one site group per CTA at 254 registers (five live
//     20-vectors per thread: two groups at 168 registers spill 1 KB per thread);
//   * nothing is accumulated with atomics: results are deterministic.
#include <algorithm>
#include <cstdlib>
#include <vector>
#include <cstdio>
#include "device_utils.cuh"
#include "kernels.h"

namespace cmb {

namespace {

// Down partials live in HBM block-major: [site block of 256][slot][c*A+x][256 sites].  A CTA
// of the up pass then walks one contiguous region (n_slots * C*A * 2 KB) instead of touching
// a different 2 MB page for every row of every node -- with the flat [slot][row][n_pad]
// layout the ring traffic alone ran at 2.2 TB/s (TLB / DRAM-page misses).
constexpr int kDSites = 256;
__host__ __device__ __forceinline__ size_t d_block(int64_t site_block, int slot, int n_slots, int rows) {
  return ((size_t)site_block * n_slots + slot) * ((size_t)rows * kDSites);
}

template <int A>
__device__ __forceinline__ void load_row(const double* __restrict__ row, double (&r)[A]) {
  if constexpr (A % 2 == 0) {
    const double2* p = reinterpret_cast<const double2*>(row);
#pragma unroll
    for (int i = 0; i < A / 2; i++) {
      double2 v = p[i];
      r[2 * i] = v.x;
      r[2 * i + 1] = v.y;
    }
  } else {
#pragma unroll
    for (int i = 0; i < A; i++) r[i] = row[i];
  }
}

// o[c][x] = sum_y T[c][x][y] v[c][y]
template <int A, int CB>
__device__ __forceinline__ void matvec(const double* __restrict__ T, const double (&v)[CB * A],
                                       double (&o)[CB * A]) {
#pragma unroll
  for (int c = 0; c < CB; c++)
#pragma unroll
    for (int x = 0; x < A; x++) {
      double row[A];
      load_row<A>(T + (c * A + x) * A, row);
      double s = row[0] * v[c * A];
#pragma unroll
      for (int y = 1; y < A; y++) s = fma(row[y], v[c * A + y], s);
      o[c * A + x] = s;
    }
}

// o[c][x] = sum_y T[c][y][x] v[c][y]   (message travelling down the edge)
template <int A, int CB>
__device__ __forceinline__ void matvec_t(const double* __restrict__ T, const double (&v)[CB * A],
                                         double (&o)[CB * A]) {
#pragma unroll
  for (int c = 0; c < CB; c++) {
#pragma unroll
    for (int y = 0; y < A; y++) {
      double row[A];
      load_row<A>(T + (c * A + y) * A, row);
#pragma unroll
      for (int x = 0; x < A; x++) o[c * A + x] = (y == 0) ? row[x] * v[c * A] : fma(row[x], v[c * A + y], o[c * A + x]);
    }
  }
}

// column pick for a resolved tip: o[c][x] = T[c][x][state]
template <int A, int CB>
__device__ __forceinline__ void tip_column(const double* __restrict__ T, int state, double (&o)[CB * A]) {
#pragma unroll
  for (int c = 0; c < CB; c++)
#pragma unroll
    for (int x = 0; x < A; x++) o[c * A + x] = T[(c * A + x) * A + state];
}

template <int A, int CB>
__device__ __forceinline__ void tip_dense(uint32_t mask, double (&d)[CB * A]) {
#pragma unroll
  for (int c = 0; c < CB; c++)
#pragma unroll
    for (int y = 0; y < A; y++) d[c * A + y] = (mask >> y) & 1u ? 1. : 0.;
}

template <int A, int NS>
__device__ __forceinline__ void matvec_n(const double* __restrict__ T, const double (&v)[NS][A], double (&o)[NS][A]) {
#pragma unroll
  for (int x = 0; x < A; x++) {
    double row[A];
    load_row<A>(T + x * A, row);
#pragma unroll
    for (int k = 0; k < NS; k++) {
      double s = row[0] * v[k][0];
#pragma unroll
      for (int y = 1; y < A; y++) s = fma(row[y], v[k][y], s);
      o[k][x] = s;
    }
  }
}
template <int A, int NS>
__device__ __forceinline__ void matvec_t_n(const double* __restrict__ T, const double (&v)[NS][A], double (&o)[NS][A]) {
#pragma unroll
  for (int y = 0; y < A; y++) {
    double row[A];
    load_row<A>(T + y * A, row);
#pragma unroll
    for (int k = 0; k < NS; k++)
#pragma unroll
      for (int x = 0; x < A; x++) o[k][x] = (y == 0) ? row[x] * v[k][0] : fma(row[x], v[k][y], o[k][x]);
  }
}
// acc[k] = sum_x u[k][x] * (W d[k])[x]
template <int A, int NS>
__device__ __forceinline__ void contract_n(const double* __restrict__ W, const double (&u)[NS][A],
                                           const double (&d)[NS][A], double (&acc)[NS]) {
#pragma unroll
  for (int k = 0; k < NS; k++) acc[k] = 0.;
#pragma unroll
  for (int x = 0; x < A; x++) {
    double row[A];
    load_row<A>(W + x * A, row);
#pragma unroll
    for (int k = 0; k < NS; k++) {
      double s = row[0] * d[k][0];
#pragma unroll
      for (int y = 1; y < A; y++) s = fma(row[y], d[k][y], s);
      acc[k] = fma(u[k][x], s, acc[k]);
    }
  }
}

// ------------------------------------------------------------------------------ down
// One warp per (site group, rate class); a lane owns NS sites (k*32 + lane), so every table
// row read from shared memory serves NS sites.  ncu r1f (NS = 1): the LSU / L1 path is the
// busiest unit of this kernel (l1tex 85 %: broadcast table reads, the per-thread message
// stack in local memory, the partial stores), DRAM 44 %.
template <int A, int NS, int CT>
__global__ void __launch_bounds__(256, (A > 4 ? 2 : 1)) k1_down(MapModel m, MapBuffers b, ChunkMeta cm, int groups, int tips_in_smem) {
  extern __shared__ __align__(128) unsigned char smem[];
  __shared__ uint32_t cmask[256];
  constexpr int AA = A * A;
  const int C = CT > 0 ? CT : m.C;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int c = warp % C, g = warp / C;
  const int64_t n_pad = b.n_pad;
  const int64_t site = ((int64_t)blockIdx.x * groups + g) * (32 * NS) + lane; // + k*32
  const int N = C * AA; // doubles per table (all classes)
  for (int i = threadIdx.x; i < 256; i += blockDim.x) cmask[i] = __ldg(m.code_mask + i);
  // The tip codes of this CTA's sites, all T rows, are staged in shared memory up front
  // (T x 64..128 bytes): fetching them node by node from HBM, one node ahead, made every node
  // cost one DRAM round trip (1.3 us per node per CTA regardless of the work per node).
  const int SGT = 32 * NS * groups;              // sites per CTA
  unsigned char* tipbuf = smem + 128 + 2 * (size_t)cm.cap;
  if (tips_in_smem) {
    const int64_t cta0 = (int64_t)blockIdx.x * SGT;
    const int per_row = SGT / 16;                // 16-byte pieces per row
    for (int i = threadIdx.x; i < m.T * per_row; i += blockDim.x) {
      const int row = i / per_row, piece = i % per_row;
      *reinterpret_cast<int4*>(tipbuf + (size_t)row * SGT + piece * 16) =
          *reinterpret_cast<const int4*>(b.tips + (size_t)row * n_pad + cta0 + piece * 16);
    }
  }
  const int lsite = g * (32 * NS) + lane;        // site inside the CTA (+ k*32)
  ChunkStream cs{cm.src, cm.off, cm.bytes, cm.n_chunks, cm.cap, nullptr, nullptr};
  cs.start(smem + 128, reinterpret_cast<uint64_t*>(smem)); // __syncthreads inside: cmask / tipbuf are visible

  double cur[NS][A];
  // message stack: the two youngest entries live in registers (t1 on top of t0), older ones
  // in local memory.  On a random 500-leaf tree 327 pushes cause 31 local spills instead of
  // 327 -- the write-through local stores were 44 % of this kernel's L1 -> L2 write traffic.
  double stk[kMaxStack][NS][A], t0[NS][A], t1[NS][A];
  int sp = 0, nc = 0;
  constexpr bool kRegCache = A <= 4;
#pragma unroll
  for (int k = 0; k < NS; k++)
#pragma unroll
    for (int i = 0; i < A; i++) cur[k][i] = 0.;

  // software pipeline: the tip codes of the next record are loaded while this one computes
  auto fetch_tips = [&](const unsigned char* rec, uint32_t (&ca)[NS], uint32_t (&cb)[NS]) {
    const int4 h = *reinterpret_cast<const int4*>(rec);
#pragma unroll
    for (int k = 0; k < NS; k++) {
      if (tips_in_smem) {
        ca[k] = ((uint32_t)h.x & kDownTipA) ? tipbuf[(size_t)h.y * SGT + lsite + k * 32] : 0u;
        cb[k] = ((uint32_t)h.x & kDownTipB) ? tipbuf[(size_t)h.z * SGT + lsite + k * 32] : 0u;
      } else {
        ca[k] = ((uint32_t)h.x & kDownTipA) ? b.tips[(size_t)h.y * n_pad + site + k * 32] : 0u;
        cb[k] = ((uint32_t)h.x & kDownTipB) ? b.tips[(size_t)h.z * n_pad + site + k * 32] : 0u;
      }
    }
  };
  // message of a tip through its edge: column pick when every lane holds a resolved state
  auto tip_message = [&](const double* tp, const uint32_t (&code)[NS], double (&out)[NS][A]) {
    uint32_t mk[NS];
    bool single = true;
#pragma unroll
    for (int k = 0; k < NS; k++) {
      mk[k] = cmask[code[k]];
      single = single && mk[k] != 0 && (mk[k] & (mk[k] - 1)) == 0;
    }
    if (__all_sync(0xffffffffu, single)) {
#pragma unroll
      for (int k = 0; k < NS; k++) {
        const int st = __ffs(mk[k]) - 1;
#pragma unroll
        for (int x = 0; x < A; x++) out[k][x] = tp[x * A + st];
      }
    } else {
      double d[NS][A];
#pragma unroll
      for (int k = 0; k < NS; k++)
#pragma unroll
        for (int y = 0; y < A; y++) d[k][y] = (mk[k] >> y) & 1u ? 1. : 0.;
      matvec_n<A, NS>(tp, d, out);
    }
  };
  uint32_t code_a[NS], code_b[NS];
  const unsigned char* rp = cs.wait(0);
  fetch_tips(rp, code_a, code_b);
  for (uint32_t kc = 0; kc < cm.n_chunks; kc++) {
    const uint32_t nrec = __ldg(cm.nrec + kc);
    for (uint32_t r = 0; r < nrec; r++) {
      const int4 h = *reinterpret_cast<const int4*>(rp);
      const uint32_t flags = (uint32_t)h.x;
      const int ntab = 1 + ((flags & kDownTipA) ? 1 : 0) + ((flags & kDownPush) ? 1 : 0);
      const unsigned char* rp_next = rp + ((16 + (size_t)ntab * N * sizeof(double) + 15) & ~size_t(15));
      if (r + 1 == nrec) rp_next = (kc + 1 < cm.n_chunks) ? cs.wait(kc + 1) : nullptr;
      uint32_t nca[NS], ncb[NS];
#pragma unroll
      for (int k = 0; k < NS; k++) nca[k] = ncb[k] = 0;
      if (rp_next) fetch_tips(rp_next, nca, ncb);
      const double* tp = reinterpret_cast<const double*>(rp + 16) + c * AA;
      double prod[NS][A];
      if (flags & kDownTipB) tip_message(tp, code_b, prod);
      else matvec_n<A, NS>(tp, cur, prod);
      tp += N;
      if (flags & kDownTipA) {
        double ma[NS][A];
        tip_message(tp, code_a, ma);
        tp += N;
#pragma unroll
        for (int k = 0; k < NS; k++)
#pragma unroll
          for (int i = 0; i < A; i++) prod[k][i] *= ma[k][i];
      } else if (kRegCache && nc == 2) {
        nc = 1;
#pragma unroll
        for (int k = 0; k < NS; k++)
#pragma unroll
          for (int i = 0; i < A; i++) prod[k][i] *= t1[k][i];
      } else if (kRegCache && nc == 1) {
        nc = 0;
#pragma unroll
        for (int k = 0; k < NS; k++)
#pragma unroll
          for (int i = 0; i < A; i++) prod[k][i] *= t0[k][i];
      } else {
        --sp;
#pragma unroll
        for (int k = 0; k < NS; k++)
#pragma unroll
          for (int i = 0; i < A; i++) prod[k][i] *= stk[sp][k][i];
      }
#pragma unroll
      for (int k = 0; k < NS; k++)
#pragma unroll
        for (int i = 0; i < A; i++) cur[k][i] = prod[k][i];
      if (h.w >= 0) {
        if constexpr (A == 4) { // [chunk][slot][class][site][state]: the layout k1_mma.cu's DMMA operands read
          double* d = b.D + d_chunk(site / kChunkSites, h.w, m.n_slots, C) +
                      ((size_t)c * kChunkSites + (site % kChunkSites)) * 4;
#pragma unroll
          for (int k = 0; k < NS; k++) {
            *reinterpret_cast<double2*>(d + k * 128) = make_double2(cur[k][0], cur[k][1]);
            *reinterpret_cast<double2*>(d + k * 128 + 2) = make_double2(cur[k][2], cur[k][3]);
          }
        } else {
          double* d = b.D + d_block(site >> 8, h.w, m.n_slots, C * A) + (size_t)(c * A) * kDSites + (site & (kDSites - 1));
#pragma unroll
          for (int k = 0; k < NS; k++)
#pragma unroll
            for (int i = 0; i < A; i++) d[i * kDSites + k * 32] = cur[k][i];
        }
      }
      if (flags & kDownPush) {
        if (!kRegCache) { // proteins: 2 x 20 doubles of register cache would halve the occupancy
          matvec_n<A, NS>(tp, cur, stk[sp]);
          ++sp;
        } else if (nc == 2) { // spill the oldest cached entry
#pragma unroll
          for (int k = 0; k < NS; k++)
#pragma unroll
            for (int i = 0; i < A; i++) { stk[sp][k][i] = t0[k][i]; t0[k][i] = t1[k][i]; }
          ++sp;
          matvec_n<A, NS>(tp, cur, t1);
        } else if (nc == 1) {
          matvec_n<A, NS>(tp, cur, t1);
          nc = 2;
        } else {
          matvec_n<A, NS>(tp, cur, t0);
          nc = 1;
        }
      }
      rp = rp_next;
#pragma unroll
      for (int k = 0; k < NS; k++) { code_a[k] = nca[k]; code_b[k] = ncb[k]; }
    }
    cs.release(kc);
  }
  // root: class likelihood L_c = sum_x pi_x root[c][x]
#pragma unroll
  for (int k = 0; k < NS; k++) {
    double l = 0.;
#pragma unroll
    for (int x = 0; x < A; x++) l = fma(cur[k][x], __ldg(m.pi + x), l);
    b.Lc[(size_t)c * n_pad + site + k * 32] = l;
  }
}

// ---------------------------------------------------------------------------- finish
// Site likelihood, log-likelihood, posterior rate, rate class with maximal likelihood
// (getLogLikelihoodPerSite / getPosteriorRatePerSite / getRateClassWithMaxPostProbPerSite,
// CoETools.cpp:507-510,669-670).
__global__ void k1_finish(MapModel m, MapBuffers b) {
  const int64_t site = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (site >= b.n_pad) return;
  double L = 0.;
  for (int c = 0; c < m.C; c++) L += b.Lc[(size_t)c * b.n_pad + site] * __ldg(m.probs + c);
  double pr = 0., best = 0.;
  int rc = 0;
  for (int c = 0; c < m.C; c++) {
    double l = b.Lc[(size_t)c * b.n_pad + site];
    pr += (l / L) * __ldg(m.probs + c) * __ldg(m.rates + c);
    if (c == 0 || l > best) { best = l; rc = c; }
  }
  b.invL[site] = 1. / L;
  b.loglik[site] = log(L);
  b.post_rate[site] = pr;
  b.rate_class[site] = rc;
}

// -------------------------------------------------------------------------------- up
// named barrier of site group g (immediate ids, so the kernel reserves 1 + 4 hardware
// barriers instead of all 16 and two CTAs fit on an SM)
__device__ __forceinline__ void group_barrier(int g, int nthreads) {
  switch (g) {
    case 0: asm volatile("bar.sync 1, %0;" ::"r"(nthreads) : "memory"); break;
    case 1: asm volatile("bar.sync 2, %0;" ::"r"(nthreads) : "memory"); break;
    case 2: asm volatile("bar.sync 3, %0;" ::"r"(nthreads) : "memory"); break;
    default: asm volatile("bar.sync 4, %0;" ::"r"(nthreads) : "memory"); break;
  }
}

// Up pass + contraction.  Shape of one CTA:
//   * G*C consumer warps: warp = (site group g, rate class c); every lane owns NS sites
//     (g*32*NS + k*32 + lane, k < NS); NS > 1 reuses each warp-uniform table row read from
//     shared memory for NS sites (the table reads, not the fp64 pipe, load the SM most:
//     ncu r1b, one site per lane: shared-memory wavefronts 58 % of peak, fp64 pipe 22 %);
//   * producer warp 1 streams the table chunks (double buffered);
//   * producer warp 2 streams, node by node, everything a node needs -- tip rows and the
//     stored partials of its inner children -- into one stage of a ring with cp.async.bulk;
//     one mbarrier full/empty pair per stage, producers back off with nanosleep.
// Consumers never read partials from global memory, so HBM latency is covered by the ring
// depth rather than by occupancy.  Cherry children (both grandchildren are tips) are not
// stored by the down pass: their partial is recomputed here from two tip codes.
// What bounds it (profiles/r1c, r1e): not HBM (ring traffic alone runs at 2.5 TB/s with the
// math switched off) but per-warp latency -- shared-memory and fixed-latency dependencies
// with 4 warps per SM sub-partition at 96 registers; see DESIGN.md "K1 up: what was tried".
struct UpParams {
  ChunkMeta cm;
  const int4* refs;     // per node 2 x int4: (flags, ref_a, ref_b, 0), (ref_a2, ref_b2, 0, 0)
  uint32_t n_nodes;
  int groups;           // G
  int n_blocks, n_tips; // stage ring depth (n_tips unused)
  uint32_t block_bytes; // C*A*SG*8
  // class block [c0, c0 + C) of a mapping with d_rows / A classes: the stored partials are rows c0*A.. of the
  // d_rows-row blocks of b.D, and a block after the first adds its terms to b.out instead of writing them
  int d_rows, d_row0, accumulate;
};
constexpr int kMaxBlocks = 8; // stage ring depth

template <int A, int NS, int MAXT, int MINB, int CT, int GT>
__global__ void __launch_bounds__(MAXT, MINB) k1_up(MapModel m, MapBuffers b, UpParams up) {
  extern __shared__ __align__(128) unsigned char smem[];
  constexpr int AA = A * A;
  constexpr int SW = 32 * NS;                     // sites per consumer warp
  // CT / GT > 0 fix the class count and the site groups at compile time (every stride becomes
  // an immediate); 0 = read them from the launch parameters
  const int C = CT > 0 ? CT : m.C, G = GT > 0 ? GT : up.groups, NSTG = up.n_blocks; // ring of per-node stages
  const int W = G * C;                            // consumer warps
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int64_t n_pad = b.n_pad;
  const int SG = SW * G;                          // sites per CTA
  const int64_t site0 = (int64_t)blockIdx.x * SG;
  const int N = C * AA;
  // smem: barriers (512 B) | red | table chunk buffers | tip ring | block ring
  uint64_t* tab_full = reinterpret_cast<uint64_t*>(smem);
  uint64_t* tab_empty = tab_full + 2;
  uint64_t* stg_full = tab_empty + 2;
  uint64_t* stg_empty = stg_full + kMaxBlocks;
  double* red = reinterpret_cast<double*>(smem + 512);
  const size_t red_bytes = (size_t)2 * W * 2 * SW * sizeof(double);
  unsigned char* tab_buf = smem + 512 + red_bytes;
  // stage = 4 tip rows (a, b, a2, b2) | partial block of child a | partial block of child b
  unsigned char* stg_ring = tab_buf + 2 * (size_t)up.cm.cap;
  const uint32_t tip_slot = 4u * (uint32_t)SG;
  const uint32_t stage_bytes = tip_slot + 2u * up.block_bytes;

  // code -> state mask table in shared memory: the lookup sits on every node's critical path
  __shared__ uint32_t cmask[256];
  for (int i = threadIdx.x; i < 256; i += blockDim.x) cmask[i] = __ldg(m.code_mask + i);
  if (threadIdx.x == 0) {
    for (int i = 0; i < 2; i++) { mbar_init(&tab_full[i], 1); mbar_init(&tab_empty[i], W); }
    for (int i = 0; i < NSTG; i++) { mbar_init(&stg_full[i], 1); mbar_init(&stg_empty[i], W); }
    mbar_fence_init();
  }
  __syncthreads();

  if (warp == W) {
    // ---- producer 1: table chunks
    if (lane == 0) {
      for (uint32_t k = 0; k < up.cm.n_chunks; k++) {
        if (k >= 2) mbar_wait_sleep(&tab_empty[k & 1], ((k >> 1) - 1) & 1, 500);
        const uint32_t nb = __ldg(up.cm.bytes + k);
        mbar_expect_tx(&tab_full[k & 1], nb);
        tma_bulk_g2s(tab_buf + (size_t)(k & 1) * up.cm.cap, up.cm.src + __ldg(up.cm.off + k), nb, &tab_full[k & 1]);
      }
    }
    return;
  }
  if (warp == W + 1) {
    // ---- producer 2: everything node n needs (tip rows, partial blocks of its inner
    //      children) into stage n % NSTG, one mbarrier phase per node
    const int rows = C * A;
    const uint32_t row_bytes = (uint32_t)SG * 8u;
    uint32_t s = 0, ph = 1;
    bool first = true;
    int4 r0 = __ldg(up.refs), r1 = __ldg(up.refs + 1);
    for (uint32_t n = 0; n < up.n_nodes; n++) {
      const int4 h0 = r0, h1 = r1;
      if (n + 1 < up.n_nodes) { r0 = __ldg(up.refs + 2 * (n + 1)); r1 = __ldg(up.refs + 2 * (n + 1) + 1); }
      const uint32_t flags = (uint32_t)h0.x;
      const bool tipa = flags & kUpTipA, tipb = flags & kUpTipB, cha = flags & kUpCherryA, chb = flags & kUpCherryB;
      const bool ina = !(tipa || cha), inb = !(tipb || chb);
      if (!first) mbar_wait_sleep(&stg_empty[s], ph, 200);
      unsigned char* st = stg_ring + (size_t)s * stage_bytes;
      if (lane == 0) {
        const uint32_t nrows = (tipa || cha) + (tipb || chb) + cha + chb;
        mbar_expect_tx(&stg_full[s], nrows * (uint32_t)SG + ((uint32_t)ina + (uint32_t)inb) * up.block_bytes);
        if (tipa || cha) tma_bulk_g2s(st, b.tips + (size_t)h0.y * n_pad + site0, SG, &stg_full[s]);
        if (tipb || chb) tma_bulk_g2s(st + SG, b.tips + (size_t)h0.z * n_pad + site0, SG, &stg_full[s]);
        if (cha) tma_bulk_g2s(st + 2 * SG, b.tips + (size_t)h1.x * n_pad + site0, SG, &stg_full[s]);
        if (chb) tma_bulk_g2s(st + 3 * SG, b.tips + (size_t)h1.y * n_pad + site0, SG, &stg_full[s]);
      }
      __syncwarp();
      if (ina) {
        const double* src = b.D + d_block(site0 >> 8, h0.y, m.n_slots, up.d_rows) + (size_t)up.d_row0 * kDSites + (site0 & (kDSites - 1));
        for (int r = lane; r < rows; r += 32)
          tma_bulk_g2s(st + tip_slot + (size_t)r * row_bytes, src + (size_t)r * kDSites, row_bytes, &stg_full[s]);
      }
      if (inb) {
        const double* src = b.D + d_block(site0 >> 8, h0.z, m.n_slots, up.d_rows) + (size_t)up.d_row0 * kDSites + (site0 & (kDSites - 1));
        for (int r = lane; r < rows; r += 32)
          tma_bulk_g2s(st + tip_slot + up.block_bytes + (size_t)r * row_bytes, src + (size_t)r * kDSites, row_bytes, &stg_full[s]);
      }
      if (++s == (uint32_t)NSTG) { s = 0; ph ^= 1; first = false; }
    }
    return;
  }

  // ---- consumers
  const int c = warp % C, g = warp / C;
  const int lsite = g * SW + lane;               // + k*32: site inside the CTA
  double Gm[NS][A];
  double stk[kMaxStack][NS][A];
  int sp = 0;
  double invL[NS];
#pragma unroll
  for (int k = 0; k < NS; k++) {
    invL[k] = b.invL[site0 + lsite + k * 32];
#pragma unroll
    for (int x = 0; x < A; x++) Gm[k][x] = __ldg(m.pi + x);
  }
  uint32_t node = 0, cs = 0, cph = 0; // stage slot and parity to wait for
  uint32_t my_items = 0; // (branch a|b, k) outputs this warp finishes: item it -> class it % C
  for (int it = 0; it < 2 * NS; it++)
    if (it % C == c) my_items |= 1u << it;

  for (uint32_t kc = 0; kc < up.cm.n_chunks; kc++) {
    mbar_wait(&tab_full[kc & 1], (kc >> 1) & 1);
    const unsigned char* rp = tab_buf + (size_t)(kc & 1) * up.cm.cap;
    const uint32_t nrec = __ldg(up.cm.nrec + kc);
    for (uint32_t r = 0; r < nrec; r++, node++) {
      const int4 h0 = *reinterpret_cast<const int4*>(rp);
      const int4 h1 = *reinterpret_cast<const int4*>(rp + 16);
      const uint32_t flags = (uint32_t)h0.x;
      const int out_a = h0.w, out_b = h1.x;
      const bool tipa = flags & kUpTipA, tipb = flags & kUpTipB, cha = flags & kUpCherryA, chb = flags & kUpCherryB;
      const double* Pa = reinterpret_cast<const double*>(rp + 32) + c * AA;
      const double* Wa = Pa + N;
      const double* Pb = Wa + N;
      const double* Wb = Pb + N;
      const double* Px = Wb + N; // cherry tables follow
      rp += 32 + (size_t)(4 + (cha ? 2 : 0) + (chb ? 2 : 0)) * N * sizeof(double);

      double Da[NS][A], Db[NS][A];
      int sa[NS], sb[NS];
      bool fasta = false, fastb = false;
      // ---- tip codes / cherry partials
      {
        mbar_wait(&stg_full[cs], cph);
        const unsigned char* ts = stg_ring + (size_t)cs * stage_bytes + lsite;
        if (tipa) {
          uint32_t mk[NS];
          bool single = true;
#pragma unroll
          for (int k = 0; k < NS; k++) {
            mk[k] = cmask[ts[k * 32]];
            single = single && mk[k] != 0 && (mk[k] & (mk[k] - 1)) == 0;
            sa[k] = __ffs(mk[k]) - 1;
          }
          fasta = __all_sync(0xffffffffu, single);
          if (!fasta) {
#pragma unroll
            for (int k = 0; k < NS; k++)
#pragma unroll
              for (int y = 0; y < A; y++) Da[k][y] = (mk[k] >> y) & 1u ? 1. : 0.;
          }
        } else if (cha) {
          uint32_t m1[NS], m2[NS];
          bool single = true;
#pragma unroll
          for (int k = 0; k < NS; k++) {
            m1[k] = cmask[ts[k * 32]];
            m2[k] = cmask[ts[2 * SG + k * 32]];
            single = single && m1[k] != 0 && (m1[k] & (m1[k] - 1)) == 0 && m2[k] != 0 && (m2[k] & (m2[k] - 1)) == 0;
          }
          const double* P1 = Px;
          const double* P2 = Px + N;
          if (__all_sync(0xffffffffu, single)) {
#pragma unroll
            for (int k = 0; k < NS; k++) {
              const int s1 = __ffs(m1[k]) - 1, s2 = __ffs(m2[k]) - 1;
#pragma unroll
              for (int x = 0; x < A; x++) Da[k][x] = P1[x * A + s1] * P2[x * A + s2];
            }
          } else {
            double d1[NS][A], d2[NS][A], t1[NS][A];
#pragma unroll
            for (int k = 0; k < NS; k++)
#pragma unroll
              for (int y = 0; y < A; y++) { d1[k][y] = (m1[k] >> y) & 1u ? 1. : 0.; d2[k][y] = (m2[k] >> y) & 1u ? 1. : 0.; }
            matvec_n<A, NS>(P1, d1, t1);
            matvec_n<A, NS>(P2, d2, Da);
#pragma unroll
            for (int k = 0; k < NS; k++)
#pragma unroll
              for (int x = 0; x < A; x++) Da[k][x] *= t1[k][x];
          }
        }
        if (tipb) {
          uint32_t mk[NS];
          bool single = true;
#pragma unroll
          for (int k = 0; k < NS; k++) {
            mk[k] = cmask[ts[SG + k * 32]];
            single = single && mk[k] != 0 && (mk[k] & (mk[k] - 1)) == 0;
            sb[k] = __ffs(mk[k]) - 1;
          }
          fastb = __all_sync(0xffffffffu, single);
          if (!fastb) {
#pragma unroll
            for (int k = 0; k < NS; k++)
#pragma unroll
              for (int y = 0; y < A; y++) Db[k][y] = (mk[k] >> y) & 1u ? 1. : 0.;
          }
        } else if (chb) {
          uint32_t m1[NS], m2[NS];
          bool single = true;
#pragma unroll
          for (int k = 0; k < NS; k++) {
            m1[k] = cmask[ts[SG + k * 32]];
            m2[k] = cmask[ts[3 * SG + k * 32]];
            single = single && m1[k] != 0 && (m1[k] & (m1[k] - 1)) == 0 && m2[k] != 0 && (m2[k] & (m2[k] - 1)) == 0;
          }
          const double* P1 = Px + (cha ? 2 * N : 0);
          const double* P2 = P1 + N;
          if (__all_sync(0xffffffffu, single)) {
#pragma unroll
            for (int k = 0; k < NS; k++) {
              const int s1 = __ffs(m1[k]) - 1, s2 = __ffs(m2[k]) - 1;
#pragma unroll
              for (int x = 0; x < A; x++) Db[k][x] = P1[x * A + s1] * P2[x * A + s2];
            }
          } else {
            double d1[NS][A], d2[NS][A], t1[NS][A];
#pragma unroll
            for (int k = 0; k < NS; k++)
#pragma unroll
              for (int y = 0; y < A; y++) { d1[k][y] = (m1[k] >> y) & 1u ? 1. : 0.; d2[k][y] = (m2[k] >> y) & 1u ? 1. : 0.; }
            matvec_n<A, NS>(P1, d1, t1);
            matvec_n<A, NS>(P2, d2, Db);
#pragma unroll
            for (int k = 0; k < NS; k++)
#pragma unroll
              for (int x = 0; x < A; x++) Db[k][x] *= t1[k][x];
          }
        }
      }
      // ---- stored partials of inner children, in ring order (a, then b)
      {
        const double* d = reinterpret_cast<const double*>(stg_ring + (size_t)cs * stage_bytes + tip_slot) + (size_t)(c * A) * SG + lsite;
        if (!(tipa || cha)) {
#pragma unroll
          for (int k = 0; k < NS; k++)
#pragma unroll
            for (int i = 0; i < A; i++) Da[k][i] = d[(size_t)i * SG + k * 32];
        }
        d += up.block_bytes / 8;
        if (!(tipb || chb)) {
#pragma unroll
          for (int k = 0; k < NS; k++)
#pragma unroll
            for (int i = 0; i < A; i++) Db[k][i] = d[(size_t)i * SG + k * 32];
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(&stg_empty[cs]); // the stage is in registers now
        if (++cs == (uint32_t)NSTG) { cs = 0; cph ^= 1; }
      }

      // ---- Ua = G o (Pb Db), branch a's class term, Ub = G o (Pa Da), branch b's class term
      double Ua[NS][A], Ub[NS][A], acc_a[NS], acc_b[NS];
      if (fastb) {
#pragma unroll
        for (int k = 0; k < NS; k++)
#pragma unroll
          for (int x = 0; x < A; x++) Ua[k][x] = Pb[x * A + sb[k]];
      } else matvec_n<A, NS>(Pb, Db, Ua);
#pragma unroll
      for (int k = 0; k < NS; k++)
#pragma unroll
        for (int x = 0; x < A; x++) Ua[k][x] = Gm[k][x] * Ua[k][x];
      if (out_a >= 0) {
        if (fasta) {
#pragma unroll
          for (int k = 0; k < NS; k++) {
            double t = 0.;
#pragma unroll
            for (int x = 0; x < A; x++) t = fma(Ua[k][x], Wa[x * A + sa[k]], t);
            acc_a[k] = t;
          }
        } else contract_n<A, NS>(Wa, Ua, Da, acc_a);
      }
      if (fasta) {
#pragma unroll
        for (int k = 0; k < NS; k++)
#pragma unroll
          for (int x = 0; x < A; x++) Ub[k][x] = Pa[x * A + sa[k]];
      } else matvec_n<A, NS>(Pa, Da, Ub);
#pragma unroll
      for (int k = 0; k < NS; k++)
#pragma unroll
        for (int x = 0; x < A; x++) Ub[k][x] = Gm[k][x] * Ub[k][x];
      if (out_b >= 0) {
        if (fastb) {
#pragma unroll
          for (int k = 0; k < NS; k++) {
            double t = 0.;
#pragma unroll
            for (int x = 0; x < A; x++) t = fma(Ub[k][x], Wb[x * A + sb[k]], t);
            acc_b[k] = t;
          }
        } else contract_n<A, NS>(Wb, Ub, Db, acc_b);
      }
      // ---- sum the C class terms of each site in class order; the 2*NS (branch, k) items
      //      of a site group are dealt round-robin to its C warps
      {
        double* rb = red + (size_t)(node & 1) * ((size_t)W * 2 * SW);
        double* mine = rb + (size_t)((g * C + c) * 2) * SW + lane;
#pragma unroll
        for (int k = 0; k < NS; k++) {
          if (out_a >= 0) mine[k * 32] = acc_a[k];
          if (out_b >= 0) mine[SW + k * 32] = acc_b[k];
        }
        group_barrier(g, 32 * C);
#pragma unroll
        for (int it = 0; it < 2 * NS; it++) {
          if (!(my_items >> it & 1u)) continue;
          const int ab = it / NS, k = it % NS;
          const int ob = ab ? out_b : out_a;
          if (ob < 0) continue;
          const double* src = rb + (size_t)(g * C * 2 + ab) * SW + k * 32 + lane;
          double t = 0.;
          for (int cc = 0; cc < C; cc++) t += src[(size_t)cc * 2 * SW];
          double* o = b.out + (size_t)ob * n_pad + site0 + lsite + k * 32;
          *o = up.accumulate ? *o + t * invL[k] : t * invL[k];
        }
      }
      // ---- messages for the children that are expanded later
      if (flags & kUpTakeA) {
        if (flags & kUpPush) {
          matvec_t_n<A, NS>(Pb, Ub, stk[sp]);
          ++sp;
        }
        matvec_t_n<A, NS>(Pa, Ua, Gm);
      } else if (flags & kUpTakeB) {
        matvec_t_n<A, NS>(Pb, Ub, Gm);
      } else if (flags & kUpPop) {
        --sp;
#pragma unroll
        for (int k = 0; k < NS; k++)
#pragma unroll
          for (int i = 0; i < A; i++) Gm[k][i] = stk[sp][k][i];
      }
    }
    __syncwarp();
    if (lane == 0) mbar_arrive(&tab_empty[kc & 1]);
  }
}

__global__ void k_transpose_out(const double* __restrict__ out, int B, int64_t n, int64_t n_pad,
                                double* __restrict__ dst, int64_t dst_stride) {
  __shared__ double tile[32][33];
  int64_t s0 = (int64_t)blockIdx.x * 32;
  int b0 = blockIdx.y * 32;
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    int br = b0 + i;
    int64_t s = s0 + threadIdx.x;
    tile[i][threadIdx.x] = (br < B && s < n) ? out[(size_t)br * n_pad + s] : 0.;
  }
  __syncthreads();
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    int64_t s = s0 + i;
    int br = b0 + threadIdx.x;
    if (s < n && br < B) dst[(size_t)s * dst_stride + br] = tile[threadIdx.x][i];
  }
}

int groups_per_cta(int C) { return C >= 8 ? 1 : 8 / C; }

template <int A, int NS, int CT>
void launch_down(const MapModel& m, const MapBuffers& b, const DevStream& s, cudaStream_t st) {
  int groups = groups_per_cta(m.C);
  while (groups > 1 && 32 * NS * groups > kDSites) groups /= 2;
  size_t smem = 128 + 2 * (size_t)s.cap;
  const size_t tip_bytes = (size_t)m.T * 32 * NS * groups;
  const int tips_in_smem = tip_bytes <= 64 * 1024 && !getenv("CMB_DOWN_GLOBAL_TIPS");
  if (tips_in_smem) smem += tip_bytes;
  CMB_CUDA(cudaFuncSetAttribute(k1_down<A, NS, CT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  k1_down<A, NS, CT><<<(unsigned)(b.n_pad / (32 * NS * groups)), 32 * groups * m.C, smem, st>>>(m, b, meta_of(s), groups,
                                                                                               tips_in_smem);
  CMB_CUDA(cudaGetLastError());
}
template <int A>
void run_down(const MapModel& m, const MapBuffers& b, const DevStream& s, cudaStream_t st) {
  // nucleotides run on the tensor-core kernels (k1_mma.cu); their stream is build_down_mma_stream's
  if constexpr (A == 4) return launch_map_down_mma(m, b, s, st);
  else return launch_down<A, 1, 0>(m, b, s, st);
}
struct UpShape { int groups, n_blocks, n_tips; size_t smem; uint32_t block_bytes; };
template <int A, int NS>
bool up_shape(int C, uint32_t cap, int max_smem, int max_warps, UpShape& sh) {
  // at most 4 site groups (named barriers 1..4); fewer when the warp budget or shared
  // memory (two stages at least) does not allow more
  for (int G = 4; G >= 1; G /= 2) {
    if (G * NS > 8 || G * C > max_warps) continue;
    const int SG = 32 * NS * G, W = G * C;
    const size_t red = (size_t)2 * W * 2 * 32 * NS * sizeof(double);
    const size_t block = (size_t)C * A * SG * 8;
    const size_t stage = 4 * (size_t)SG + 2 * block;
    const size_t fixed = 512 + red + 2 * (size_t)cap;
    if ((size_t)max_smem < fixed + 2 * stage) continue;
    sh.groups = G;
    sh.n_tips = 0;
    sh.n_blocks = (int)std::min<size_t>(kMaxBlocks, ((size_t)max_smem - fixed) / stage);
    sh.block_bytes = (uint32_t)block;
    sh.smem = fixed + (size_t)sh.n_blocks * stage;
    return true;
  }
  return false;
}

template <int A, int NS, int MAXT, int MINB, int CT = 0, int GT = 0>
bool try_up(const MapModel& m, const MapBuffers& b, const DevStream& s, cudaStream_t st, int c0 = 0, int c_total = 0) {
  int dev = 0, max_smem = 0;
  CMB_CUDA(cudaGetDevice(&dev));
  CMB_CUDA(cudaDeviceGetAttribute(&max_smem, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev));
  UpShape sh;
  max_smem = max_smem / MINB - 1024; // the system reserves 1 KB of shared memory per CTA
  if (CT > 0 && m.C != CT) return false;
  if (!up_shape<A, NS>(m.C, s.cap, max_smem, MAXT / 32 - 2, sh)) return false;
  if (GT > 0 && sh.groups != GT) return false;
  const int SG = 32 * NS * sh.groups;
  if (b.n_pad % SG) return false;
  UpParams up;
  up.cm = meta_of(s);
  up.refs = s.aux.as<int4>();
  up.n_nodes = s.n_records;
  up.groups = sh.groups;
  up.n_blocks = sh.n_blocks;
  up.n_tips = sh.n_tips;
  up.block_bytes = sh.block_bytes;
  up.d_rows = (c_total > 0 ? c_total : m.C) * A;
  up.d_row0 = c0 * A;
  up.accumulate = c0 > 0;
  CMB_CUDA(cudaFuncSetAttribute(k1_up<A, NS, MAXT, MINB, CT, GT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sh.smem));
  k1_up<A, NS, MAXT, MINB, CT, GT><<<(unsigned)(b.n_pad / SG), 32 * (sh.groups * m.C + 2), sh.smem, st>>>(m, b, up);
  CMB_CUDA(cudaGetLastError());
  return true;
}

template <int A>
void run_up(const MapModel& m, const MapBuffers& b, const DevStream& s, cudaStream_t st, int c0, int c_total) {
  if constexpr (A == 4) return launch_map_up_mma(m, b, s, st);
  // proteins: one site group per CTA (C class warps + 2 producers, <= 255 registers).  Two groups
  // (320 threads, 168 registers) spill 1 KB per thread of the five live 20-vectors: 12.3 vs 4.9 ms
  // per 20 000 sites at config 5.  More than kScalarUpClasses classes do not fit shared memory (two
  // record chunks of 3.2 KB x 4 x C plus two stages of C stored partials: 236 KB at C = 5 on a B200's
  // 227 KB), so the caller runs those in class blocks (Context::ensure_streams, run_map).
  else if (!try_up<A, 1, 192, 1>(m, b, s, st, c0, c_total))
    fail("mapping up pass: no launch shape fits shared memory for A = %d, C = %d", A, m.C);
}

} // namespace

void check_map_support(int A, int C) {
  if (A != 4 && A != 20)
    fail("mapping kernels are built for A = 4 (nucleotides) and A = 20 (proteins); got A = %d", A);
  if (C < 1 || C > 8) fail("mapping kernels support 1..8 rate classes; got C = %d", C);
}

void launch_map_down(const MapModel& m, const MapBuffers& b, const DevStream& s, cudaStream_t st) {
  if (b.n_pad % 256) fail("internal: n_pad must be a multiple of 256");
  if (m.A == 4) run_down<4>(m, b, s, st);
  else if (m.A == 20) run_down<20>(m, b, s, st);
  else fail("no mapping kernel for A = %d", m.A);
}
void launch_map_up(const MapModel& m, const MapBuffers& b, const DevStream& s, cudaStream_t st, int c0, int cb) {
  if (c0 < 0 || cb < 0 || c0 + cb > m.C || (c0 > 0 && cb == 0)) fail("internal: bad class block %d + %d of %d", c0, cb, m.C);
  if (cb > 0 && (m.A != 20 || cb > kScalarUpClasses)) fail("internal: class blocks are for the scalar protein up pass (<= %d classes)", kScalarUpClasses);
  MapModel mb = m;
  if (cb > 0) mb.C = cb;
  if (m.A == 4) run_up<4>(mb, b, s, st, c0, m.C);
  else if (m.A == 20) run_up<20>(mb, b, s, st, c0, m.C);
  else fail("no mapping kernel for A = %d", m.A);
}
void launch_map_finish(const MapModel& m, const MapBuffers& b, cudaStream_t st) {
  k1_finish<<<(unsigned)((b.n_pad + 255) / 256), 256, 0, st>>>(m, b);
  CMB_CUDA(cudaGetLastError());
}
void launch_transpose_out(const double* out, int B, int64_t n, int64_t n_pad, double* dst, cudaStream_t st,
                          int64_t dst_stride) {
  dim3 grid((unsigned)((n + 31) / 32), (unsigned)((B + 31) / 32)), block(32, 8);
  k_transpose_out<<<grid, block, 0, st>>>(out, B, n, n_pad, dst, dst_stride > 0 ? dst_stride : B);
  CMB_CUDA(cudaGetLastError());
}

} // namespace cmb
