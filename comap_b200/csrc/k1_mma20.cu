// K1 for proteins (A = 20) on the FP64 tensor cores (DMMA m8n8k4): down pass, up pass + contraction.
//
// Contract: Bio++ DRHomogeneousTreeLikelihood::initialize + LegacySubstitutionMappingTools::
// computeSubstitutionVectors; reference call sites CoETools.cpp:209,358-359,395-397, AnalysisTools.cpp:592-611,
// ClusterTools.cpp:224-227; SURVEY.md s3.3, s8 a1/a4.  For A = 20 the path is FP64-bound (15 flop per byte,
// SURVEY.md s8d), and the thread-per-site kernels of k1_map.cu reach 0.30 of the FP64 peak: every FMA there needs a
// warp-uniform shared-memory operand (ncu r1k: 254 registers, 9 % warps active, FP64 pipe 26 %).  Here every
// 20 x 20 matrix-vector product of 8 sites is 15 DMMA.8x8x4 (3 n-tiles x 5 k-tiles, 5/6 of the lanes' work useful)
// whose B operands come precomputed in the op stream (schedule.cpp build_*_mma20_stream).
//
// Lane mapping: a warp owns 16 sites (two 8-site groups) of ONE rate class; lane = (site s = lane / 4, q = lane % 4)
// holds states 4 kt + q, kt = 0..4, of every 20-vector -- five registers per vector, the DMMA A-operand layout, and
// (by the column permutation of the fragments) also the layout the products come out in, so chains of products
// need no shuffle.  A CTA = 4 consumer warps (64 sites) + a producer warp that streams, node by node, the class's
// record, the tip rows and the children's partial chunks through a shared-memory ring with TMA bulk copies
// (k1_mma.cu's scheme).  The grid is (site chunks) x (rate classes): the classes of a site run in different CTAs,
// write their contributions to a per-class partial output and a last small kernel adds them in class order
// (deterministic; 1 / L is folded into the root message, so the partials are already n / L).
//
// Partials in HBM: [64-site chunk][slot][class][k-tile][site][4 states] -- a lane's double sits at consecutive
// addresses (256 B per DMMA operand row) and one bulk copy moves a (child, class) chunk of 10 KB.
#include <algorithm>
#include <cstdlib>
#include <type_traits>
#include "device_utils.cuh"
#include "kernels.h"

namespace cmb {
namespace {

constexpr int SG = kChunkSites20;   // sites per CTA
constexpr int NG = 2;               // 8-site groups per warp
constexpr int W = SG / (8 * NG);    // consumer warps
constexpr int kStages20 = 8;
constexpr int kFr = 15 * 32;        // doubles of one matrix' fragments
constexpr int kRaw = 400;           // doubles of one raw (transposed) table

__device__ __forceinline__ void dmma_acc(double& d0, double& d1, double a, double b) {
  asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};" : "+d"(d0), "+d"(d1) : "d"(a), "d"(b));
}
__host__ __device__ inline size_t d_chunk20(int64_t chunk, int slot, int n_slots, int C, int c) {
  return (((size_t)chunk * n_slots + slot) * C + c) * ((size_t)SG * 20);
}

// y = M x for the warp's 2 x 8 sites; F = the 15 fragments of M
__device__ __forceinline__ void matvec20(const double* F, int lane, const double (&x)[5][NG], double (&y)[5][NG]) {
#pragma unroll
  for (int nt = 0; nt < 3; nt++) {
    double c0[NG], c1[NG];
#pragma unroll
    for (int g = 0; g < NG; g++) c0[g] = c1[g] = 0.;
#pragma unroll
    for (int kt = 0; kt < 5; kt++) {
      const double f = F[(nt * 5 + kt) * 32 + lane];
#pragma unroll
      for (int g = 0; g < NG; g++) dmma_acc(c0[g], c1[g], x[kt][g], f);
    }
#pragma unroll
    for (int g = 0; g < NG; g++) {
      y[2 * nt][g] = c0[g];
      if (2 * nt + 1 < 5) y[2 * nt + 1][g] = c1[g];
    }
  }
}
// column of a raw transposed table for a resolved tip state, or the sum of the columns an ambiguity mask allows
template <bool MASK>
__device__ __forceinline__ void tip_vector(const double* RT, int q, const uint32_t (&code)[NG], double (&y)[5][NG]) {
#pragma unroll
  for (int g = 0; g < NG; g++) {
    if constexpr (!MASK) {
#pragma unroll
      for (int kt = 0; kt < 5; kt++) y[kt][g] = RT[code[g] * 20 + 4 * kt + q];
    } else {
#pragma unroll
      for (int kt = 0; kt < 5; kt++) y[kt][g] = 0.;
      for (int st = 0; st < 20; st++)
        if ((code[g] >> st) & 1u) {
#pragma unroll
          for (int kt = 0; kt < 5; kt++) y[kt][g] += RT[st * 20 + 4 * kt + q];
        }
    }
  }
}
// codes of this lane's sites -> states, or -> masks when some site of the warp is ambiguous (returns true)
template <bool STATES>
__device__ __forceinline__ bool tip_codes(const unsigned char* row, const uint32_t* cmask, uint32_t (&code)[NG]) {
#pragma unroll
  for (int g = 0; g < NG; g++) code[g] = row[8 * g];
  if constexpr (STATES) return false;
  else {
    bool single = true;
#pragma unroll
    for (int g = 0; g < NG; g++) { code[g] = cmask[code[g]]; single = single && __popc(code[g]) == 1; }
    if (__all_sync(0xffffffffu, single)) {
#pragma unroll
      for (int g = 0; g < NG; g++) code[g] = __ffs(code[g]) - 1;
      return false;
    }
    return true;
  }
}
__device__ __forceinline__ void load_chunk(const double* blk, double (&d)[5][NG]) { // blk: lane offset applied
#pragma unroll
  for (int kt = 0; kt < 5; kt++)
#pragma unroll
    for (int g = 0; g < NG; g++) d[kt][g] = blk[(kt * SG + 8 * g) * 4];
}
__device__ __forceinline__ void hadamard(const double (&a)[5][NG], const double (&b)[5][NG], double (&y)[5][NG]) {
#pragma unroll
  for (int kt = 0; kt < 5; kt++)
#pragma unroll
    for (int g = 0; g < NG; g++) y[kt][g] = a[kt][g] * b[kt][g];
}
__device__ __forceinline__ void dot20(const double (&a)[5][NG], const double (&b)[5][NG], double (&s)[NG]) {
#pragma unroll
  for (int g = 0; g < NG; g++) {
    s[g] = a[0][g] * b[0][g];
#pragma unroll
    for (int kt = 1; kt < 5; kt++) s[g] = fma(a[kt][g], b[kt][g], s[g]);
  }
}

// ------------------------------------------------------------------------------------------- up
struct Up20Params {
  const unsigned char* stream;
  const uint32_t *rec_off, *rec_bytes;  // [node * C + class]
  const int4* refs;                     // per node 2 x int4: (flags, ref_a, ref_b, tips_off), (-, -, blk_off, 0)
  double* part;                         // [C][B][n_pad] per-class contributions
  uint32_t n_nodes, stage_bytes;
  int n_stages, B;
};
struct Lane20 {
  int lane, q, lsite;
  double* out;      // part + class * B * n_pad + site0 + warp * 16 + 8 (q & 1) + s8
  int64_t n_pad;
};

template <int KA, int KB, bool STATES>
__device__ __forceinline__ void node_step20(const unsigned char* stage, int4 h0, const Lane20& ln, const uint32_t* cmask,
                                            double (&G)[5][NG], double (*stk)[5][NG], uint64_t* empty_bar) {
  constexpr int kInner = 0, kTip = 1;
  const double* tab = reinterpret_cast<const double*>(stage + sizeof(UpMmaHdr));
  const double* tab_a = tab;
  const double* tab_b = tab + (KA == kInner ? 3 * kFr : 2 * kRaw);
  const unsigned char* ts = stage + h0.y + ln.lsite;
  const double* blk_a = reinterpret_cast<const double*>(stage + h0.z) + ln.lsite * 4 + ln.q;
  const double* blk_b = blk_a + (KA == kInner ? SG * 20 : 0);
  double acc_a[NG], acc_b[NG];
  if constexpr (KA == kInner) {          // both inner: b's message waits on the stack
    double Da[5][NG], Db[5][NG], X[5][NG], U[5][NG], T[5][NG], Gn[5][NG];
    load_chunk(blk_b, Db);
    matvec20(tab_b, ln.lane, Db, X);               // S_b = P_b D_b
    hadamard(G, X, U);                             // U_a = G o S_b
    load_chunk(blk_a, Da);
    matvec20(tab_a + kFr, ln.lane, Da, T);         // T_a = W_a D_a
    dot20(U, T, acc_a);
    matvec20(tab_a + 2 * kFr, ln.lane, U, Gn);     // message to a
    matvec20(tab_a, ln.lane, Da, X);               // S_a = P_a D_a
    hadamard(G, X, U);                             // U_b = G o S_a
    matvec20(tab_b + kFr, ln.lane, Db, T);         // T_b = W_b D_b
    dot20(U, T, acc_b);
    double (*push)[NG] = stk[(h0.x >> 8) & 0xff];
    matvec20(tab_b + 2 * kFr, ln.lane, U, X);      // message to b
#pragma unroll
    for (int kt = 0; kt < 5; kt++)
#pragma unroll
      for (int g = 0; g < NG; g++) { push[kt][g] = X[kt][g]; G[kt][g] = Gn[kt][g]; }
  } else {
    uint32_t ca[NG], cb[NG];
    const bool mask_a = tip_codes<STATES>(ts, cmask, ca);
    double Sa[5][NG], U[5][NG], T[5][NG];
    if (mask_a) tip_vector<true>(tab_a, ln.q, ca, Sa); else tip_vector<false>(tab_a, ln.q, ca, Sa);
    if constexpr (KB == kInner) {        // a tip, b inner
      double Db[5][NG], X[5][NG];
      load_chunk(blk_b, Db);
      matvec20(tab_b, ln.lane, Db, X);             // S_b
      hadamard(G, X, U);                           // U_a
      if (mask_a) tip_vector<true>(tab_a + kRaw, ln.q, ca, T); else tip_vector<false>(tab_a + kRaw, ln.q, ca, T);
      dot20(U, T, acc_a);
      hadamard(G, Sa, U);                          // U_b
      matvec20(tab_b + kFr, ln.lane, Db, T);       // T_b
      dot20(U, T, acc_b);
      matvec20(tab_b + 2 * kFr, ln.lane, U, G);    // message to b = the new running message
    } else {                             // both tips
      const bool mask_b = tip_codes<STATES>(ts + SG, cmask, cb);
      double Sb[5][NG];
      if (mask_b) tip_vector<true>(tab_b, ln.q, cb, Sb); else tip_vector<false>(tab_b, ln.q, cb, Sb);
      hadamard(G, Sb, U);
      if (mask_a) tip_vector<true>(tab_a + kRaw, ln.q, ca, T); else tip_vector<false>(tab_a + kRaw, ln.q, ca, T);
      dot20(U, T, acc_a);
      hadamard(G, Sa, U);
      if (mask_b) tip_vector<true>(tab_b + kRaw, ln.q, cb, T); else tip_vector<false>(tab_b + kRaw, ln.q, cb, T);
      dot20(U, T, acc_b);
      const int pop_level = (h0.x >> 16) & 0xff;
      if (pop_level != 0xff) {
        const double (*pop)[NG] = stk[pop_level];
#pragma unroll
        for (int kt = 0; kt < 5; kt++)
#pragma unroll
          for (int g = 0; g < NG; g++) G[kt][g] = pop[kt][g];
      }
    }
  }
  const int* hdr = reinterpret_cast<const int*>(stage);
  const int ob = hdr[4 + ((ln.q >> 1) & 1)];       // lanes with q & 2 own branch b
  __syncwarp();
  if (ln.lane == 0) mbar_arrive(empty_bar);        // the stage has been read
  // sum over the four state lanes of a site (transposing reduction as in k1_mma.cu): lane q ends up with
  // (branch = q >> 1, group = q & 1)
  double v[NG];
#pragma unroll
  for (int g = 0; g < NG; g++) {
    const double send = (ln.q & 2) ? acc_a[g] : acc_b[g];
    const double keep = (ln.q & 2) ? acc_b[g] : acc_a[g];
    v[g] = keep + __shfl_xor_sync(0xffffffffu, send, 2);
  }
  const double send = (ln.q & 1) ? v[0] : v[1];
  const double keep = (ln.q & 1) ? v[1] : v[0];
  const double t = keep + __shfl_xor_sync(0xffffffffu, send, 1);
  if (ob >= 0) ln.out[(size_t)ob * ln.n_pad] = t;
}

template <int MINB, bool STATES>
__global__ void __launch_bounds__(32 * (W + 1), MINB) k1_up_mma20(MapModel m, MapBuffers b, Up20Params up) {
  extern __shared__ __align__(128) unsigned char smem[];
  const uint32_t stage_bytes = up.stage_bytes;
  const int NSTG = up.n_stages;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int cls = blockIdx.y, C = m.C;
  const int64_t site0 = (int64_t)blockIdx.x * SG;
  uint64_t* stg_full = reinterpret_cast<uint64_t*>(smem);
  uint64_t* stg_empty = stg_full + kStages20;
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
    // ---- producer: (node, class) record, tip rows, partial chunks of the inner children -> stage n % NSTG
    uint32_t s = 0, ph = 1;
    bool first = true;
    const int64_t n_pad = b.n_pad;
    for (uint32_t n0 = 0; n0 < up.n_nodes; n0 += 32) {
      const uint32_t mine = min(n0 + lane, up.n_nodes - 1);
      const int4 r0 = __ldg(up.refs + 2 * mine), r1 = __ldg(up.refs + 2 * mine + 1);
      const uint32_t off = __ldg(up.rec_off + (size_t)mine * C + cls), nb = __ldg(up.rec_bytes + (size_t)mine * C + cls);
      const uint32_t cnt = min(32u, up.n_nodes - n0);
      for (uint32_t j = 0; j < cnt; j++) {
        const uint32_t flags = (uint32_t)__shfl_sync(0xffffffffu, r0.x, j);
        const int ref_a = __shfl_sync(0xffffffffu, r0.y, j), ref_b = __shfl_sync(0xffffffffu, r0.z, j);
        const uint32_t tips_off = (uint32_t)__shfl_sync(0xffffffffu, r0.w, j), blk_off = (uint32_t)__shfl_sync(0xffffffffu, r1.z, j);
        const uint32_t roff = __shfl_sync(0xffffffffu, off, j), rnb = __shfl_sync(0xffffffffu, nb, j);
        if (!first) mbar_wait_sleep(&stg_empty[s], ph, 200);
        if (lane == 0) {
          const bool tipa = flags & kUpTipA, tipb = flags & kUpTipB;
          unsigned char* st = stg_ring + (size_t)s * stage_bytes;
          constexpr uint32_t kBlock = SG * 160;
          mbar_expect_tx(&stg_full[s], rnb + ((uint32_t)tipa + (uint32_t)tipb) * SG + ((uint32_t)!tipa + (uint32_t)!tipb) * kBlock);
          tma_bulk_g2s(st, up.stream + roff, rnb, &stg_full[s]);
          if (tipa) tma_bulk_g2s(st + tips_off, b.tips + (size_t)ref_a * n_pad + site0, SG, &stg_full[s]);
          if (tipb) tma_bulk_g2s(st + tips_off + SG, b.tips + (size_t)ref_b * n_pad + site0, SG, &stg_full[s]);
          if (!tipa) tma_bulk_g2s(st + blk_off, b.D + d_chunk20(blockIdx.x, ref_a, m.n_slots, C, cls), kBlock, &stg_full[s]);
          if (!tipb) tma_bulk_g2s(st + blk_off + (tipa ? 0 : kBlock), b.D + d_chunk20(blockIdx.x, ref_b, m.n_slots, C, cls), kBlock, &stg_full[s]);
        }
        __syncwarp();
        if (++s == (uint32_t)NSTG) { s = 0; ph ^= 1; first = false; }
      }
    }
    return;
  }

  // ---- consumers
  Lane20 ln;
  ln.lane = lane; ln.q = lane & 3;
  ln.lsite = warp * (8 * NG) + (lane >> 2);
  ln.n_pad = b.n_pad;
  ln.out = up.part + (size_t)cls * up.B * b.n_pad + site0 + warp * (8 * NG) + 8 * (lane & 1) + (lane >> 2);
  double G[5][NG];
  double stk[kMaxStack][5][NG];
#pragma unroll
  for (int g = 0; g < NG; g++) {
    const double il = b.invL[site0 + ln.lsite + 8 * g]; // 1 / L folded into the root message (the contraction is linear in it)
#pragma unroll
    for (int kt = 0; kt < 5; kt++) G[kt][g] = __ldg(m.pi + 4 * kt + ln.q) * il;
  }
  uint32_t cs = 0, cph = 0;
  for (uint32_t node = 0; node < up.n_nodes; node++) {
    mbar_wait(&stg_full[cs], cph);
    const unsigned char* stage = stg_ring + (size_t)cs * stage_bytes;
    const int4 h0 = *reinterpret_cast<const int4*>(stage); // kase | push level << 8 | pop level << 16, tips_off, blk_off, flags
    switch (h0.x & 0xff) {
      case 0: node_step20<0, 0, STATES>(stage, h0, ln, cmask, G, stk, &stg_empty[cs]); break;
      case 3: node_step20<1, 0, STATES>(stage, h0, ln, cmask, G, stk, &stg_empty[cs]); break;
      case 4: node_step20<1, 1, STATES>(stage, h0, ln, cmask, G, stk, &stg_empty[cs]); break;
    }
    if (++cs == (uint32_t)NSTG) { cs = 0; cph ^= 1; }
  }
}

// out[b][site] = sum over classes, in class order, of the per-class contributions
__global__ void k1_sum_classes(int C, int B, int64_t n_pad, const double* __restrict__ part, double* __restrict__ out) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (int64_t)B * n_pad) return;
  double s = part[i];
  for (int c = 1; c < C; c++) s += part[(size_t)c * B * n_pad + i];
  out[i] = s;
}

// ------------------------------------------------------------------------------------------- down
struct Down20Params {
  const unsigned char* stream;
  const uint32_t *rec_off, *rec_bytes;  // [node * C + class]
  const int4* refs;                     // per node (flags | levels, row_a, row_b, 0)
  uint32_t n_nodes, rec_cap;
  int n_stages;
};

template <int MINB, bool STATES>
__global__ void __launch_bounds__(32 * (W + 1), MINB) k1_down_mma20(MapModel m, MapBuffers b, Down20Params dp) {
  extern __shared__ __align__(128) unsigned char smem[];
  const uint32_t stage_bytes = dp.rec_cap + 2 * SG;
  const int NSTG = dp.n_stages;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int cls = blockIdx.y, C = m.C;
  const int64_t n_pad = b.n_pad;
  const int64_t site0 = (int64_t)blockIdx.x * SG;
  uint64_t* stg_full = reinterpret_cast<uint64_t*>(smem);
  uint64_t* stg_empty = stg_full + kStages20;
  unsigned char* stg_ring = smem + 128;
  double* stack = reinterpret_cast<double*>(stg_ring + (size_t)NSTG * stage_bytes); // [level][kt][site][4]
  __shared__ uint32_t cmask[STATES ? 1 : 256];
  if constexpr (!STATES)
    for (int i = threadIdx.x; i < 256; i += blockDim.x) cmask[i] = __ldg(m.code_mask + i);
  if (threadIdx.x == 0) {
    for (int i = 0; i < NSTG; i++) { mbar_init(&stg_full[i], 1); mbar_init(&stg_empty[i], W); }
    mbar_fence_init();
  }
  __syncthreads();

  if (warp == W) {
    uint32_t s = 0, ph = 1;
    bool first = true;
    for (uint32_t n0 = 0; n0 < dp.n_nodes; n0 += 32) {
      const uint32_t mine = min(n0 + lane, dp.n_nodes - 1);
      const int4 r0 = __ldg(dp.refs + mine);
      const uint32_t off = __ldg(dp.rec_off + (size_t)mine * C + cls), nb = __ldg(dp.rec_bytes + (size_t)mine * C + cls);
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

  const int q = lane & 3, lsite = warp * (8 * NG) + (lane >> 2);
  double cur[5][NG];
#pragma unroll
  for (int kt = 0; kt < 5; kt++)
#pragma unroll
    for (int g = 0; g < NG; g++) cur[kt][g] = 0.;
  double* my_stack = stack + lsite * 4 + q;                        // + level * SG * 20 + (kt * SG + 8 g) * 4
  double* my_D = b.D + d_chunk20(blockIdx.x, 0, m.n_slots, C, cls) + lsite * 4 + q;
  const size_t slot_stride = (size_t)C * SG * 20;

  uint32_t cs = 0, cph = 0;
  for (uint32_t node = 0; node < dp.n_nodes; node++) {
    mbar_wait(&stg_full[cs], cph);
    const unsigned char* stage = stg_ring + (size_t)cs * stage_bytes;
    const int4 h = *reinterpret_cast<const int4*>(stage);
    const uint32_t flags = (uint32_t)h.x;
    const bool tipa = flags & kDownTipA, tipb = flags & kDownTipB;
    const double* T0 = reinterpret_cast<const double*>(stage + 16);
    const unsigned char* ts = stage + dp.rec_cap + lsite;
    double Ma[5][NG], Mb[5][NG];
    const double* Fv;                                              // fragments of v's own edge (push)
    auto tip_message = [&](const unsigned char* row, const double* RT, double (&M)[5][NG]) {
      uint32_t code[NG];
      if (tip_codes<STATES>(row, cmask, code)) tip_vector<true>(RT, q, code, M); else tip_vector<false>(RT, q, code, M);
    };
    if (tipa) {                       // cherry: two column picks
      tip_message(ts, T0, Ma);
      tip_message(ts + SG, T0 + kRaw, Mb);
      Fv = T0 + 2 * kRaw;
    } else if (tipb) {                // a's partial is the running one
      matvec20(T0, lane, cur, Ma);
      tip_message(ts + SG, T0 + kFr, Mb);
      Fv = T0 + kFr + kRaw;
    } else {                          // a's message waits on the stack, b's partial is the running one
      matvec20(T0, lane, cur, Mb);
      const double* e = my_stack + (size_t)((flags >> 16) & 0xff) * (SG * 20);
#pragma unroll
      for (int kt = 0; kt < 5; kt++)
#pragma unroll
        for (int g = 0; g < NG; g++) Ma[kt][g] = e[(kt * SG + 8 * g) * 4];
      Fv = T0 + kFr;
    }
    hadamard(Ma, Mb, cur);
    if (h.w >= 0) {
      double* d = my_D + (size_t)h.w * slot_stride;
#pragma unroll
      for (int kt = 0; kt < 5; kt++)
#pragma unroll
        for (int g = 0; g < NG; g++) d[(kt * SG + 8 * g) * 4] = cur[kt][g];
    }
    if (flags & kDownPush) {
      double M[5][NG];
      matvec20(Fv, lane, cur, M);
      double* e = my_stack + (size_t)((flags >> 24) & 0xff) * (SG * 20);
#pragma unroll
      for (int kt = 0; kt < 5; kt++)
#pragma unroll
        for (int g = 0; g < NG; g++) e[(kt * SG + 8 * g) * 4] = M[kt][g];
    }
    __syncwarp();
    if (lane == 0) mbar_arrive(&stg_empty[cs]);
    if (++cs == (uint32_t)NSTG) { cs = 0; cph ^= 1; }
  }
  // ---- root: class likelihood L_c = sum_x pi_x root[x]
#pragma unroll
  for (int g = 0; g < NG; g++) {
    double v = 0.;
#pragma unroll
    for (int kt = 0; kt < 5; kt++) v = fma(cur[kt][g], __ldg(m.pi + 4 * kt + q), v);
    v += __shfl_xor_sync(0xffffffffu, v, 1);
    v += __shfl_xor_sync(0xffffffffu, v, 2);
    if (q == 0) b.Lc[(size_t)cls * n_pad + site0 + lsite + 8 * g] = v;
  }
}

int max_smem_optin() {
  int dev = 0, v = 0;
  CMB_CUDA(cudaGetDevice(&dev));
  CMB_CUDA(cudaDeviceGetAttribute(&v, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev));
  return v;
}

template <int MINB, bool STATES>
bool try_up20(const MapModel& m, const MapBuffers& b, const DevStream& s, double* part, cudaStream_t st) {
  const int max_smem = max_smem_optin() / MINB - 1024 - 1024;
  const size_t stage = ((size_t)s.stage_bytes + 127) & ~size_t(127);
  if ((size_t)max_smem < 128 + 2 * stage) return false;
  Up20Params up;
  up.stream = s.bytes.as<unsigned char>(); up.rec_off = s.off.as<uint32_t>(); up.rec_bytes = s.nbytes.as<uint32_t>();
  up.refs = s.aux.as<int4>(); up.part = part; up.n_nodes = s.n_records; up.stage_bytes = (uint32_t)stage; up.B = m.B;
  // the message stack and a few spills live in local memory behind the L1 that shared memory is carved from
  // (k1_mma.cu measured a ring beyond ~80 KB per CTA slower at two CTAs per SM)
  const size_t ring = MINB > 1 ? std::min<size_t>((size_t)max_smem - 128, 96 * 1024) : (size_t)max_smem - 128;
  up.n_stages = (int)std::max<size_t>(2, std::min<size_t>(kStages20, ring / stage));
  const size_t smem = 128 + (size_t)up.n_stages * stage;
  if (smem > (size_t)max_smem) return false;
  CMB_CUDA(cudaFuncSetAttribute(k1_up_mma20<MINB, STATES>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  k1_up_mma20<MINB, STATES><<<dim3((unsigned)(b.n_pad / SG), (unsigned)m.C), 32 * (W + 1), smem, st>>>(m, b, up);
  CMB_CUDA(cudaGetLastError());
  return true;
}

template <int MINB, bool STATES>
bool try_down20(const MapModel& m, const MapBuffers& b, const DevStream& s, cudaStream_t st) {
  const int max_smem = max_smem_optin() / MINB - 1024 - 1024;
  const size_t stage = (size_t)s.cap + 2 * (size_t)SG, level = (size_t)SG * 160;
  Down20Params dp;
  dp.stream = s.bytes.as<unsigned char>(); dp.rec_off = s.off.as<uint32_t>(); dp.rec_bytes = s.nbytes.as<uint32_t>();
  dp.refs = s.aux.as<int4>(); dp.n_nodes = s.n_records; dp.rec_cap = s.cap;
  const size_t stack = (size_t)std::max(1, s.stack_depth) * level;
  dp.n_stages = kStages20;
  while (dp.n_stages > 2 && 128 + dp.n_stages * stage + stack > (size_t)max_smem) dp.n_stages /= 2;
  const size_t smem = 128 + dp.n_stages * stage + stack;
  if (smem > (size_t)max_smem) return false;
  CMB_CUDA(cudaFuncSetAttribute(k1_down_mma20<MINB, STATES>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  k1_down_mma20<MINB, STATES><<<dim3((unsigned)(b.n_pad / SG), (unsigned)m.C), 32 * (W + 1), smem, st>>>(m, b, dp);
  CMB_CUDA(cudaGetLastError());
  return true;
}

} // namespace

// false: no launch shape fits.  cmb_map reports that as an error: it does not fall back to the scalar kernels.
// Context::ensure_streams sends trees deeper than 12 levels there up front, and on a B200 (227 KB per CTA)
// one CTA per SM holds a 12-level stack (120 KB) with 8 stages, so the error is not reached there.
bool launch_map_down_mma20(const MapModel& m, const MapBuffers& b, const DevStream& s, cudaStream_t st) {
  if (m.A != 20 || b.n_pad % SG) return false;
  if (m.states_only) return try_down20<2, true>(m, b, s, st) || try_down20<1, true>(m, b, s, st);
  return try_down20<2, false>(m, b, s, st) || try_down20<1, false>(m, b, s, st);
}
bool launch_map_up_mma20(const MapModel& m, const MapBuffers& b, const DevStream& s, double* part, cudaStream_t st) {
  if (m.A != 20 || b.n_pad % SG) return false;
  const bool ok = m.states_only ? (try_up20<2, true>(m, b, s, part, st) || try_up20<1, true>(m, b, s, part, st))
                                : (try_up20<2, false>(m, b, s, part, st) || try_up20<1, false>(m, b, s, part, st));
  if (!ok) return false;
  const int64_t n = (int64_t)m.B * b.n_pad;
  k1_sum_classes<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(m.C, m.B, b.n_pad, part, b.out);
  CMB_CUDA(cudaGetLastError());
  return true;
}

} // namespace cmb
