// K4: agglomerative clustering of sites on the device.
//
// Replaces Bio++ HierarchicalClustering(method, matrix, rootTree = false) + computeTree()
// (call sites CoMap.cpp:460-485, ClusterTools.cpp:260-262; SURVEY.md s8 a14):
//   repeat while more than two clusters live: take the FIRST strictly smallest entry over
//   live pairs i<j in id order; the parent takes slot i, slot j dies; distances to every
//   other live k become w1 d(i,k) + w2 d(j,k) + w4 |d(i,k) - d(j,k)| with
//   (.5,.5,+.5) complete, (.5,.5,-.5) single, (n_i/(n_i+n_j), n_j/(n_i+n_j), 0) average;
//   height(parent) = d(i,j)/2; the last two clusters are joined at d/2.
// The reference rescans the whole matrix per merge (O(S^3)); here one persistent
// cooperative kernel keeps, per live row, the first minimum over live columns j>i
// (value + column), so a merge costs an argmin over S cached row minima, one row/column
// update and a rescan of the few rows whose cached minimum was invalidated -- O(S^2)
// in the common case -- with the reference's tie-breaking preserved exactly.
#include "kernels.h"
#include <algorithm>
#include <cstdlib>
#include <string>
#include <cooperative_groups.h>

namespace cg = cooperative_groups;

namespace cmb {
namespace {

constexpr int CT = 512;

struct ClusterParams {
  int64_t S;
  int linkage;
  double* mat;          // [S][S] symmetric, consumed
  double* rmin_val;     // [S] first minimum over live j>i
  int32_t* rmin_idx;    // [S] its column, -1 if none
  uint8_t* alive;       // [S]
  double* len;          // [S] height of the cluster in the slot
  int32_t* nleaves;     // [S]
  int32_t* node;        // [S] dendrogram node in the slot
  int32_t* wl;          // [2][S] worklist: rows whose cached minimum has to be rescanned
  double* part_val;     // [grid] per-CTA first minimum of the new row a
  int32_t* part_idx;
  double* scan_val;     // [grid] per-CTA first minimum of its slice of the cached row minima
  int32_t* scan_idx;
  int32_t* scan_col;     // [grid] ... and the column of that minimum (saves a dependent load after the grid sync)
  double* seg_val;      // [grid] partial minima of row segments (a queued row is rescanned by several CTAs)
  int32_t* seg_idx;
  int32_t* seg_cnt;     // [grid] segments of a queued row finished so far
  int32_t* wl_count;    // [2]
  int32_t *left, *right; // [S-1]
  double* height;       // [S-1]
};

struct Best { double v; int i; };
__device__ __forceinline__ bool better(double v, int i, const Best& b) {
  return b.i < 0 || v < b.v || (v == b.v && i < b.i);
}
// Warp argmin with smallest-index tie-break in three REDUX steps on an order-preserving integer
// image of the double (high word, low word, index) instead of five shuffle + fp64-compare rounds;
// the result is valid in every lane.  -0.0 is folded into +0.0 first (they compare equal).
__device__ __forceinline__ Best warp_best(Best b) {
  const bool has = b.i >= 0;
  const long long bits = __double_as_longlong(__dadd_rn(b.v, 0.));
  const unsigned long long k = has ? (unsigned long long)(bits ^ ((bits >> 63) | (long long)0x8000000000000000ull)) : ~0ull;
  const unsigned hi = (unsigned)(k >> 32), lo = (unsigned)k;
  const unsigned mhi = __reduce_min_sync(0xffffffffu, hi);
  const unsigned mlo = __reduce_min_sync(0xffffffffu, hi == mhi ? lo : 0xffffffffu);
  const unsigned mi = __reduce_min_sync(0xffffffffu, has && hi == mhi && lo == mlo ? (unsigned)b.i : 0xffffffffu);
  if (mi == 0xffffffffu) return Best{0., -1};
  const unsigned long long mk = ((unsigned long long)mhi << 32) | mlo;
  const long long mb = (mk >> 63) ? (long long)(mk ^ 0x8000000000000000ull) : (long long)~mk;
  return Best{__longlong_as_double(mb), (int)mi};
}
// block-wide argmin with smallest-index tie-break; result valid in every thread
__device__ Best block_best(Best b, Best* sh) {
  b = warp_best(b);
  const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
  __syncthreads();
  if (l == 0) sh[w] = b;
  __syncthreads();
  return warp_best(l < (int)(blockDim.x >> 5) ? sh[l] : Best{0., -1}); // every warp reduces the warp results itself
}

// first minimum of row r over live columns j>r (skipping `skip`).  The loads of a batch of
// U columns per thread are issued together (liveness byte and matrix entry are independent),
// so a 160 KB row costs a few L2 round trips instead of one per column.
__device__ Best scan_columns(const ClusterParams& p, int r, int skip, int64_t lo, int64_t hi, Best* sh) {
  constexpr int U = 8;
  Best b{0., -1};
  const double* row = p.mat + (size_t)r * p.S;
  for (int64_t base = lo; base < hi; base += (int64_t)blockDim.x * U) {
    double v[U];
    uint8_t al[U];
#pragma unroll
    for (int u = 0; u < U; u++) {
      const int64_t j = base + (int64_t)u * blockDim.x + threadIdx.x;
      al[u] = j < hi ? p.alive[j] : 0;
      v[u] = j < hi ? row[j] : 0.;
    }
#pragma unroll
    for (int u = 0; u < U; u++) {
      const int64_t j = base + (int64_t)u * blockDim.x + threadIdx.x;
      if (al[u] && j != skip && !(v[u] != v[u]) && better(v[u], (int)j, b)) { b.v = v[u]; b.i = (int)j; }
    }
  }
  return block_best(b, sh);
}
__device__ void rescan_row(const ClusterParams& p, int r, int skip, Best* sh) {
  const Best b = scan_columns(p, r, skip, r + 1, p.S, sh);
  if (threadIdx.x == 0) { p.rmin_val[r] = b.v; p.rmin_idx[r] = b.i; }
}

__global__ void __launch_bounds__(CT) k4_init_rows(ClusterParams p) {
  __shared__ Best sh[32];
  for (int r = blockIdx.x; r < p.S; r += gridDim.x) {
    rescan_row(p, r, -1, sh);
    __syncthreads();
  }
}

// One merge = (1) every CTA finds the first global minimum among the cached row minima
// (dead rows carry index -1); (A) the grid rewrites row / column a, updates in place the cached
// minimum of every row k < a that only has to compare its new entry, queues the rows whose
// cached minimum pointed at a or b for a rescan, and reduces the new row a's own minimum on the
// fly (per-CTA partial); grid sync; (B) bookkeeping, row a's minimum from the partials, rescans;
// grid sync.  ncu / clock64 on config 5 (S = 20 000) before this layout: 73 us per merge, of
// which 21 us in (1) and 47 us in serial rescans of row a and ~40 queued rows.  Now (-DCMB_K4_TIMING,
// cycles per merge on a mid-grid CTA): scan 3300 | barrier 2800 | combine 3400 | update 1400 |
// barrier 6400 (waits for CTA 0's 4000) | rescans 2800 (slowest CTA 8200) | barrier 10000.  A barrier
// costs ~2500 cycles and a round trip to data another SM has just written ~1000, whatever the grid
// size (16..148 CTAs measured the same).  A two-barrier variant that rescans a queued row inside the
// CTA that found it (kept as tools/experiments/k4_two_barrier_variant.cu.txt, parity-green) was slower, 29 us per
// merge: one CTA needs five dependent batches per 160 KB row while the rest of the grid waits.  Per-CTA
// queue slots instead of the global atomic worklist, and keeping block 0 out of the row update, changed
// nothing either: the second barrier costs 6000 cycles with or without them (its fence waits for the
// scattered column-a stores).  What did help: argmin reductions through REDUX on an order-preserving
// integer image of the doubles instead of shuffle + fp64-compare rounds (every phase ends in one):
// 15.5 -> 12 us per merge (scan 1800 | barrier 2700 | combine 2000 | update 730 | barrier 4900 |
// rescans 2300, slowest CTA 6700 | barrier 8200).  A hand-written barrier (red.release.gpu on a monotone
// counter + ld.acquire.gpu poll) instead of cooperative_groups' grid.sync() measured the same 2700 cycles.
// NP independent dendrograms (replicates of the clustering null) advance in lock step through the same
// three barriers: a merge is a chain of barrier and memory latencies, not work, so a second and a
// fourth problem ride along almost for free.
constexpr int kMaxBatch = 4;
struct ClusterBatch { ClusterParams p[kMaxBatch]; };

template <int NP>
__device__ __forceinline__ void block_best_n(Best (&b)[NP], Best (*sh)[32]) {
  const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
#pragma unroll
  for (int q = 0; q < NP; q++) b[q] = warp_best(b[q]);
  __syncthreads();
  if (l == 0) {
#pragma unroll
    for (int q = 0; q < NP; q++) sh[q][w] = b[q];
  }
  __syncthreads();
  if constexpr (NP == 1) { // every warp reduces the warp results itself: no third barrier
    b[0] = warp_best(l < (int)(blockDim.x >> 5) ? sh[0][l] : Best{0., -1});
  } else {                 // REDUX issue is the limit with 3 NP per warp: one warp reduces, all read
    if (w == 0) {
#pragma unroll
      for (int q = 0; q < NP; q++) {
        const Best t = warp_best(l < (int)(blockDim.x >> 5) ? sh[q][l] : Best{0., -1});
        if (l == 0) sh[q][0] = t;
      }
    }
    __syncthreads();
#pragma unroll
    for (int q = 0; q < NP; q++) b[q] = sh[q][0];
  }
}

template <int NP>
__global__ void __launch_bounds__(CT) k4_cluster(const __grid_constant__ ClusterBatch B) {
  cg::grid_group grid = cg::this_grid();
  __shared__ Best sh[NP][32];
  __shared__ int sh_col[NP];
  const int64_t S = B.p[0].S;
  const int linkage = B.p[0].linkage;
  const int G = (int)gridDim.x;
  const int64_t gtid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x, gsz = (int64_t)G * blockDim.x;
  const int64_t per = (S + G - 1) / G, lo = (int64_t)blockIdx.x * per, hi = lo + per < S ? lo + per : S;
#ifdef CMB_K4_TIMING
  long long tacc[8] = {0, 0, 0, 0, 0, 0, 0, 0}, t0 = 0, t1 = 0;
#define K4_T(slot) { t1 = clock64(); tacc[slot] += t1 - t0; t0 = t1; }
#else
#define K4_T(slot)
#endif
  for (int64_t step = 0; step + 2 < S; step++) {
#ifdef CMB_K4_TIMING
    t0 = clock64();
#endif
    // (1) first global minimum of the cached row minima: every CTA scans its slice (the loads of
    //     all problems are issued together), publishes (value, row, column), grid barrier, then all
    //     CTAs reduce the per-CTA partials
    Best b[NP];
    int my_i[NP], my_col[NP];
    {
      int ix0[NP]; double v0[NP];
      const int64_t i0 = lo + threadIdx.x;
#pragma unroll
      for (int q = 0; q < NP; q++) {
        ix0[q] = -1; v0[q] = 0.;
        if (i0 < hi) { ix0[q] = B.p[q].rmin_idx[i0]; v0[q] = B.p[q].rmin_val[i0]; }
      }
#pragma unroll
      for (int q = 0; q < NP; q++) {
        b[q] = Best{0., -1}; my_col[q] = -1;
        if (ix0[q] >= 0) { b[q].v = v0[q]; b[q].i = (int)i0; my_col[q] = ix0[q]; }
        for (int64_t i = i0 + blockDim.x; i < hi; i += blockDim.x) { // only above S = grid x block
          const int ix = B.p[q].rmin_idx[i];
          const double v = B.p[q].rmin_val[i];
          if (ix >= 0 && better(v, (int)i, b[q])) { b[q].v = v; b[q].i = (int)i; my_col[q] = ix; }
        }
        my_i[q] = b[q].i;
      }
    }
    block_best_n<NP>(b, sh);
#pragma unroll
    for (int q = 0; q < NP; q++) {
      if (threadIdx.x == 0) { B.p[q].scan_val[blockIdx.x] = b[q].v; B.p[q].scan_idx[blockIdx.x] = b[q].i; }
      if (my_i[q] >= 0 && my_i[q] == b[q].i) B.p[q].scan_col[blockIdx.x] = my_col[q]; // a row belongs to one thread
    }
    K4_T(0)
    grid.sync();
    K4_T(1)
    // the column travels with the partial, so no load depends on the reduced row index
    {
      int pi0[NP], pc0[NP]; double pv0[NP];
      const int c0 = (int)threadIdx.x;
#pragma unroll
      for (int q = 0; q < NP; q++) { // one round trip for all problems
        pi0[q] = -1; pc0[q] = -1; pv0[q] = 0.;
        if (c0 < G) { pi0[q] = B.p[q].scan_idx[c0]; pv0[q] = B.p[q].scan_val[c0]; pc0[q] = B.p[q].scan_col[c0]; }
      }
#pragma unroll
      for (int q = 0; q < NP; q++) {
        b[q] = Best{0., -1};
        if (pi0[q] >= 0) { b[q].v = pv0[q]; b[q].i = pi0[q]; my_col[q] = pc0[q]; }
        for (int c = c0 + (int)blockDim.x; c < G; c += blockDim.x) { // only on grids above one block's threads
          const int i = B.p[q].scan_idx[c];
          const double v = B.p[q].scan_val[c];
          const int col = B.p[q].scan_col[c];
          if (i >= 0 && better(v, i, b[q])) { b[q].v = v; b[q].i = i; my_col[q] = col; }
        }
        my_i[q] = b[q].i;
      }
    }
    block_best_n<NP>(b, sh);
    int a[NP], bb[NP];
    double dab[NP], w1[NP], w2[NP], w4[NP];
    bool none = false;
#pragma unroll
    for (int q = 0; q < NP; q++) {
      a[q] = b[q].i;
      none |= a[q] < 0;
      if (a[q] >= 0 && my_i[q] == a[q]) sh_col[q] = my_col[q]; // rows are unique across the partials: one writer
    }
    if (none) return; // nothing mergeable (NaN distances), the same in every CTA: host reports the error
    __syncthreads();
#pragma unroll
    for (int q = 0; q < NP; q++) {
      bb[q] = sh_col[q];
      dab[q] = b[q].v;
      if (linkage == 1) { w1[q] = .5; w2[q] = .5; w4[q] = -.5; }
      else if (linkage == 0) { w1[q] = .5; w2[q] = .5; w4[q] = .5; }
      else {
        double na = (double)B.p[q].nleaves[a[q]], nb = (double)B.p[q].nleaves[bb[q]];
        w1[q] = na / (na + nb); w2[q] = nb / (na + nb); w4[q] = 0.;
      }
    }
    K4_T(2)
    // (A) new distances to the merged cluster (slot a).  After the barrier the cached minimum of row k is
    //     read and written by the thread that owns k only, so a row that only sees a new column compares in
    //     place; rows whose minimum pointed at a or bb are queued; the new row a's own minimum is reduced on
    //     the fly (per-CTA partial)
    Best ra[NP];
    {
      uint8_t live0[NP]; double d10[NP], d20[NP], cv0[NP]; int ci0[NP];
      // the CTA that owns the lowest rows is the slowest of this phase (most of the queue atomics are
      // its): each problem deals its rows to the CTAs with a different rotation
      int64_t k0[NP];
#pragma unroll
      for (int q = 0; q < NP; q++) { // one round trip for all problems
        k0[q] = gtid + (int64_t)q * (G / NP) * blockDim.x;
        if (k0[q] >= gsz) k0[q] -= gsz;
        live0[q] = 0; d10[q] = d20[q] = cv0[q] = 0.; ci0[q] = -1;
        if (k0[q] < S) {
          live0[q] = B.p[q].alive[k0[q]];
          d10[q] = B.p[q].mat[(size_t)a[q] * S + k0[q]]; d20[q] = B.p[q].mat[(size_t)bb[q] * S + k0[q]];
          ci0[q] = B.p[q].rmin_idx[k0[q]]; cv0[q] = B.p[q].rmin_val[k0[q]];
        }
      }
#pragma unroll
      for (int q = 0; q < NP; q++) {
        const ClusterParams& p = B.p[q];
        int32_t* wl = p.wl + (step & 1) * S;
        int32_t* wlc = p.wl_count + (step & 1);
        ra[q] = Best{0., -1};
        const int aq = a[q], bq = bb[q];
        auto row = [&](int64_t k, uint8_t live, double d1, double d2, int ci, double cv) {
          if (k == aq || k == bq || !live) return;
          // left-to-right, unfused, as the reference's C++ expression evaluates
          const double nd = __dadd_rn(__dadd_rn(__dadd_rn(__dmul_rn(w1[q], d1), __dmul_rn(w2[q], d2)), __dmul_rn(0., dab[q])),
                                      __dmul_rn(w4[q], fabs(__dadd_rn(d1, -d2))));
          p.mat[(size_t)aq * S + k] = nd;
          p.mat[(size_t)k * S + aq] = nd;
          if (k > aq) {
            if (!(nd != nd) && better(nd, (int)k, ra[q])) { ra[q].v = nd; ra[q].i = (int)k; }
            if (k < bq && ci == bq) wl[atomicAdd(wlc, 1)] = (int32_t)k;  // lost its minimum's column
          } else {
            if (ci == aq || ci == bq) wl[atomicAdd(wlc, 1)] = (int32_t)k; // minimum pointed at a merged slot
            else if (!(nd != nd) && (ci < 0 || nd < cv || (nd == cv && aq < ci))) { p.rmin_val[k] = nd; p.rmin_idx[k] = aq; }
          }
        };
        if (k0[q] < S) row(k0[q], live0[q], d10[q], d20[q], ci0[q], cv0[q]);
        for (int64_t k = k0[q] + gsz; k < S; k += gsz) // only above S = grid x block
          row(k, p.alive[k], p.mat[(size_t)aq * S + k], p.mat[(size_t)bq * S + k], p.rmin_idx[k], p.rmin_val[k]);
      }
    }
    block_best_n<NP>(ra, sh);
    if (threadIdx.x == 0) {
#pragma unroll
      for (int q = 0; q < NP; q++) { B.p[q].part_val[blockIdx.x] = ra[q].v; B.p[q].part_idx[blockIdx.x] = ra[q].i; }
    }
    K4_T(3)
    grid.sync();
    K4_T(4)
    // (B) bookkeeping and row a's cached minimum from the per-CTA partials (block 0), queued rescans
    int n_wl[NP], n_all = 0;
#pragma unroll
    for (int q = 0; q < NP; q++) n_wl[q] = B.p[q].wl_count[step & 1];
    if (blockIdx.x == 0) {
      // slot state of a and bb, loaded before the reduction of the partials hides their latency
      double len_a[NP]; int node_a[NP], node_b[NP], nl_a[NP], nl_b[NP];
      Best t[NP];
#pragma unroll
      for (int q = 0; q < NP; q++) {
        const ClusterParams& p = B.p[q];
        len_a[q] = 0.; node_a[q] = node_b[q] = nl_a[q] = nl_b[q] = 0;
        if (threadIdx.x == 0) { len_a[q] = p.len[a[q]]; node_a[q] = p.node[a[q]]; node_b[q] = p.node[bb[q]]; nl_a[q] = p.nleaves[a[q]]; nl_b[q] = p.nleaves[bb[q]]; }
        t[q] = Best{0., -1};
      }
      {
        int pi0[NP]; double pv0[NP];
        const int c0 = (int)threadIdx.x;
#pragma unroll
        for (int q = 0; q < NP; q++) { // one round trip for all problems
          pi0[q] = -1; pv0[q] = 0.;
          if (c0 < G) { pi0[q] = B.p[q].part_idx[c0]; pv0[q] = B.p[q].part_val[c0]; }
        }
#pragma unroll
        for (int q = 0; q < NP; q++) {
          if (pi0[q] >= 0) { t[q].v = pv0[q]; t[q].i = pi0[q]; }
          for (int c = c0 + (int)blockDim.x; c < G; c += blockDim.x) {
            const int i = B.p[q].part_idx[c];
            const double v = B.p[q].part_val[c];
            if (i >= 0 && better(v, i, t[q])) { t[q].v = v; t[q].i = i; }
          }
        }
      }
      block_best_n<NP>(t, sh);
      if (threadIdx.x == 0) {
#pragma unroll
        for (int q = 0; q < NP; q++) {
          const ClusterParams& p = B.p[q];
          const double half = dab[q] / 2.;
          const double d0 = half - len_a[q];
          p.left[step] = node_a[q];
          p.right[step] = node_b[q];
          p.height[step] = len_a[q] + d0;
          p.node[a[q]] = (int32_t)(S + step);
          p.len[a[q]] = len_a[q] + d0;
          p.nleaves[a[q]] = nl_a[q] + nl_b[q];
          p.alive[bb[q]] = 0;
          p.rmin_idx[bb[q]] = -1;  // dead rows drop out of (1)
          p.rmin_val[a[q]] = t[q].v;
          p.rmin_idx[a[q]] = t[q].i;
          p.wl_count[(step + 1) & 1] = 0;
        }
      }
      __syncthreads();
    }
#pragma unroll
    for (int q = 0; q < NP; q++) n_all += n_wl[q];
    // Every queued row (of any problem) is rescanned by nseg CTAs (one batch of loads each instead of up
    // to five dependent ones); the CTA that finishes a row's last segment combines the partial minima.
    const int nseg = n_all > 0 && n_all * 2 <= G ? (G / n_all < 8 ? G / n_all : 8) : 1;
    // block 0 is busy with the bookkeeping: the work starts at the other end of the grid
    for (int it = G - 1 - (int)blockIdx.x; it < n_all * nseg; it += G) {
      const int w_all = it / nseg, seg = it % nseg;
      int q = 0, w = w_all;
#pragma unroll
      for (int qq = 0; qq < NP - 1; qq++)
        if (q == qq && w >= n_wl[qq]) { w -= n_wl[qq]; q = qq + 1; }
      const ClusterParams& p = B.p[q];
      const int skip = bb[q];
      const int r = (p.wl + (step & 1) * S)[w];
      if (nseg == 1) rescan_row(p, r, skip, sh[0]);
      else {
        const ClusterParams& p0 = B.p[0]; // segment scratch of problem 0 serves the whole batch
        const int64_t L = S - r - 1, slo = r + 1 + L * seg / nseg, shi = r + 1 + L * (seg + 1) / nseg;
        const Best t = scan_columns(p, r, skip, slo, shi, sh[0]);
        __shared__ int last;
        if (threadIdx.x == 0) {
          p0.seg_val[w_all * nseg + seg] = t.v;
          p0.seg_idx[w_all * nseg + seg] = t.i;
          __threadfence();
          last = atomicAdd(&p0.seg_cnt[w_all], 1) == nseg - 1;
        }
        __syncthreads();
        if (last && threadIdx.x < 32) {
          __threadfence();
          Best c{0., -1};
          if ((int)threadIdx.x < nseg) {
            c.i = __ldcg(&p0.seg_idx[w_all * nseg + threadIdx.x]);
            c.v = __ldcg(&p0.seg_val[w_all * nseg + threadIdx.x]);
          }
          c = warp_best(c);
          if (threadIdx.x == 0) { p.rmin_val[r] = c.v; p.rmin_idx[r] = c.i; p0.seg_cnt[w_all] = 0; }
        }
      }
      __syncthreads();
    }
    K4_T(5)
    grid.sync();
    K4_T(6)
  }
#ifdef CMB_K4_TIMING
  if (threadIdx.x == 0 && (blockIdx.x == 0 || blockIdx.x == 77 || blockIdx.x == gridDim.x - 1))
    printf("k4 timing cta %d: scan %lld sync1 %lld combine %lld update %lld sync2 %lld rescans %lld sync3 %lld (cycles per step of %d merges)\n",
           blockIdx.x, tacc[0] / (S - 2), tacc[1] / (S - 2), tacc[2] / (S - 2), tacc[3] / (S - 2), tacc[4] / (S - 2), tacc[5] / (S - 2), tacc[6] / (S - 2), NP);
#endif
  // finalStep: join the last two clusters at d/2
  if (gtid < NP) {
    const ClusterParams& p = B.p[gtid];
    int i1 = -1, i2 = -1;
    for (int64_t i = 0; i < S; i++)
      if (p.alive[i]) { if (i1 < 0) i1 = (int)i; else i2 = (int)i; }
    const double d = p.mat[(size_t)i1 * S + i2] / 2;
    p.left[S - 2] = p.node[i1];
    p.right[S - 2] = p.node[i2];
    p.height[S - 2] = p.len[i1] + (d - p.len[i1]);
  }
}

// ---- the same merge loop inside ONE thread-block cluster ----------------------------------
// A grid barrier costs ~2500 cycles and every exchange through global memory ~1000 more; a merge
// has three of each.  Sixteen CTAs of one cluster hold the cached row minima in their shared memory
// (slice r of the rows in CTA r), exchange partial minima and the rescan queue with remote
// shared-memory stores and meet at cluster barriers; only the matrix itself stays in HBM / L2.
// Per merge: (P1) slice argmin -> partial to every CTA; barrier; (P2) every CTA reduces the 16
// partials, updates row / column a for the rows of its slice (cached minima local), sends its
// partial of the new row a to that row's owner and its queued rows to everybody; barrier; (P3) queued
// rows are dealt round-robin, each rescanned by one CTA, result stored into the owner's cache;
// barrier.  Measured (S = 20 000, cycles per merge): slice argmin 2100 | barrier 1100 | reduce 1250 | update 3600 |
// publish 2700 | barrier 1500+ | rescans up to 13 000 on the CTAs that hold a row | barrier: 16 us per merge.
// Splitting every queued row over the 16 CTAs (as the grid kernel does) is the missing step; until then the
// grid kernel is the default and this one is selected with CMB_K4_LAYOUT=cluster.
constexpr int NC = 16, NT = 1024, QMAX = 8;

struct DsmLayout {
  int per; size_t o_rv, o_pv, o_rav, o_ri, o_pi, o_pc, o_rai, o_rn, o_rl, o_ovf, o_alive, bytes;
  __host__ __device__ explicit DsmLayout(int64_t S) {
    per = (int)((S + NC - 1) / NC);
    size_t o = 0;
    o_rv = o; o += 8 * (size_t)per; o_pv = o; o += 8 * NC; o_rav = o; o += 8 * NC;
    o_ri = o; o += 4 * (size_t)per; o_pi = o; o += 4 * NC; o_pc = o; o += 4 * NC; o_rai = o; o += 4 * NC;
    o_rn = o; o += 4 * NC; o_rl = o; o += 4 * NC * QMAX; o_ovf = o; o += 4 * (size_t)per;
    o_alive = o; o += (size_t)S; bytes = (o + 15) & ~size_t(15);
  }
};

__device__ Best scan_row_dsm(const double* __restrict__ row, const uint8_t* alive_s, int r, int64_t S, Best* sh) {
  constexpr int U = 10; // 10 240 columns per batch of loads
  Best b{0., -1};
  for (int64_t base = r + 1; base < S; base += (int64_t)NT * U) {
    double v[U];
#pragma unroll
    for (int u = 0; u < U; u++) {
      const int64_t j = base + (int64_t)u * NT + threadIdx.x;
      v[u] = j < S ? row[j] : 0.;
    }
#pragma unroll
    for (int u = 0; u < U; u++) {
      const int64_t j = base + (int64_t)u * NT + threadIdx.x;
      if (j < S && alive_s[j] && !(v[u] != v[u]) && better(v[u], (int)j, b)) { b.v = v[u]; b.i = (int)j; }
    }
  }
  return block_best(b, sh);
}

__global__ void __launch_bounds__(NT, 1) k4_cluster_dsm(ClusterParams p) {
  cg::cluster_group cluster = cg::this_cluster();
  const int rank = (int)cluster.block_rank(), tid = (int)threadIdx.x;
  extern __shared__ __align__(16) unsigned char dsm[];
  __shared__ Best sh[32];
  __shared__ int sh_col, sh_a, sh_bb, rs_n, sh_ntot, sh_list[NC * QMAX], rs_loc[QMAX];
  __shared__ double sh_d;
  const int64_t S = p.S;
  const DsmLayout L(S);
  const int per = L.per, lo = rank * per, hi = (int)((int64_t)lo + per < S ? lo + per : S);
  double* rv = (double*)(dsm + L.o_rv); double* pv = (double*)(dsm + L.o_pv); double* rav = (double*)(dsm + L.o_rav);
  int* ri = (int*)(dsm + L.o_ri); int* pi = (int*)(dsm + L.o_pi); int* pc = (int*)(dsm + L.o_pc);
  int* rai = (int*)(dsm + L.o_rai); int* rn = (int*)(dsm + L.o_rn); int* rl = (int*)(dsm + L.o_rl);
  int* ovf = (int*)(dsm + L.o_ovf); uint8_t* alive_s = dsm + L.o_alive;
  for (int i = lo + tid; i < hi; i += NT) { rv[i - lo] = p.rmin_val[i]; ri[i - lo] = p.rmin_idx[i]; }
  for (int64_t i = tid; i < S; i += NT) alive_s[i] = 1;
  __syncthreads();
  cluster.sync(); // every CTA of the cluster is running: remote shared memory may be written
#ifdef CMB_K4_TIMING
  long long tacc[8] = {0, 0, 0, 0, 0, 0, 0, 0}, t0 = 0, t1 = 0;
#endif
  for (int64_t step = 0; step + 2 < S; step++) {
#ifdef CMB_K4_TIMING
    t0 = clock64();
#endif
    // (P1) first minimum of this CTA's slice of the cached row minima, published to every CTA
    Best b{0., -1};
    int my_col = -1;
    for (int i = lo + tid; i < hi; i += NT) {
      const int ix = ri[i - lo];
      const double v = rv[i - lo];
      if (ix >= 0 && better(v, i, b)) { b.v = v; b.i = i; my_col = ix; }
    }
    const int my_i = b.i;
    b = block_best(b, sh);
    if (my_i >= 0 && my_i == b.i) sh_col = my_col; // a row belongs to one thread: one writer
    __syncthreads();
    if (tid < NC) {
      cluster.map_shared_rank(pv, tid)[rank] = b.v;
      cluster.map_shared_rank(pi, tid)[rank] = b.i;
      cluster.map_shared_rank(pc, tid)[rank] = b.i >= 0 ? sh_col : -1;
    }
    K4_T(0)
    cluster.sync();
    K4_T(1)
    // (P2) every CTA reduces the 16 partials
    if (tid < 32) {
      Best c{0., -1};
      int col = -1;
      if (tid < NC) { c.v = pv[tid]; c.i = pi[tid]; col = pc[tid]; }
      const Best w = warp_best(c);
      if (w.i < 0) { if (tid == 0) sh_a = -1; }
      else if (c.i == w.i) { sh_a = w.i; sh_bb = col; sh_d = w.v; } // rows are unique across the partials
      if (tid == 0) rs_n = 0;
    }
    __syncthreads();
    const int a = sh_a;
    if (a < 0) return; // nothing mergeable (NaN distances), the same in every CTA: host reports the error
    const int bb = sh_bb;
    const double dab = sh_d;
    double w1, w2, w4;
    if (p.linkage == 1) { w1 = .5; w2 = .5; w4 = -.5; }
    else if (p.linkage == 0) { w1 = .5; w2 = .5; w4 = .5; }
    else {
      double na = (double)p.nleaves[a], nb = (double)p.nleaves[bb];
      w1 = na / (na + nb); w2 = nb / (na + nb); w4 = 0.;
    }
    // dendrogram bookkeeping (rank 0, thread 0): loads now, stores in (P3)
    double len_a = 0.; int node_a = 0, node_b = 0, nl_a = 0, nl_b = 0;
    if (rank == 0 && tid == 0) { len_a = p.len[a]; node_a = p.node[a]; node_b = p.node[bb]; nl_a = p.nleaves[a]; nl_b = p.nleaves[bb]; }
    if (tid == 0) alive_s[bb] = 0; // every CTA keeps its own copy of the liveness bytes
    K4_T(2)
    Best ra{0., -1}; // first minimum of the new row a over live columns k > a (this slice)
    for (int k = lo + tid; k < hi; k += NT) {
      const int kl = k - lo;
      const uint8_t live = alive_s[k];
      const double d1 = p.mat[(size_t)a * S + k], d2 = p.mat[(size_t)bb * S + k];
      const int ci = ri[kl];
      const double cv = rv[kl];
      if (k == bb) { ri[kl] = -1; continue; } // dead rows drop out of (P1)
      if (k == a || !live) continue;
      // left-to-right, unfused, as the reference's C++ expression evaluates
      const double nd = __dadd_rn(__dadd_rn(__dadd_rn(__dmul_rn(w1, d1), __dmul_rn(w2, d2)), __dmul_rn(0., dab)),
                                  __dmul_rn(w4, fabs(__dadd_rn(d1, -d2))));
      p.mat[(size_t)a * S + k] = nd;
      p.mat[(size_t)k * S + a] = nd;
      bool rescan = false;
      if (k > a) {
        if (!(nd != nd) && better(nd, k, ra)) { ra.v = nd; ra.i = k; }
        rescan = k < bb && ci == bb;                                     // lost its minimum's column
      } else {
        if (ci == a || ci == bb) rescan = true;                         // minimum pointed at a merged slot
        else if (!(nd != nd) && (ci < 0 || nd < cv || (nd == cv && a < ci))) { rv[kl] = nd; ri[kl] = a; }
      }
      if (rescan) {
        const int q = atomicAdd(&rs_n, 1);
        if (q < QMAX) rs_loc[q] = k; else ovf[q - QMAX] = k;
      }
    }
    K4_T(3)
    ra = block_best(ra, sh); // its barriers also publish the queue and this CTA's column-a stores to the CTA
    const int n_found = rs_n, n_q = n_found < QMAX ? n_found : QMAX;
    if (tid == 0) {
      const int oa = a / per;
      cluster.map_shared_rank(rav, oa)[rank] = ra.v;
      cluster.map_shared_rank(rai, oa)[rank] = ra.i;
    }
    if (tid < NC) {
      cluster.map_shared_rank(rn, tid)[rank] = n_q;
      int* dst = cluster.map_shared_rank(rl, tid) + rank * QMAX;
      for (int q = 0; q < n_q; q++) dst[q] = rs_loc[q];
    }
    // more than QMAX queued rows in one slice (rare): rescanned here; row k changes only in column a,
    // which this CTA has just written
    for (int q = QMAX; q < n_found; q++) {
      __syncthreads();
      const int r = ovf[q - QMAX];
      const Best t = scan_row_dsm(p.mat + (size_t)r * S, alive_s, r, S, sh);
      if (tid == 0) { rv[r - lo] = t.v; ri[r - lo] = t.i; }
    }
    K4_T(4)
    cluster.sync();
    K4_T(5)
    // (P3) row a's minimum at its owner, queued rows dealt round-robin, bookkeeping
    if (a / per == rank && tid < 32) {
      Best c{0., -1};
      if (tid < NC) { c.v = rav[tid]; c.i = rai[tid]; }
      c = warp_best(c);
      if (tid == 0) { rv[a - lo] = c.v; ri[a - lo] = c.i; }
    }
    if (tid < NC * QMAX) {
      const int src = tid / QMAX, q = tid % QMAX;
      int pos = q, tot = 0;
      for (int r2 = 0; r2 < NC; r2++) { const int c = rn[r2]; if (r2 < src) pos += c; tot += c; }
      if (q < rn[src]) sh_list[pos] = rl[tid];
      if (tid == 0) sh_ntot = tot;
    }
    __syncthreads();
    const int n_tot = sh_ntot;
    for (int w = rank; w < n_tot; w += NC) {
      const int r = sh_list[w];
      const Best t = scan_row_dsm(p.mat + (size_t)r * S, alive_s, r, S, sh);
      if (tid == 0) {
        const int o = r / per;
        cluster.map_shared_rank(rv, o)[r - o * per] = t.v;
        cluster.map_shared_rank(ri, o)[r - o * per] = t.i;
      }
      __syncthreads();
    }
    if (rank == 0 && tid == 0) {
      const double half = dab / 2.;
      const double d0 = half - len_a;
      p.left[step] = node_a;
      p.right[step] = node_b;
      p.height[step] = len_a + d0;
      p.node[a] = (int32_t)(S + step);
      p.len[a] = len_a + d0;
      p.nleaves[a] = nl_a + nl_b;
    }
    K4_T(6)
    cluster.sync();
    K4_T(7)
  }
#ifdef CMB_K4_TIMING
  if (tid == 0 && (rank == 0 || rank == 7 || rank == 15))
    printf("k4 dsm timing rank %d: scan %lld b1 %lld reduce %lld update %lld publish %lld b2 %lld rescans %lld b3 %lld (cycles per merge)\n",
           rank, tacc[0] / (S - 2), tacc[1] / (S - 2), tacc[2] / (S - 2), tacc[3] / (S - 2), tacc[4] / (S - 2), tacc[5] / (S - 2), tacc[6] / (S - 2), tacc[7] / (S - 2));
#endif
  // finalStep: join the last two clusters at d/2
  if (rank == 0 && tid == 0) {
    int i1 = -1, i2 = -1;
    for (int64_t i = 0; i < S; i++)
      if (alive_s[i]) { if (i1 < 0) i1 = (int)i; else i2 = (int)i; }
    const double d = p.mat[(size_t)i1 * S + i2] / 2;
    p.left[S - 2] = p.node[i1];
    p.right[S - 2] = p.node[i2];
    p.height[S - 2] = p.len[i1] + (d - p.len[i1]);
  }
}

// launches the cluster kernel when its shared-memory caches fit and the device can place the cluster
bool try_cluster_dsm(ClusterParams& p, cudaStream_t st) {
  // opt-in (CMB_K4_LAYOUT=cluster): parity-green, but at S = 20 000 it needs 16 us per merge against 12 us for
  // the grid kernel -- a queued row is rescanned by ONE CTA (13 000 cycles) while the other 15 wait
  const char* e = std::getenv("CMB_K4_LAYOUT");
  if (!e || std::string(e) != "cluster") return false;
  const DsmLayout L(p.S);
  if (L.bytes > 200 * 1024) return false;
  if (cudaFuncSetAttribute(k4_cluster_dsm, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)L.bytes) != cudaSuccess ||
      cudaFuncSetAttribute(k4_cluster_dsm, cudaFuncAttributeNonPortableClusterSizeAllowed, 1) != cudaSuccess) {
    cudaGetLastError();
    return false;
  }
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(NC); cfg.blockDim = dim3(NT); cfg.dynamicSmemBytes = L.bytes; cfg.stream = st;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeClusterDimension;
  at[0].val.clusterDim.x = NC; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
  cfg.attrs = at; cfg.numAttrs = 1;
  int n_clusters = 0;
  if (cudaOccupancyMaxActiveClusters(&n_clusters, k4_cluster_dsm, &cfg) != cudaSuccess || n_clusters < 1) {
    cudaGetLastError();
    return false;
  }
  CMB_CUDA(cudaLaunchKernelEx(&cfg, k4_cluster_dsm, p));
  return true;
}

__global__ void k4_init_state(ClusterParams p) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= p.S) return;
  p.alive[i] = 1;
  p.len[i] = 0.;
  p.nleaves[i] = 1;
  p.node[i] = (int32_t)i;
  if (i < 2) p.wl_count[i] = 0;
  if (i < p.S - 1) { p.left[i] = -1; p.right[i] = -1; p.height[i] = 0.; }
}

// Compensation group statistic (Statistics.h:267-294): 1 - ||sum_j v_j|| / sum_j ||v_j||,
// one thread per group, branches in id order, unfused arithmetic.
__global__ void k4_group_compensation(int64_t n_groups, const int32_t* __restrict__ members,
                                      const int64_t* __restrict__ offsets, int B, int64_t S_pad,
                                      const double* __restrict__ out, double* __restrict__ stat) {
  const int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= n_groups) return;
  const int64_t m0 = offsets[g], m1 = offsets[g + 1];
  double sumsq2 = 0., sumnorms = 0.;
  for (int b = 0; b < B; b++) {
    double s = 0.;
    for (int64_t m = m0; m < m1; m++) s = __dadd_rn(s, out[(size_t)b * S_pad + members[m]]);
    sumsq2 = __dadd_rn(sumsq2, __dmul_rn(s, s));
  }
  for (int64_t m = m0; m < m1; m++) {
    double q = 0.;
    for (int b = 0; b < B; b++) {
      double v = out[(size_t)b * S_pad + members[m]];
      q = __dadd_rn(q, __dmul_rn(v, v));
    }
    sumnorms = __dadd_rn(sumnorms, sqrt(q));
  }
  stat[g] = __dadd_rn(1., -(sqrt(sumsq2) / sumnorms));
}

} // namespace

namespace {
ClusterParams make_params(int64_t S, int linkage, double* mat, DevBuf& work, int32_t* left_dev, int32_t* right_dev,
                          double* height_dev, cudaStream_t st) {
  size_t o_val = 0, o_idx = align256(o_val + 8 * S), o_alive = align256(o_idx + 4 * S), o_len = align256(o_alive + S),
         o_nl = align256(o_len + 8 * S), o_node = align256(o_nl + 4 * S), o_wl = align256(o_node + 4 * S),
         o_wlc = align256(o_wl + 8 * S), o_pv = align256(o_wlc + 64), o_pi = align256(o_pv + 8 * 1024),
         o_sv = align256(o_pi + 4 * 1024), o_si = align256(o_sv + 8 * 1024), o_sc = align256(o_si + 4 * 1024),
         o_gv = align256(o_sc + 4 * 1024), o_gi = align256(o_gv + 8 * 1024), o_gc = align256(o_gi + 4 * 1024),
         o_end = align256(o_gc + 4 * 1024);
  work.reserve(o_end);
  unsigned char* w = work.as<unsigned char>();
  ClusterParams p;
  p.S = S; p.linkage = linkage; p.mat = mat;
  p.rmin_val = (double*)(w + o_val); p.rmin_idx = (int32_t*)(w + o_idx); p.alive = w + o_alive;
  p.len = (double*)(w + o_len); p.nleaves = (int32_t*)(w + o_nl); p.node = (int32_t*)(w + o_node);
  p.wl = (int32_t*)(w + o_wl); p.wl_count = (int32_t*)(w + o_wlc);
  p.part_val = (double*)(w + o_pv); p.part_idx = (int32_t*)(w + o_pi);
  p.scan_val = (double*)(w + o_sv); p.scan_idx = (int32_t*)(w + o_si); p.scan_col = (int32_t*)(w + o_sc);
  p.seg_val = (double*)(w + o_gv); p.seg_idx = (int32_t*)(w + o_gi); p.seg_cnt = (int32_t*)(w + o_gc);
  CMB_CUDA(cudaMemsetAsync(p.seg_cnt, 0, 4 * 1024, st));
  p.left = left_dev; p.right = right_dev; p.height = height_dev;
  return p;
}

template <int NP>
void launch_batch_kernel(ClusterBatch& B, int grid, cudaStream_t st) {
  int per_sm = 0;
  CMB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k4_cluster<NP>, CT, 0));
  if (per_sm < 1) fail("k4_cluster cannot be made resident");
  void* args[] = {&B};
  CMB_CUDA(cudaLaunchCooperativeKernel((void*)k4_cluster<NP>, dim3(grid), dim3(CT), args, 0, st));
}
} // namespace

// np (1..4) dendrograms over matrices of the same size, advanced in lock step by one cooperative kernel
int launch_cluster_batch(int np, int64_t S, int linkage, double* const* mats, DevBuf* works, int32_t* const* left_dev,
                         int32_t* const* right_dev, double* const* height_dev, cudaStream_t st) {
  if (np < 1 || np > kMaxBatch) fail("launch_cluster_batch: 1..%d problems per launch", kMaxBatch);
  if (cluster_rnn_selected(S, linkage)) { // rounds of reciprocal pairs: bandwidth, not a chain of barriers; no batching needed
    int n = 0;
    for (int q = 0; q < np; q++) n += launch_cluster_rnn(S, linkage, mats[q], works[q], left_dev[q], right_dev[q], height_dev[q], st);
    return n;
  }
  int dev = 0, sms = 0;
  CMB_CUDA(cudaGetDevice(&dev));
  CMB_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  const int grid = std::min(sms, 1024); // one CTA per SM
  ClusterBatch B;
  for (int q = 0; q < np; q++) {
    B.p[q] = make_params(S, linkage, mats[q], works[q], left_dev[q], right_dev[q], height_dev[q], st);
    k4_init_state<<<(unsigned)((S + 255) / 256), 256, 0, st>>>(B.p[q]);
    CMB_CUDA(cudaGetLastError());
    k4_init_rows<<<grid, CT, 0, st>>>(B.p[q]);
    CMB_CUDA(cudaGetLastError());
  }
  for (int q = np; q < kMaxBatch; q++) B.p[q] = B.p[0];
  if (np == 1 && try_cluster_dsm(B.p[0], st)) return 3;
  if (np == 1) launch_batch_kernel<1>(B, grid, st);
  else if (np == 2) launch_batch_kernel<2>(B, grid, st);
  else if (np == 3) launch_batch_kernel<3>(B, grid, st);
  else launch_batch_kernel<4>(B, grid, st);
  return 2 * np + 1;
}

int launch_cluster(int64_t S, int linkage, double* mat, DevBuf& work, int32_t* left_dev, int32_t* right_dev,
                   double* height_dev, cudaStream_t st) {
  return launch_cluster_batch(1, S, linkage, &mat, &work, &left_dev, &right_dev, &height_dev, st);
}

void launch_group_compensation(int64_t n_groups, const int32_t* members, const int64_t* offsets, int B,
                               int64_t S_pad, const double* out, double* stat, cudaStream_t st) {
  if (n_groups == 0) return;
  k4_group_compensation<<<(unsigned)((n_groups + 127) / 128), 128, 0, st>>>(n_groups, members, offsets, B, S_pad, out, stat);
  CMB_CUDA(cudaGetLastError());
}

} // namespace cmb
