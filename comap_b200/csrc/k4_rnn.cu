// K4, large matrices: agglomerative clustering by rounds of reciprocal nearest neighbours.
//
// The reference (Bio++ HierarchicalClustering + computeTree; call sites CoMap.cpp:460-485,
// ClusterTools.cpp:260-262) merges ONE pair per step: the first strictly smallest entry over live pairs i < j
// in id order.  k4_cluster.cu replays that chain literally -- 19 999 dependent steps of three grid barriers at
// S = 20 000, 12 us each, 0.24 s per dendrogram with the memory system idle.  Complete and average linkage are
// reducible (d(i u j, k) >= min(d(i,k), d(j,k))), so a pair that is each other's nearest neighbour stays so
// until it is merged, whatever happens elsewhere: all such pairs can be merged in the same round.  With the
// reference's tie-break the condition is "reciprocal FIRST minimum": j is the first index attaining the
// minimum of row i AND i the first attaining the minimum of row j.  (Ties of row i then sit at indices > j and
// ties of row j at indices > i, and under complete / average linkage a later cluster can only tie with i when
// both of its parts did, so nothing ever precedes (i, j) in the reference's scan order at that distance.)
// When no such pair exists the round merges the reference's own next pair -- the first global minimum -- so
// every round makes progress and a clique of m identical sites costs m - 1 cheap rounds.
//
// One round = collect the rows whose cached nearest neighbour is stale -> rescan them (first minimum over the
// whole row) -> list the reciprocal pairs -> rewrite the merged rows / columns with the reference's unfused
// Lance-Williams expression -> bookkeeping.  Two pairs merged in the same round meet in one entry: it is
// computed as the reference would, the merge with the smaller (distance, i, j) first.  The host then orders
// the S - 1 merges as the reference creates them (children before parents, smallest (distance, i, j) first)
// and numbers the inner nodes in that order.
//
// What is NOT identical to the sequential replay: a merge of a later round may precede, in the reference's
// order, one of an earlier round, so an entry between their clusters nests the same four Lance-Williams
// updates in another order and can differ in the last bit (0.5 a + 0.5 b + 0.5 |a - b| is not exactly
// max(a, b) in floating point).  Heights agree to 1e-12 relative instead of bit for bit, which is why the
// exact kernel stays in charge of small matrices (and of single linkage, where new ties can appear).
// ~35 rounds + one per member of the largest clique of identical sites at S = 20 000; O(S^2) bytes in total.
#include "kernels.h"
#include <cooperative_groups.h>
#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <string>
#include <tuple>
#include <vector>

namespace cg = cooperative_groups;

namespace cmb {
namespace {

constexpr int RT = 256;

struct RnnParams {
  int64_t S;
  int linkage;
  double* mat;          // [S][S] symmetric, consumed
  uint8_t* alive;       // [S]
  double* len;          // [S] height of the cluster in the slot
  int32_t* nleaves;     // [S]
  int32_t* node;        // [S] dendrogram node in the slot (leaf id, or S + merge index in creation order)
  double* nn_val;       // [S] minimum of the row over live k != i ...
  int32_t* nn_idx;      // [S] ... and the FIRST index attaining it (-1: no finite entry)
  int32_t* dirty;       // [S] cached nearest neighbour is stale (queued for the next scan)
  long long* role;      // [S] (round << 32) | 2 q (keeps its slot in pair q) or 2 q + 1 (dies in pair q); other rounds: none
  int32_t* wl;          // [2][S] worklists of stale rows, used alternately
  int32_t *pair_i, *pair_j; // [S / 2 + 2] this round's merges
  double *pair_d, *pair_w1, *pair_w2;
  double* part_v;       // [grid] per-CTA first global minimum (value, lo, hi) for rounds without a reciprocal pair
  int32_t *part_lo, *part_hi;
  double* seg_v;        // [grid] partial minima of row segments (a stale row may be scanned by several CTAs)
  int32_t *seg_i, *seg_cnt;
  int32_t* counters;    // [0..1] pairs of even / odd rounds, [2..3] stale rows queued for even / odd rounds,
                        // [4..6] the last two slots and their counter, [9] error
  int32_t *m_left, *m_right, *m_i, *m_j; // [S - 1] merge records in creation order
  double *m_height, *m_d;
};

struct Best { double v; int i; };
__device__ __forceinline__ bool better(double v, int i, const Best& b) {
  return b.i < 0 || v < b.v || (v == b.v && i < b.i);
}
__device__ __forceinline__ Best warp_best(Best b) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const double v = __shfl_xor_sync(0xffffffffu, b.v, o);
    const int i = __shfl_xor_sync(0xffffffffu, b.i, o);
    if (i >= 0 && better(v, i, b)) { b.v = v; b.i = i; }
  }
  return b;
}
__device__ Best block_best(Best b, Best* sh) {
  b = warp_best(b);
  const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
  __syncthreads();
  if (l == 0) sh[w] = b;
  __syncthreads();
  return warp_best(l < (int)(blockDim.x >> 5) ? sh[l] : Best{0., -1});
}
// first pair in the reference's scan order among the smallest values: key (value, lo, hi), lo < 0 = none
struct Cand { double v; int lo, hi; };
__device__ __forceinline__ bool cand_less(const Cand& a, const Cand& b) {
  if (a.lo < 0) return false;
  if (b.lo < 0) return true;
  return a.v < b.v || (a.v == b.v && (a.lo < b.lo || (a.lo == b.lo && a.hi < b.hi)));
}
__device__ Cand block_cand(Cand c, Cand* sh) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    Cand t;
    t.v = __shfl_xor_sync(0xffffffffu, c.v, o);
    t.lo = __shfl_xor_sync(0xffffffffu, c.lo, o);
    t.hi = __shfl_xor_sync(0xffffffffu, c.hi, o);
    if (cand_less(t, c)) c = t;
  }
  const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
  __syncthreads();
  if (l == 0) sh[w] = c;
  __syncthreads();
  c = l < (int)(blockDim.x >> 5) ? sh[l] : Cand{0., -1, -1};
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    Cand t;
    t.v = __shfl_xor_sync(0xffffffffu, c.v, o);
    t.lo = __shfl_xor_sync(0xffffffffu, c.lo, o);
    t.hi = __shfl_xor_sync(0xffffffffu, c.hi, o);
    if (cand_less(t, c)) c = t;
  }
  return c;
}

__global__ void k4r_init(RnnParams p) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < 16) p.counters[i] = i == 2 ? (int32_t)p.S : 0;   // round 0 scans every row
  if (i < 1024) p.seg_cnt[i] = 0;
  if (i >= p.S) return;
  p.alive[i] = 1; p.len[i] = 0.; p.nleaves[i] = 1; p.node[i] = (int32_t)i;
  p.dirty[i] = 0; p.role[i] = -1; p.nn_idx[i] = -1; p.nn_val[i] = 0.;
  p.wl[i] = (int32_t)i;
}

struct LW { double w1, w2, w4, dab; };
// left-to-right, unfused, as the reference's C++ expression evaluates (same as k4_cluster.cu)
__device__ __forceinline__ double lance_williams(const LW& w, double d1, double d2) {
  return __dadd_rn(__dadd_rn(__dadd_rn(__dmul_rn(w.w1, d1), __dmul_rn(w.w2, d2)), __dmul_rn(0., w.dab)),
                   __dmul_rn(w.w4, fabs(__dadd_rn(d1, -d2))));
}
__device__ __forceinline__ bool key_less(double d1, int i1, int j1, double d2, int i2, int j2) {
  if (d1 != d2) return d1 < d2 || (d2 != d2 && !(d1 != d1)); // NaN sorts last
  return i1 < i2 || (i1 == i2 && j1 < j2);
}

// All rounds in ONE persistent cooperative kernel; a round is three phases separated by grid barriers:
//   (A) first minimum of every stale row (queued by the previous round), rows split over several CTAs when few
//   (B) reciprocal pairs -> merge list with their Lance-Williams weights; per-CTA first global minimum for
//       rounds without a reciprocal pair (ties)
//   (C) new rows / columns of the merged slots, queue of the rows whose cached minimum went stale, bookkeeping
// Host-driven rounds (six launches and a read-back each) measured 32 ms per 20 000-site dendrogram, six
// barriers per round 28.5 ms (42 % of the warp stalls at barriers, the rest memory latency of one row per CTA).
constexpr int kSegMax = 8;
__global__ void __launch_bounds__(RT) k4r_rounds(RnnParams p) {
  cg::grid_group grid = cg::this_grid();
  __shared__ Best sh[32];
  __shared__ Cand shc[32];
  __shared__ int sh_last;
  const int64_t S = p.S;
  const int G = (int)gridDim.x;
  const int64_t gtid = (int64_t)blockIdx.x * RT + threadIdx.x, gsz = (int64_t)G * RT;
  constexpr int CW = RT * 4;
  const int64_t n_blk = (S + CW - 1) / CW;
  const double w4 = p.linkage == 0 ? .5 : p.linkage == 1 ? -.5 : 0.;
  volatile int32_t* cnt = p.counters;
  int64_t merged = 0;
  int round = 0;
  for (; merged < S - 1; round++) {
    const int par = round & 1;
    // ---- (A) first minimum of every stale row over the live columns k != r (NaN entries are skipped)
    {
      const int n = cnt[2 + par];
      const int32_t* wl = p.wl + (size_t)par * S;
      const int nseg = n > 0 && n * 2 <= G ? (G / n < kSegMax ? G / n : kSegMax) : 1;
      constexpr int U = 16;
      for (int it = blockIdx.x; it < n * nseg; it += G) {
        const int w = it / nseg, seg = it % nseg;
        const int r = wl[w];
        const int64_t lo = S * seg / nseg, hi = S * (seg + 1) / nseg;
        const double* row = p.mat + (size_t)r * S;
        Best b{0., -1};
        for (int64_t base = lo; base < hi; base += (int64_t)RT * U) {
          double v[U];
          uint8_t al[U];
#pragma unroll
          for (int u = 0; u < U; u++) {
            const int64_t k = base + (int64_t)u * RT + threadIdx.x;
            al[u] = k < hi ? p.alive[k] : 0;
            v[u] = k < hi ? row[k] : 0.;
          }
#pragma unroll
          for (int u = 0; u < U; u++) {
            const int64_t k = base + (int64_t)u * RT + threadIdx.x;
            if (al[u] && k != r && !(v[u] != v[u]) && better(v[u], (int)k, b)) { b.v = v[u]; b.i = (int)k; }
          }
        }
        b = block_best(b, sh);
        if (nseg == 1) {
          if (threadIdx.x == 0) { p.nn_val[r] = b.v; p.nn_idx[r] = b.i; p.dirty[r] = 0; }
        } else { // the CTA that finishes the row's last segment combines the partial minima
          if (threadIdx.x == 0) {
            p.seg_v[w * nseg + seg] = b.v; p.seg_i[w * nseg + seg] = b.i;
            __threadfence();
            sh_last = atomicAdd(&p.seg_cnt[w], 1) == nseg - 1;
          }
          __syncthreads();
          if (sh_last && threadIdx.x < 32) {
            __threadfence();
            Best c{0., -1};
            if ((int)threadIdx.x < nseg) { c.i = __ldcg(&p.seg_i[w * nseg + threadIdx.x]); c.v = __ldcg(&p.seg_v[w * nseg + threadIdx.x]); }
            c = warp_best(c);
            if (threadIdx.x == 0) { p.nn_val[r] = c.v; p.nn_idx[r] = c.i; p.dirty[r] = 0; p.seg_cnt[w] = 0; }
          }
        }
        __syncthreads();
      }
      if (gtid == 0) { cnt[par] = 0; cnt[4] = -1; cnt[5] = -1; cnt[6] = 0; } // this round's pair counter, the last-two slots
    }
    grid.sync();
    // ---- (B) reciprocal first minima (i, j), i < j, nn(i) = j and nn(j) = i; per-CTA first global minimum
    const bool last2 = (S - merged) == 2;
    {
      Cand c{0., -1, -1};
      for (int64_t i = gtid; i < S; i += gsz) {
        if (!p.alive[i]) continue;
        if (last2) { cnt[4 + (atomicAdd((int32_t*)&cnt[6], 1) & 1)] = (int32_t)i; continue; }
        const int j = p.nn_idx[i];
        if (j < 0) continue;
        const double v = p.nn_val[i];
        const Cand t{v, j < (int)i ? j : (int)i, j < (int)i ? (int)i : j};
        if (cand_less(t, c)) c = t;
        if (j <= (int)i || p.nn_idx[j] != (int)i) continue;
        const int q = atomicAdd((int32_t*)&cnt[par], 1);
        p.pair_i[q] = (int)i; p.pair_j[q] = j; p.pair_d[q] = v;
        double w1 = .5, w2 = .5;
        if (p.linkage == 2) {
          const double na = (double)p.nleaves[i], nb = (double)p.nleaves[j];
          w1 = na / (na + nb); w2 = nb / (na + nb);
        }
        p.pair_w1[q] = w1; p.pair_w2[q] = w2;
        const long long tag = (long long)round << 32;
        p.role[i] = tag | (long long)(2 * q); p.role[j] = tag | (long long)(2 * q + 1);
      }
      c = block_cand(c, shc);
      if (threadIdx.x == 0) { p.part_v[blockIdx.x] = c.v; p.part_lo[blockIdx.x] = c.lo; p.part_hi[blockIdx.x] = c.hi; }
      if (gtid == 0) cnt[2 + (par ^ 1)] = 0; // the queue the next round scans is filled in (C)
    }
    grid.sync();
    // ---- merges of this round: the reciprocal pairs, else the reference's next merge (first global minimum in
    //      (i, j) order), else -- two clusters left -- their join whatever the distance (finalStep upstream)
    int n_pairs = cnt[par];
    bool single = false;   // one merge that is not in the pair list / role table
    int s_i = -1, s_j = -1;
    double s_d = 0., s_w1 = .5, s_w2 = .5;
    if (n_pairs == 0) {
      if (last2) {
        const int a = cnt[4], b = cnt[5];
        s_i = a < b ? a : b; s_j = a < b ? b : a;
        s_d = p.mat[(size_t)s_i * S + s_j];
      } else {
        Cand c{0., -1, -1};
        for (int t = threadIdx.x; t < G; t += RT) {
          const Cand x{__ldcg(&p.part_v[t]), __ldcg(&p.part_lo[t]), __ldcg(&p.part_hi[t])};
          if (cand_less(x, c)) c = x;
        }
        c = block_cand(c, shc);
        s_i = c.lo; s_j = c.hi; s_d = c.v;
      }
      if (s_i < 0 || s_j < 0) { // nothing finite left to merge (NaN distances): the host reports it
        if (gtid == 0) cnt[9] = 1;
        return;
      }
      if (p.linkage == 2) {
        const double na = (double)p.nleaves[s_i], nb = (double)p.nleaves[s_j];
        s_w1 = na / (na + nb); s_w2 = nb / (na + nb);
      }
      single = true;
      n_pairs = 1;
    }
    // ---- (C) new row / column of every merged slot; work item = (pair, block of RT * 4 columns)
    int32_t* wl_next = p.wl + (size_t)(par ^ 1) * S;
    auto queue = [&](int k) { // row k's cached minimum is stale: scanned next round (once)
      if (atomicExch(&p.dirty[k], 1) == 0) wl_next[atomicAdd((int32_t*)&cnt[2 + (par ^ 1)], 1)] = k;
    };
    const long long tag = (long long)round << 32;
    for (int64_t it = blockIdx.x; it < (int64_t)n_pairs * n_blk; it += G) {
      // block-major: CTAs that run together work on the same block of rows k, so the scattered mirror writes
      // mat[k][i] of a round stay inside the same ~1000 rows (TLB reach) instead of touching every row per pair
      const int q = (int)(it % n_pairs);
      const int64_t k0 = (it / n_pairs) * CW;
      const int i = single ? s_i : p.pair_i[q], j = single ? s_j : p.pair_j[q];
      LW wq;
      wq.dab = single ? s_d : p.pair_d[q]; wq.w1 = single ? s_w1 : p.pair_w1[q]; wq.w2 = single ? s_w2 : p.pair_w2[q]; wq.w4 = w4;
      const double* ri = p.mat + (size_t)i * S;
      const double* rj = p.mat + (size_t)j * S;
#pragma unroll
      for (int u = 0; u < 4; u++) {
        const int64_t k = k0 + (int64_t)u * RT + threadIdx.x;
        if (k >= S || k == i || k == j || !p.alive[k]) continue;
        const long long rk = single ? -1 : p.role[k];
        double nd;
        if ((rk & ~0xffffffffLL) != tag) { // row k is not merged this round
          nd = lance_williams(wq, ri[k], rj[k]);
          // its cached nearest neighbour is stale when it pointed at a merged slot, or when the new entry
          // undercuts it (possible by an ulp under average linkage)
          const int ci = p.nn_idx[k];
          if (ci == i || ci == j) queue((int)k);
          else if (!(nd != nd)) {
            const double cv = p.nn_val[k];
            if (ci < 0 || nd < cv || (nd == cv && i < ci)) queue((int)k);
          }
        } else {
          const int r2 = (int)(rk & 0xffffffffLL);
          if (r2 & 1) continue;               // k dies this round
          const int q2 = r2 >> 1;             // k keeps its slot in pair q2: one of the two pairs writes the entry
          if (q2 < q) continue;
          const int i2 = (int)k, j2 = p.pair_j[q2];
          LW w2;
          w2.dab = p.pair_d[q2]; w2.w1 = p.pair_w1[q2]; w2.w2 = p.pair_w2[q2]; w2.w4 = w4;
          const double a = ri[i2], b = rj[i2], c = ri[j2], e = rj[j2];
          if (key_less(wq.dab, i, j, w2.dab, i2, j2))   // this pair first, as the reference would
            nd = lance_williams(w2, lance_williams(wq, a, b), lance_williams(wq, c, e));
          else
            nd = lance_williams(wq, lance_williams(w2, a, c), lance_williams(w2, b, e));
        }
        p.mat[(size_t)i * S + k] = nd;
        p.mat[(size_t)k * S + i] = nd;
      }
    }
    // ---- bookkeeping: merge records in creation order, slot state (nothing the loop above reads)
    for (int64_t q = gtid; q < n_pairs; q += gsz) {
      const int i = single ? s_i : p.pair_i[q], j = single ? s_j : p.pair_j[q];
      const double d = single ? s_d : p.pair_d[q];
      const int64_t m = merged + q;
      const double half = d / 2., len_i = p.len[i];
      const double h = len_i + (half - len_i);   // as k4_cluster.cu (TreeTemplate branch lengths upstream)
      p.m_left[m] = p.node[i]; p.m_right[m] = p.node[j];
      p.m_height[m] = h; p.m_d[m] = d; p.m_i[m] = i; p.m_j[m] = j;
      p.node[i] = (int32_t)(S + m);
      p.len[i] = h;
      p.nleaves[i] += p.nleaves[j];
      p.alive[j] = 0; p.nn_idx[j] = -1;
      queue(i);
    }
    merged += n_pairs;
    grid.sync();
  }
}

} // namespace

bool cluster_rnn_selected(int64_t S, int linkage) {
  const char* algo = getenv("CMB_K4_ALGO"); // "exact" | "rnn"; default: by size
  if (linkage == 1) return false;                  // single linkage creates new ties: exact replay only
  if (algo && std::string(algo) == "exact") return false;
  if (algo && std::string(algo) == "rnn") return S >= 3;
  return S >= 2048;
}

// Dendrogram of one matrix by reciprocal-pair rounds; left / right / height (device, [S-1]) in the reference's
// creation order.  Returns the number of kernel launches.
int launch_cluster_rnn(int64_t S, int linkage, double* mat, DevBuf& work, int32_t* left_dev, int32_t* right_dev,
                       double* height_dev, cudaStream_t st) {
  size_t o = 0;
  auto take = [&](size_t bytes) { size_t at = o; o = align256(o + bytes); return at; };
  const size_t o_alive = take(S), o_len = take(8 * S), o_nl = take(4 * S), o_node = take(4 * S), o_nv = take(8 * S),
               o_ni = take(4 * S), o_dirty = take(4 * S), o_role = take(8 * S), o_wl = take(8 * S), o_pi = take(4 * (S / 2 + 2)),
               o_pj = take(4 * (S / 2 + 2)), o_pd = take(8 * (S / 2 + 2)), o_w1 = take(8 * (S / 2 + 2)), o_w2 = take(8 * (S / 2 + 2)),
               o_pv = take(8 * 1024), o_plo = take(4 * 1024), o_phi = take(4 * 1024), o_sv = take(8 * 1024), o_si = take(4 * 1024),
               o_sc = take(4 * 1024), o_cnt = take(64), o_ml = take(4 * S), o_mr = take(4 * S), o_mi = take(4 * S), o_mj = take(4 * S),
               o_mh = take(8 * S), o_md = take(8 * S);
  work.reserve(o);
  unsigned char* w = work.as<unsigned char>();
  RnnParams p;
  p.S = S; p.linkage = linkage; p.mat = mat;
  p.alive = w + o_alive; p.len = (double*)(w + o_len); p.nleaves = (int32_t*)(w + o_nl); p.node = (int32_t*)(w + o_node);
  p.nn_val = (double*)(w + o_nv); p.nn_idx = (int32_t*)(w + o_ni); p.dirty = (int32_t*)(w + o_dirty); p.role = (long long*)(w + o_role);
  p.wl = (int32_t*)(w + o_wl); p.pair_i = (int32_t*)(w + o_pi); p.pair_j = (int32_t*)(w + o_pj); p.pair_d = (double*)(w + o_pd);
  p.pair_w1 = (double*)(w + o_w1); p.pair_w2 = (double*)(w + o_w2);
  p.part_v = (double*)(w + o_pv); p.part_lo = (int32_t*)(w + o_plo); p.part_hi = (int32_t*)(w + o_phi);
  p.seg_v = (double*)(w + o_sv); p.seg_i = (int32_t*)(w + o_si); p.seg_cnt = (int32_t*)(w + o_sc);
  p.counters = (int32_t*)(w + o_cnt);
  p.m_left = (int32_t*)(w + o_ml); p.m_right = (int32_t*)(w + o_mr); p.m_i = (int32_t*)(w + o_mi); p.m_j = (int32_t*)(w + o_mj);
  p.m_height = (double*)(w + o_mh); p.m_d = (double*)(w + o_md);

  int dev = 0, sms = 0, per_sm = 0;
  CMB_CUDA(cudaGetDevice(&dev));
  CMB_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  CMB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k4r_rounds, RT, 0));
  if (per_sm < 1) fail("k4r_rounds cannot be made resident");
  const int grid = std::min(sms * std::min(per_sm, 4), 1024);
  const unsigned gS = (unsigned)((S + RT - 1) / RT);
  int launches = 2;
  k4r_init<<<gS, RT, 0, st>>>(p);
  CMB_CUDA(cudaGetLastError());
  void* args[] = {&p};
  CMB_CUDA(cudaLaunchCooperativeKernel((void*)k4r_rounds, dim3(grid), dim3(RT), args, 0, st));
  int32_t h_cnt[16];
  CMB_CUDA(cudaMemcpyAsync(h_cnt, p.counters, sizeof h_cnt, cudaMemcpyDeviceToHost, st));
  CMB_CUDA(cudaStreamSynchronize(st));
  if (h_cnt[9]) { // nothing mergeable: NaN distances; the caller reports it (left = -1)
    CMB_CUDA(cudaMemsetAsync(left_dev, 0xff, 4 * (S - 1), st));
    return launches;
  }
  // ---- the reference's creation order: children before parents, smallest (distance, i, j) first
  const int64_t M = S - 1;
  std::vector<int32_t> ml(M), mr(M), mi(M), mj(M);
  std::vector<double> mh(M), md(M);
  CMB_CUDA(cudaMemcpyAsync(ml.data(), p.m_left, 4 * M, cudaMemcpyDeviceToHost, st));
  CMB_CUDA(cudaMemcpyAsync(mr.data(), p.m_right, 4 * M, cudaMemcpyDeviceToHost, st));
  CMB_CUDA(cudaMemcpyAsync(mi.data(), p.m_i, 4 * M, cudaMemcpyDeviceToHost, st));
  CMB_CUDA(cudaMemcpyAsync(mj.data(), p.m_j, 4 * M, cudaMemcpyDeviceToHost, st));
  CMB_CUDA(cudaMemcpyAsync(mh.data(), p.m_height, 8 * M, cudaMemcpyDeviceToHost, st));
  CMB_CUDA(cudaMemcpyAsync(md.data(), p.m_d, 8 * M, cudaMemcpyDeviceToHost, st));
  CMB_CUDA(cudaStreamSynchronize(st));
  // key of a merge = (distance, i, j), raised to its children's keys where a Lance-Williams rounding made a
  // parent an ulp closer than its child: the reference merges such a parent right after the child
  struct Key { double d; int32_t i, j, m; };
  auto less = [](const Key& a, const Key& b) {
    if (a.d != b.d) return a.d < b.d;
    if (a.i != b.i) return a.i < b.i;
    if (a.j != b.j) return a.j < b.j;
    return a.m < b.m;
  };
  std::vector<Key> keys(M);
  for (int64_t m = 0; m < M; m++) { // children were created in earlier rounds: smaller m
    Key k{md[m] != md[m] ? INFINITY : md[m], mi[m], mj[m], (int32_t)m};
    for (int32_t ch : {ml[m], mr[m]})
      if (ch >= S) {
        const Key& c = keys[ch - S];
        if (less(k, c)) { k.d = c.d; k.i = c.i; k.j = c.j; }
      }
    keys[m] = k;
  }
  std::vector<Key> sorted_keys(keys);
  std::sort(sorted_keys.begin(), sorted_keys.end(), less);
  std::vector<int32_t> final_id(M, -1), order(M);
  for (int64_t r = 0; r < M; r++) { order[r] = sorted_keys[r].m; final_id[sorted_keys[r].m] = (int32_t)(S + r); }
  for (int64_t m = 0; m < M; m++)
    for (int32_t ch : {ml[m], mr[m]})
      if (ch >= S && final_id[ch - S] >= final_id[m]) fail("internal: clustering rounds produced a parent before its child");
  std::vector<int32_t> fl(M), fr(M);
  std::vector<double> fh(M);
  for (int64_t r = 0; r < M; r++) {
    const int32_t m = order[r];
    fl[r] = ml[m] >= S ? final_id[ml[m] - S] : ml[m];
    fr[r] = mr[m] >= S ? final_id[mr[m] - S] : mr[m];
    fh[r] = mh[m];
  }
  CMB_CUDA(cudaMemcpyAsync(left_dev, fl.data(), 4 * M, cudaMemcpyHostToDevice, st));
  CMB_CUDA(cudaMemcpyAsync(right_dev, fr.data(), 4 * M, cudaMemcpyHostToDevice, st));
  CMB_CUDA(cudaMemcpyAsync(height_dev, fh.data(), 8 * M, cudaMemcpyHostToDevice, st));
  CMB_CUDA(cudaStreamSynchronize(st)); // the host vectors go out of scope
  return launches;
}

} // namespace cmb
