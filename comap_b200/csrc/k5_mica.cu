// K5: Mica's statistics (CoMap/Mica.cpp) -- mutual information, joint entropy and entropy of alignment COLUMNS
// (no substitution mapping: the mapping only supplies the norms that condition the null, Mica.cpp:336-339).
//
// Replaces SiteTools::mutualInformation / jointEntropy / entropy(site, resolveUnknowns = true) at Mica.cpp:92, 354,
// 357, 430-431, 524-525, 574-575, 660 [Bio++ bpp-seq, from memory; the reference ships no output of mica: parity
// unpinned].  A character compatible with k states adds 1/k to each of them (a pair 1/(k1 k2) to each combination),
// frequencies = counts / number of sequences, the joint table is renormalised by its total and the marginals are
// taken from it; sums run rows then columns, as restated in the oracle (orc_site_pair).
//
// Layout: the alignment is the tip matrix K1 reads, [T][S_pad] codes with the 256-entry code -> state-mask table.
// k5_pairs / k5_listed / k5_entropy: one thread per pair (site); T byte loads per column (coalesced over the 32 pairs of
// a warp, which share site i and walk consecutive sites j), then the table's A^2 cells.  For A <= 4, T <= 65535 and no
// ambiguous character the joint table sits in packed registers, otherwise in local memory (pair_stats below).  Not a tiled
// kernel: the work per pair is a histogram, not a dot product.
// k5_permutations (null.method = permutations, up to 1000 evaluations per pair): one warp per pair, see there.
#include "kernels.h"
#include <algorithm>
#include <cstdlib>
#include "device_utils.cuh"

namespace cmb {
namespace {

// a column of codes, strided in global memory (the tip matrix)
struct Col {
  const uint8_t* p;
  size_t stride;
  __device__ __forceinline__ uint32_t operator[](int t) const { return p[(size_t)t * stride]; }
};
// a lane's private column in shared memory (the permutation test): four characters per 32-bit word, words of one lane
// `stride4` bytes apart, so a lane always stays in its own bank whatever character it touches
struct LaneCol {
  uint8_t* p;
  int stride4;
  __device__ __forceinline__ uint32_t operator[](int t) const { return p[(t >> 2) * stride4 + (t & 3)]; }
  __device__ __forceinline__ uint8_t& at(int t) const { return p[(t >> 2) * stride4 + (t & 3)]; }
};

// MI and joint entropy from the joint table (orc_site_pair's order: rows, then columns).  freq(x, y) returns count / n.
// Loops stay rolled: one copy of the two logarithms and three divisions per kernel, not A^2 of them (unrolled over its
// 16 cells the permutation kernel's loop body was 70 KB of SASS and ncu put 27 % of its stalls on instruction fetches).
// p1 / p2 are register arrays for A <= 4, read and written through compile-time-indexed selects.
template <int A>
__device__ __forceinline__ double pick(const double (&v)[A], int k) {
  if constexpr (A <= 4) {
    double r = v[0];
#pragma unroll
    for (int i = 1; i < A; i++) r = k == i ? v[i] : r;
    return r;
  } else return v[k];
}
template <int A>
__device__ __forceinline__ void put(double (&v)[A], int k, double val) {
  if constexpr (A <= 4) {
#pragma unroll
    for (int i = 0; i < A; i++) v[i] = k == i ? val : v[i];
  } else v[k] = val;
}
template <int A, class Freq>
__device__ __forceinline__ void table_stats(Freq freq, double& mi, double& hj) {
  double p1[A], p2[A];
#pragma unroll
  for (int x = 0; x < A; x++) { p1[x] = 0.; p2[x] = 0.; }
  double tot = 0.;
#pragma unroll 1
  for (int x = 0; x < A; x++)
#pragma unroll 1
    for (int y = 0; y < A; y++) {
      const double pxy = freq(x, y);
      tot += pxy;
      put<A>(p1, x, pick<A>(p1, x) + pxy);
      put<A>(p2, y, pick<A>(p2, y) + pxy);
    }
#pragma unroll
  for (int x = 0; x < (A <= 4 ? A : 0); x++) { p1[x] /= tot; p2[x] /= tot; }
  if constexpr (A > 4) {
#pragma unroll 1
    for (int x = 0; x < A; x++) { p1[x] /= tot; p2[x] /= tot; }
  }
  double m = 0., h = 0.;
#pragma unroll 1
  for (int x = 0; x < A; x++)
#pragma unroll 1
    for (int y = 0; y < A; y++) {
      const double pxy = freq(x, y) / tot;
      if (pxy > 0.) { m += pxy * log(pxy / (pick<A>(p1, x) * pick<A>(p2, y))); h += pxy * log(pxy); }
    }
  mi = m; hj = -h;
}

// The joint table in local memory, filled in sequence order exactly as the oracle does: any alphabet, any character.
template <int A, class C1, class C2>
__device__ __noinline__ void pair_stats_generic(const C1 c1, const C2 c2, int T, const uint32_t* __restrict__ cmask, double& mi,
                                                double& hj) {
  constexpr uint32_t full = A >= 32 ? 0xffffffffu : (1u << A) - 1u;
  double cnt[A * A];
#pragma unroll 1
  for (int k = 0; k < A * A; k++) cnt[k] = 0.;
  for (int t = 0; t < T; t++) {
    const uint32_t m1 = cmask[c1[t]] & full, m2 = cmask[c2[t]] & full;
    const int k1 = __popc(m1), k2 = __popc(m2);
    if (k1 == 1 && k2 == 1) cnt[(__ffs(m1) - 1) * A + __ffs(m2) - 1] += 1.;
    else if (k1 && k2) {
      const double w = 1. / ((double)k1 * (double)k2);
      for (int x = 0; x < A; x++)
        if ((m1 >> x) & 1u)
          for (int y = 0; y < A; y++)
            if ((m2 >> y) & 1u) cnt[x * A + y] += w;
    }
  }
  const double n = (double)T;
  table_stats<A>([&](int x, int y) { return cnt[x * A + y] / n; }, mi, hj);
}

// A <= 4 and no ambiguous character in either column (almost every pair of a real alignment, every pair of a simulated
// one): the joint table never leaves the registers.  Counts sit in packed 16-bit fields, one 64-bit word per state of the
// first column, so no register is indexed by data; integers convert exactly, so the result is bit for bit the generic
// path's.  A pair that does hold an ambiguous character takes the generic path, and so does every pair of an alignment of
// more than 65535 sequences: a cell counts up to T sequences, and a 65536th would carry into the next state's field.
template <int A, class C1, class C2>
__device__ __forceinline__ void pair_stats(const C1 c1, const C2 c2, int T, const uint32_t* __restrict__ cmask, double& mi, double& hj) {
  if constexpr (A <= 4) {
    if (T <= 65535) {
      constexpr uint32_t full = (1u << A) - 1u;
      unsigned long long w[A];
#pragma unroll
      for (int x = 0; x < A; x++) w[x] = 0ull;
      bool ambiguous = false;
      for (int t = 0; t < T; t++) {
        const uint32_t m1 = cmask[c1[t]] & full, m2 = cmask[c2[t]] & full;
        const int k1 = __popc(m1), k2 = __popc(m2);
        if (k1 == 1 && k2 == 1) {
          const unsigned long long inc = 1ull << (16 * (__ffs(m2) - 1));
#pragma unroll
          for (int x = 0; x < A; x++) w[x] += (m1 >> x) & 1u ? inc : 0ull;
        } else if (k1 && k2) ambiguous = true;
      }
      if (!ambiguous) {
        const double n = (double)T;
        table_stats<A>([&](int x, int y) {
          unsigned long long r = w[0];
#pragma unroll
          for (int i = 1; i < A; i++) r = x == i ? w[i] : r;
          return (double)(unsigned)((r >> (16 * y)) & 0xffffull) / n;
        }, mi, hj);
        return;
      }
    }
  }
  pair_stats_generic<A, C1, C2>(c1, c2, T, cmask, mi, hj);
}

// The permutation test's evaluation when neither column holds an ambiguous character: the private copies carry state
// indices, so the histogram needs no mask table, and count / n comes from a table of the T + 1 possible quotients
// (the same correctly rounded divisions, done once per CTA).  Same table_stats, same bits as pair_stats on the same table.
template <int A>
__device__ __forceinline__ void packed_histogram(const LaneCol s1, const LaneCol s2, int T, unsigned long long (&w)[A]) {
#pragma unroll
  for (int x = 0; x < A; x++) w[x] = 0ull;
  for (int t = 0; t < T; t++) {
    const uint32_t a = s1[t];
    const unsigned long long inc = 1ull << (16 * s2[t]);
#pragma unroll
    for (int x = 0; x < A; x++)
      if (a == (uint32_t)x) w[x] += inc;
  }
}
template <int A>
__device__ __forceinline__ unsigned packed_cell(const unsigned long long (&w)[A], int x, int y) {
  unsigned long long r = w[0];
#pragma unroll
  for (int i = 1; i < A; i++) r = x == i ? w[i] : r;
  return (unsigned)((r >> (16 * y)) & 0xffffull);
}
// one copy per kernel (not inlined): the observed table and every shuffled one go through the very same instructions
template <int A>
struct Packed { unsigned long long w[A]; };      // by value: the caller's words stay in registers
template <int A>
__device__ __noinline__ double2 packed_stats_call(const Packed<A> p, const double* __restrict__ quot) {
  double2 r;
  table_stats<A>([&](int x, int y) { return quot[packed_cell<A>(p.w, x, y)]; }, r.x, r.y);
  return r;
}
template <int A>
__device__ __forceinline__ void packed_stats(const unsigned long long (&w)[A], const double* __restrict__ quot, double& mi, double& hj) {
  Packed<A> p;
#pragma unroll
  for (int x = 0; x < A; x++) p.w[x] = w[x];
  const double2 r = packed_stats_call<A>(p, quot);
  mi = r.x; hj = r.y;
}
// sum of (c / T) ln(c / T) over the cells, from a table: MI differs from it by a term the shuffles cannot change (the
// marginal entropies), so it orders shuffled and observed tables as MI does in real arithmetic
template <int A>
__device__ __forceinline__ double packed_filter(const unsigned long long (&w)[A], const double* __restrict__ plogp) {
  double f = 0.;
#pragma unroll 1
  for (int x = 0; x < A; x++)
#pragma unroll
    for (int y = 0; y < A; y++) f += plogp[packed_cell<A>(w, x, y)];
  return f;
}
template <int A>
__device__ __forceinline__ void indexed_stats(const LaneCol s1, const LaneCol s2, int T, const double* __restrict__ quot, double& mi,
                                              double& hj) {
  if constexpr (A <= 4) {
    unsigned long long w[A];
    packed_histogram<A>(s1, s2, T, w);
    packed_stats<A>(w, quot, mi, hj);
  } else {
    uint16_t cnt[A * A];
#pragma unroll 1
    for (int k = 0; k < A * A; k++) cnt[k] = 0;
    for (int t = 0; t < T; t++) cnt[s1[t] * A + s2[t]]++;
    table_stats<A>([&](int x, int y) { return quot[cnt[x * A + y]]; }, mi, hj);
  }
}

template <int A>
__global__ void __launch_bounds__(128) k5_entropy(int T, int64_t n, int64_t n_pad, const uint8_t* __restrict__ tips,
                                                  const uint32_t* __restrict__ cmask, double* __restrict__ entropy) {
  const int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= n) return;
  constexpr uint32_t full = A >= 32 ? 0xffffffffu : (1u << A) - 1u;
  double cnt[A];
#pragma unroll
  for (int x = 0; x < A; x++) cnt[x] = 0.;
  for (int t = 0; t < T; t++) {
    const uint32_t m = __ldg(cmask + tips[(size_t)t * n_pad + s]) & full;
    const int k = __popc(m);
    if (!k) continue;
    const double w = 1. / (double)k;
    for (int x = 0; x < A; x++)
      if ((m >> x) & 1u) cnt[x] += w;
  }
  double h = 0.;
  for (int x = 0; x < A; x++) {
    const double f = cnt[x] / (double)T;
    if (f != 0.) h += f * log(f);
  }
  entropy[s] = -h;
}

// all pairs i < j of one alignment, dense upper triangle in the reference's order (i ascending, j ascending)
template <int A>
__global__ void __launch_bounds__(128) k5_pairs(int T, int64_t S, int64_t n_pad, const uint8_t* __restrict__ tips,
                                                const uint32_t* __restrict__ cmask, double* __restrict__ mi,
                                                double* __restrict__ hj) {
  const int64_t i = blockIdx.y;
  const int64_t j = i + 1 + (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= S) return;
  double m, h;
  pair_stats<A>(Col{tips + i, (size_t)n_pad}, Col{tips + j, (size_t)n_pad}, T, cmask, m, h);
  const int64_t idx = i * S - i * (i + 1) / 2 + (j - i - 1);
  mi[idx] = m;
  if (hj) hj[idx] = h;
}

// site a[r] against site b[r] (possibly of another tip matrix): the null's j <-> j pairs and the bootstrap's pair lists
template <int A>
__global__ void __launch_bounds__(128) k5_listed(int T, int64_t n, const uint8_t* __restrict__ t1, int64_t np1,
                                                 const uint8_t* __restrict__ t2, int64_t np2, const int32_t* __restrict__ a,
                                                 const int32_t* __restrict__ b, const uint32_t* __restrict__ cmask,
                                                 double* __restrict__ mi, double* __restrict__ hj) {
  const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= n) return;
  const int64_t s1 = a ? a[r] : r, s2 = b ? b[r] : r;
  double m, h;
  pair_stats<A>(Col{t1 + s1, (size_t)np1}, Col{t2 + s2, (size_t)np2}, T, cmask, m, h);
  mi[r] = m;
  if (hj) hj[r] = h;
}

// null.method = permutations (miTest, Mica.cpp:92-118): per pair, both columns are shuffled until 5 shuffled MIs reach the
// observed one or max_perm shuffles were drawn; p = (count + 1) / (shuffles + 1); a pair with a constant column (unknown
// characters ignored) gets p = 1 after 0 shuffles.
//
// Upstream shuffles its two copies in place, again and again, with an unseeded generator.  A uniformly random
// permutation applied to any arrangement gives a uniformly random arrangement independent of the one it started from,
// so shuffle q is drawn here from the ORIGINAL columns: same distribution of (count, shuffles), and the shuffles of
// a pair no longer form a chain.  That is the whole design: pairs stop after anything between 5 and max_perm
// shuffles, and with one pair per lane (the first version, 85 ms on the BacteriaSSU shape; 41 ms with a work queue)
// the few lanes holding a 1000-shuffle pair outlive everything else -- ncu counted 7.9 active threads per warp.
// One WARP per pair instead: lane l of trip k scores shuffle 32 k + l - 1 (lane 0 of the first trip scores the
// observed columns), a ballot of `rep >= mi` and a population count find the shuffle at which upstream's loop would
// have stopped, and at most 31 evaluations per pair are wasted.  Every branch but the ambiguous-character path is
// warp-uniform: 16.4 ms; 10.4 with rolled table loops, state indices in the private copies, a quotient table and two
// draws per generator word; 6.8 with the interval filter in front of the reference's formula (profiles/r2w_k5_history.txt).
// Shuffle q of pair idx, column c: inside-out Fisher-Yates (s[0] = c[0]; for k = 1 .. T-1: j = floor(w (k + 1) / 2^32),
// s[k] = s[j], s[j] = c[k]), the words w taken in order from Philox4x32-10 blocks with counter (idx lo, idx hi, q,
// c << 24 | block) and key = seed.  When T <= 256 a word serves two draws: after the first, w <- w (k + 1) mod 2^32 (the
// fraction the first draw left over) feeds the next k -- half the generator calls for a bias below 2^-16.  Restated
// word for word in the oracle (orc_mica_permutation_test).
// The observed and the shuffled MIs come from the same call site, so equal joint tables give equal bits and
// `rep >= mi` sees the exact ties a discrete statistic produces.
//
// A shard (shard_index, shard_count) owns the pairs idx = shard_index + k shard_count, k = 0 .. n_rows - 1: the counter
// hands out k, the outputs are written at k.  Shuffle q of pair idx depends on (seed, idx, q) only, so a shard's rows
// are bit for bit the same rows of the whole table (shard_count = 1).
// Register budget: MIN_CTAS = 5 CTAs of 128 per SM, 95 registers, nothing spilled (6 and 8 measured: DESIGN.md s4, K5).
// The budget stays in the template arguments so that the kernel keeps its name, k5_permutations<A, 5>.
template <int A, int MIN_CTAS>
__global__ void __launch_bounds__(128, MIN_CTAS) k5_permutations(int T, int64_t S, int64_t n_rows, int shard_index,
                                                       int shard_count, int64_t n_pad,
                                                       const uint8_t* __restrict__ tips, const uint32_t* __restrict__ cmask,
                                                       uint64_t seed, int max_perm, int use_filter,
                                                       unsigned long long* __restrict__ next, double* __restrict__ pvalue,
                                                       int32_t* __restrict__ nperm) {
  extern __shared__ __align__(16) unsigned char k5_smem[];
  const int nt = blockDim.x, lane = threadIdx.x & 31, warp = threadIdx.x >> 5, T4 = (T + 3) >> 2;
  uint32_t* s_mask = reinterpret_cast<uint32_t*>(k5_smem);                     // [256]
  double* quot = reinterpret_cast<double*>(k5_smem + 1024);                    // [T + 1]: c / T
  double* plogp = quot + (T + 1);                                              // [T + 1]: (c / T) ln(c / T)
  const size_t q_bytes = ((size_t)(T + 1) * 16 + 15) & ~(size_t)15;
  uint8_t* o1 = k5_smem + 1024 + q_bytes + (size_t)warp * 8 * T4;              // the warp's pair: [2][4 T4]
  uint8_t* o2 = o1 + 4 * T4;
  uint8_t* priv = k5_smem + 1024 + q_bytes + (size_t)(nt >> 5) * 8 * T4;       // [2][T4][nt] words
  const LaneCol s1{priv + 4 * threadIdx.x, 4 * nt}, s2{priv + (size_t)4 * T4 * nt + 4 * threadIdx.x, 4 * nt};
  for (int k = threadIdx.x; k < 256; k += nt) s_mask[k] = cmask[k];
  for (int k = threadIdx.x; k <= T; k += nt) {
    const double f = (double)k / (double)T;
    quot[k] = f;
    plogp[k] = k ? f * log(f) : 0.;
  }
  __syncthreads();
  constexpr uint32_t full = A >= 32 ? 0xffffffffu : (1u << A) - 1u;
  constexpr unsigned ALL = 0xffffffffu;
  const uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32);
  const bool two_per_word = T <= 256;            // ranges <= 256: the second draw of a word is biased by < 2^-16
  for (;;) {
    __syncwarp();
    unsigned long long got = 0;
    if (lane == 0) got = atomicAdd(next, 1ull);
    const int64_t row = (int64_t)__shfl_sync(ALL, got, 0);
    if (row >= n_rows) break;
    const int64_t idx = shard_index + row * (int64_t)shard_count;
    // idx = i S - i (i + 1) / 2 + (j - i - 1): row i from the root of the quadratic, then one step either way
    const double b = 2. * (double)S - 1.;
    int64_t i = (int64_t)((b - sqrt(b * b - 8. * (double)idx)) * 0.5);
    if (i < 0) i = 0;
    if (i > S - 2) i = S - 2;
    while (i > 0 && i * S - i * (i + 1) / 2 > idx) i--;
    while (i < S - 2 && (i + 1) * S - (i + 1) * (i + 2) / 2 <= idx) i++;
    const int64_t j = i + 1 + (idx - (i * S - i * (i + 1) / 2));
    // SiteTools::isConstant(site, ignoreUnknown = true): the characters that are not fully unknown are all the same.
    // Resolved characters are kept as state indices; one ambiguous character sends the pair down the generic path.
    uint32_t lo1 = 0xffffffffu, hi1 = 0u, lo2 = 0xffffffffu, hi2 = 0u;
    bool amb = false;
    for (int t = lane; t < T; t += 32) {
      const uint32_t a = tips[(size_t)t * n_pad + i], c = tips[(size_t)t * n_pad + j];
      const uint32_t ma = s_mask[a] & full, mc = s_mask[c] & full;
      if (ma != full) { lo1 = min(lo1, a); hi1 = max(hi1, a); }
      if (mc != full) { lo2 = min(lo2, c); hi2 = max(hi2, c); }
      amb |= __popc(ma) != 1 || __popc(mc) != 1;
    }
    lo1 = __reduce_min_sync(ALL, lo1); hi1 = __reduce_max_sync(ALL, hi1);
    lo2 = __reduce_min_sync(ALL, lo2); hi2 = __reduce_max_sync(ALL, hi2);
    amb = __any_sync(ALL, amb);
    if (lo1 >= hi1 || lo2 >= hi2) {              // one character at most (none: lo = 2^32 - 1 > hi = 0)
      if (lane == 0) { pvalue[row] = 1.; nperm[row] = 0; }
      continue;
    }
    for (int t = lane; t < T; t += 32) {
      const uint32_t a = tips[(size_t)t * n_pad + i], c = tips[(size_t)t * n_pad + j];
      o1[t] = (uint8_t)(amb ? a : __ffs(s_mask[a] & full) - 1);
      o2[t] = (uint8_t)(amb ? c : __ffs(s_mask[c] & full) - 1);
    }
    __syncwarp();
    int count = 0, shuffles = max_perm;
    double mi = 0., f_obs = 0.;
    unsigned long long w_obs[A <= 4 ? A : 1] = {};
    bool have_mi = false;
    for (int base = -1; base < max_perm; base += 32) {
      const int q = base + lane;
      if (q < 0) {
        for (int t = 0; t < T; t++) { s1.at(t) = o1[t]; s2.at(t) = o2[t]; }
      } else {
#pragma unroll 1
        for (int column = 0; column < 2; column++) {
          const LaneCol& col = column ? s2 : s1;
          const uint8_t* src = column ? o2 : o1;
          col.at(0) = src[0];
          int k = 1;
          for (uint32_t blk = 0; k < T; blk++) {
            uint32_t c[4] = {(uint32_t)idx, (uint32_t)((uint64_t)idx >> 32), (uint32_t)q, ((uint32_t)column << 24) | blk};
            philox4x32_10(c, k0, k1);
#pragma unroll
            for (int u = 0; u < 4; u++) {
              uint32_t w = c[u];
              if (k < T) {
                const unsigned long long pr = (unsigned long long)w * (uint32_t)(k + 1);
                const int p = (int)(pr >> 32);
                col.at(k) = col.at(p);
                col.at(p) = src[k];
                w = (uint32_t)pr;                 // the fraction left over: uniform enough for one more small range
                k++;
              }
              if (two_per_word && k < T) {
                const int p = (int)__umulhi(w, (uint32_t)(k + 1));
                col.at(k) = col.at(p);
                col.at(p) = src[k];
                k++;
              }
            }
          }
        }
      }
      const bool valid = q >= 0 && q < max_perm;
      bool hit;
      bool filtered = false;
      if constexpr (A <= 4) {
        if (!amb && use_filter) {
          // The comparison `rep >= mi` is all a shuffle contributes, and in real arithmetic it is the comparison of the
          // two tables' sums of p ln p (the marginals do not move).  Those sums come from a table, error < 1e-14; only
          // when a shuffled sum lies within 1e-12 of the observed one -- a tie, which the reference's formula settles by
          // its own rounding -- does the warp evaluate that formula, for the observed table (once) and the shuffled ones.
          filtered = true;
          unsigned long long w[A];
          packed_histogram<A>(s1, s2, T, w);
          const double f = packed_filter<A>(w, plogp);
          if (base < 0) {
            f_obs = __shfl_sync(ALL, f, 0);
#pragma unroll
            for (int x = 0; x < A; x++) w_obs[x] = __shfl_sync(ALL, w[x], 0);
            have_mi = false;
          }
          const double d = f - f_obs;
          if (__any_sync(ALL, valid && fabs(d) <= 1e-12)) {
            double m, h;
            if (!have_mi) { packed_stats<A>(w_obs, quot, mi, h); have_mi = true; }
            packed_stats<A>(w, quot, m, h);
            hit = valid && m >= mi;
          } else hit = valid && d > 0.;
        }
      }
      if (!filtered) {
        double m, h;
        if (amb) pair_stats_generic<A>(s1, s2, T, s_mask, m, h);
        else indexed_stats<A>(s1, s2, T, quot, m, h);
        if (base < 0) mi = __shfl_sync(ALL, m, 0);
        hit = valid && m >= mi;
      }
      const unsigned hits = __ballot_sync(ALL, hit);
      const int c = __popc(hits);
      if (count + c >= 5) {                      // the shuffle that brought the count to 5
        unsigned r = hits;
        for (int k = count; k < 4; k++) r &= r - 1;
        shuffles = base + (__ffs(r) - 1) + 1;
        count = 5;
        break;
      }
      count += c;
    }
    if (lane == 0) { pvalue[row] = (double)(count + 1) / (double)(shuffles + 1); nperm[row] = shuffles; }
  }
}

// Mica.cpp:341-361: average MI of every site with all the others, j ascending
__global__ void k5_average(int64_t S, const double* __restrict__ mi, double* __restrict__ avg) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= S) return;
  double sum = 0.;
  for (int64_t j = 0; j < S; j++) {
    if (j == i) continue;
    const int64_t lo = j < i ? j : i, hi = j < i ? i : j;
    sum += mi[lo * S - lo * (lo + 1) / 2 + (hi - lo - 1)];
  }
  avg[i] = sum / (double)(S - 1);
}

// the other columns of a row of mica's table: i, j, Hmin = min entropy, Nmin = min norm (NaN without a mapping)
__global__ void k5_rows(int64_t S, const double* __restrict__ entropy, const double* __restrict__ norm, int32_t* __restrict__ oi,
                        int32_t* __restrict__ oj, double* __restrict__ hmin, double* __restrict__ nmin) {
  const int64_t i = blockIdx.y;
  const int64_t j = i + 1 + (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= S) return;
  const int64_t idx = i * S - i * (i + 1) / 2 + (j - i - 1);
  oi[idx] = (int32_t)i; oj[idx] = (int32_t)j;
  const double a = entropy[i], b = entropy[j];
  hmin[idx] = a < b ? a : b;                       // std::min(entropy[i], entropy[j])
  if (nmin) {
    if (norm) { const double x = norm[i], y = norm[j]; nmin[idx] = x < y ? x : y; }
    else nmin[idx] = nan("");
  }
}

__global__ void k5_min2(int64_t n, const double* __restrict__ a, const double* __restrict__ b, double* __restrict__ out) {
  const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (r < n) out[r] = a[r] < b[r] ? a[r] : b[r];
}

} // namespace

void launch_mica_entropy(int A, int T, int64_t n, int64_t n_pad, const uint8_t* tips, const uint32_t* cmask, double* entropy,
                         cudaStream_t st) {
  const unsigned g = (unsigned)((n + 127) / 128);
  if (A == 4) k5_entropy<4><<<g, 128, 0, st>>>(T, n, n_pad, tips, cmask, entropy);
  else if (A == 20) k5_entropy<20><<<g, 128, 0, st>>>(T, n, n_pad, tips, cmask, entropy);
  else fail("mica kernels are built for A = 4 and A = 20 (got %d)", A);
  CMB_CUDA(cudaGetLastError());
}
void launch_mica_pairs(int A, int T, int64_t S, int64_t n_pad, const uint8_t* tips, const uint32_t* cmask, double* mi, double* hj,
                       cudaStream_t st) {
  if (S < 2) return;
  if (S > 65535) fail("mica: %lld sites exceed the 65535 rows one launch scores", (long long)S);
  dim3 grid((unsigned)((S - 1 + 127) / 128), (unsigned)(S - 1));
  if (A == 4) k5_pairs<4><<<grid, 128, 0, st>>>(T, S, n_pad, tips, cmask, mi, hj);
  else if (A == 20) k5_pairs<20><<<grid, 128, 0, st>>>(T, S, n_pad, tips, cmask, mi, hj);
  else fail("mica kernels are built for A = 4 and A = 20 (got %d)", A);
  CMB_CUDA(cudaGetLastError());
}
void launch_mica_listed(int A, int T, int64_t n, const uint8_t* t1, int64_t np1, const uint8_t* t2, int64_t np2, const int32_t* a,
                        const int32_t* b, const uint32_t* cmask, double* mi, double* hj, cudaStream_t st) {
  if (n == 0) return;
  const unsigned g = (unsigned)((n + 127) / 128);
  if (A == 4) k5_listed<4><<<g, 128, 0, st>>>(T, n, t1, np1, t2, np2, a, b, cmask, mi, hj);
  else if (A == 20) k5_listed<20><<<g, 128, 0, st>>>(T, n, t1, np1, t2, np2, a, b, cmask, mi, hj);
  else fail("mica kernels are built for A = 4 and A = 20 (got %d)", A);
  CMB_CUDA(cudaGetLastError());
}
void launch_mica_permutations(int A, int T, int64_t S, int64_t n_pad, const uint8_t* tips, const uint32_t* cmask, uint64_t seed,
                              int max_perm, int shard_index, int shard_count, int64_t n_rows, unsigned long long* next,
                              double* pvalue, int32_t* nperm, cudaStream_t st) {
  if (S < 2 || n_rows == 0) return;
  if (T < 2) fail("mica permutations: at least two sequences are needed");
  if (T > 65535) fail("mica: %d sequences exceed the 16-bit cells of the joint table", T);
  const size_t T4 = ((size_t)T + 3) / 4;
  const size_t q_bytes = ((size_t)(T + 1) * 16 + 15) & ~(size_t)15;
  auto bytes = [&](int nt) { return 1024 + q_bytes + (size_t)(nt / 32) * 8 * T4 + 8 * T4 * nt; };  // masks | c / T, (c / T) ln(c / T) | warps' pairs | private copies
  int nt = 128;
  while (nt > 32 && bytes(nt) > 64 * 1024) nt >>= 1;
  const size_t smem = bytes(nt);
  if (smem > 200 * 1024) fail("mica permutations: %d sequences exceed the shared memory of a one-warp CTA", T);
  auto kernel = A == 4 ? k5_permutations<4, 5> : A == 20 ? k5_permutations<20, 5> : nullptr;
  if (!kernel) fail("mica kernels are built for A = 4 and A = 20 (got %d)", A);
  CMB_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  int dev = 0, sms = 0, per_sm = 0;
  CMB_CUDA(cudaGetDevice(&dev));
  CMB_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  CMB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, nt, smem));
  if (per_sm < 1) fail("mica permutations: the kernel does not fit an SM (T = %d)", T);
  // persistent warps, one wave; the shard's pairs are handed out by a counter: no more warps than pairs
  const int64_t ctas = std::min<int64_t>((int64_t)sms * per_sm, (n_rows + nt / 32 - 1) / (nt / 32));
  CMB_CUDA(cudaMemsetAsync(next, 0, sizeof(unsigned long long), st));
  // CMB_K5_FILTER=0: every shuffle through the reference's formula (same table; for A/B runs and tests)
  static const int use_filter = [] { const char* e = getenv("CMB_K5_FILTER"); return e ? atoi(e) : 1; }();
  kernel<<<(unsigned)ctas, nt, smem, st>>>(T, S, n_rows, shard_index, shard_count, n_pad, tips, cmask, seed, max_perm, use_filter,
                                           next, pvalue, nperm);
  CMB_CUDA(cudaGetLastError());
}
void launch_mica_average(int64_t S, const double* mi, double* avg, cudaStream_t st) {
  k5_average<<<(unsigned)((S + 127) / 128), 128, 0, st>>>(S, mi, avg);
  CMB_CUDA(cudaGetLastError());
}
void launch_mica_rows(int64_t S, const double* entropy, const double* norm, int32_t* oi, int32_t* oj, double* hmin, double* nmin,
                      cudaStream_t st) {
  if (S < 2) return;
  dim3 grid((unsigned)((S - 1 + 127) / 128), (unsigned)(S - 1));
  k5_rows<<<grid, 128, 0, st>>>(S, entropy, norm, oi, oj, hmin, nmin);
  CMB_CUDA(cudaGetLastError());
}
void launch_min2(int64_t n, const double* a, const double* b, double* out, cudaStream_t st) {
  if (n == 0) return;
  k5_min2<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(n, a, b, out);
  CMB_CUDA(cudaGetLastError());
}

} // namespace cmb
