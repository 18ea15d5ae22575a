// K2: site-pair statistics on the device.
//
//  * k2_paired   -- null distribution: statistic of site j of batch 1 with site j of batch 2
//                   (AnalysisTools.cpp:637-640), one thread per pair, coalesced over sites.
//  * k2_tiles    -- all pairs i<j of the mapped alignment (CoETools.cpp:672-724) or the full
//                   distance matrix (CoMap.cpp:432-440): 64x64 register-tiled fp64 Gram
//                   tiles over the [branch][site] matrix; centring / indicator transforms
//                   are fused into the tile load, the statistic, the filters and the
//                   p-value lookup (binary search in the sorted per-bin null) into the
//                   epilogue.  Statistics formulas: Statistics.h:164-265; VectorTools::cor
//                   = cov/(sd sd) with the unbiased factors kept as the reference has them.
//  * null binning + per-bin sort (Domain.cpp:113-122, CoETools.cpp:650-652) with CUB radix
//    sorts (library code, not a hot step: 1e6 keys).
#include "device_utils.cuh"
#include "kernels.h"
#include <cub/cub.cuh>
#include <cuda/functional>
#include <cstdlib>

namespace cmb {
namespace {

// Domain(0, nmax, K).getIndex, CoMap/Domain.cpp:46-59,113-122 (bounds_[i] = mini + i*w)
__device__ __forceinline__ int domain_index(double nmax, int K, double x) {
  double w = nmax / (double)K;
  double upper = 0. + (double)K * w;
  if (x < 0. || x >= upper || !(x == x)) return -1;
  for (int i = 1; i < K + 1; i++)
    if (x < 0. + (double)i * w) return i - 1;
  return -1;
}

// ---------------------------------------------------------------------------- paired
// Exactness: p-values count null values strictly below an observed statistic
// (CoETools.cpp:715), and low-rate sites produce massive ties (e.g. r = 1 between two
// constant sites), so a 1-ulp change of a statistic moves counts by dozens.  All pair
// statistics therefore replicate the reference's operation order (VectorTools::mean ->
// center -> scalar, sums over branches in id order) with explicitly unfused multiplies
// and adds: given identical mapping vectors they are bit-identical to the CPU restatement.
__device__ __forceinline__ double mul_(double a, double b) { return __dmul_rn(a, b); }
__device__ __forceinline__ double add_(double a, double b) { return __dadd_rn(a, b); }

// mv (nullable): the observed alignment's mean vector, subtracted from both sites before a
// correlation (CorrectedCorrelationStatistic, Statistics.h:176-205); the norms stay raw.
// DiscreteMutualInformationStatistic with the bounds {0, threshold, 10000} of statistic=MI(threshold=..)
// (CoETools.cpp:590-595, Statistics.h:307-329): every branch entry becomes the category [v >= threshold]
// and the statistic is [Bio++, from memory] VectorTools::miDiscrete(c1, c2, base = 2.7182818):
//   sum over the occupied cells (k1, k2) in key order of  (n12 / n) * log(n12 * n / (n1[k1] * n2[k2])) / log(base).
// n1x / n1y: branches of the first / second site in category 1, n11: in category 1 for both.
__device__ __forceinline__ double mi_binary(double n, double n1x, double n1y, double n11) {
  const double cx[2] = {n - n1x, n1x}, cy[2] = {n - n1y, n1y};
  const double c12[2][2] = {{n - n1x - n1y + n11, n1y - n11}, {n1x - n11, n11}};
  const double lb = log(2.7182818);
  double s = 0.;
#pragma unroll
  for (int a = 0; a < 2; a++)
#pragma unroll
    for (int b = 0; b < 2; b++)
      if (c12[a][b] > 0.) s = add_(s, mul_(c12[a][b] / n, log(mul_(c12[a][b], n) / mul_(cx[a], cy[b]))) / lb);
  return s;
}

// statistic=MI with nijt=Label and nijt.average=no (CoETools.cpp:577-589): the bounds -0.5, 0.5, ..., A(A-1)+0.5 make
// the category of a branch its substitution label (0 = no substitution) and the statistic is the same
// [Bio++, from memory] miDiscrete over every occupied cell of the joint table.  Most branches of a site carry no
// substitution, so only the branches where either site has one are listed (packed keys); the (0, 0) cell and the
// marginals of category 0 follow from the list.  A pair with more than kMiList such branches re-reads its columns.
constexpr int kMiList = 64;
__device__ __forceinline__ int label_of(double v) {
  if (!(v >= -0.5)) return 0;          // below the first bound the reference's Domain throws; labels never are
  int k = (int)floor(v);
  if (v >= (double)k + 0.5) k++;
  return k > 65535 ? 65535 : k;
}
__device__ __forceinline__ double mi_term(double n, double lb, double c12, double c1, double c2) {
  return mul_(c12 / n, log(mul_(c12, n) / mul_(c1, c2))) / lb;
}
__device__ __noinline__ double mi_labels(const double* __restrict__ x, size_t sx, const double* __restrict__ y, size_t sy, int B) {
  int keys[kMiList];
  int m = 0, n1 = 0, n2 = 0;
  for (int b = 0; b < B; b++) {
    const int a = label_of(x[(size_t)b * sx]), c = label_of(y[(size_t)b * sy]);
    if (a | c) {
      if (m < kMiList) keys[m] = a << 16 | c;
      m++; n1 += a != 0; n2 += c != 0;
    }
  }
  const double n = (double)B, lb = log(2.7182818);
  const double c10 = (double)(B - n1), c20 = (double)(B - n2);
  double s = 0.;
  if (B - m > 0) s = mi_term(n, lb, (double)(B - m), c10, c20);
  if (m <= kMiList) {
    for (int e = 0; e < m; e++) {
      const int key = keys[e], a = key >> 16, c = key & 0xffff;
      bool first = true;
      for (int f = 0; f < e; f++) first = first && keys[f] != key;
      if (!first) continue;
      int c12 = 0, c1 = 0, c2 = 0;
      for (int f = 0; f < m; f++) { c12 += keys[f] == key; c1 += (keys[f] >> 16) == a; c2 += (keys[f] & 0xffff) == c; }
      s = add_(s, mi_term(n, lb, (double)c12, a ? (double)c1 : c10, c ? (double)c2 : c20));
    }
  } else {
    for (int b = 0; b < B; b++) {
      const int a = label_of(x[(size_t)b * sx]), c = label_of(y[(size_t)b * sy]);
      if (!(a | c)) continue;
      int c12 = 0, c1 = 0, c2 = 0;
      bool first = true;
      for (int f = 0; f < B; f++) {
        const int a2 = label_of(x[(size_t)f * sx]), c2v = label_of(y[(size_t)f * sy]);
        if (a2 == a && c2v == c) { c12++; if (f < b) first = false; }
        c1 += a2 == a; c2 += c2v == c;
      }
      if (first) s = add_(s, mi_term(n, lb, (double)c12, (double)c1, (double)c2));
    }
  }
  return s;
}

template <int STAT>
__global__ void __launch_bounds__(128) k2_paired(double thr, int B, int64_t n, int64_t n_pad, int64_t n_pad2, const double* __restrict__ o1,
                          const double* __restrict__ o2, const double* __restrict__ mv, const double* __restrict__ mv2,
                          double* __restrict__ stat, double* __restrict__ nmin, const int32_t* __restrict__ col1,
                          const int32_t* __restrict__ col2) {
  const int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= n) return;
  // pattern-compressed mappings: the vectors of pair j live in columns col1[j] / col2[j]
  o1 += col1 ? col1[j] - j : 0;
  o2 += col2 ? col2[j] - j : 0;
  constexpr int stat_id = STAT;
  const double nb = (double)B;
  double sx = 0., sy = 0., qx = 0., qy = 0., sxy = 0., s3 = 0., cnt = 0.;
  for (int b = 0; b < B; b++) {
    const double x = o1[(size_t)b * n_pad + j], y = o2[(size_t)b * n_pad2 + j];
    if (mv) {
      sx = add_(sx, add_(x, -mv[b]));
      sy = add_(sy, add_(y, -mv2[b]));
    } else {
      sx = add_(sx, x);
      sy = add_(sy, y);
    }
    qx = add_(qx, mul_(x, x));
    qy = add_(qy, mul_(y, y));
    if (stat_id == 2) sxy = add_(sxy, mul_(x, y));
    if (stat_id == 3 && x >= 1. && y >= 1.) cnt += 1.;
    if (stat_id == 4) { double t = add_(x, y); s3 = add_(s3, mul_(t, t)); }
    if (stat_id == 6) { cnt += (x >= thr && y >= thr) ? 1. : 0.; sxy += x >= thr ? 1. : 0.; s3 += y >= thr ? 1. : 0.; }
  }
  double r;
  if (stat_id == 6) r = mi_binary(nb, sxy, s3, cnt);
  else if (stat_id == 7) r = mi_labels(o1 + j, (size_t)n_pad, o2 + j, (size_t)n_pad2, B);
  else if (stat_id == 0 || stat_id == 1) {
    const double mx = sx / nb, my = sy / nb;
    double cxy = 0., cxx = 0., cyy = 0.;
    for (int b = 0; b < B; b++) {
      double x = o1[(size_t)b * n_pad + j], y = o2[(size_t)b * n_pad2 + j];
      if (mv) { x = add_(x, -mv[b]); y = add_(y, -mv2[b]); }
      x = add_(x, -mx);
      y = add_(y, -my);
      cxy = add_(cxy, mul_(x, y));
      cxx = add_(cxx, mul_(x, x));
      cyy = add_(cyy, mul_(y, y));
    }
    cxy = cxy / nb * nb / (nb - 1.);
    cxx = cxx / nb * nb / (nb - 1.);
    cyy = cyy / nb * nb / (nb - 1.);
    r = stat_id == 0 ? cxy / mul_(sqrt(cxx), sqrt(cyy)) : cxy;
  } else if (stat_id == 2) r = sxy / mul_(sqrt(qx), sqrt(qy));
  else if (stat_id == 3) r = cnt;
  else r = add_(1., -(sqrt(s3) / add_(sqrt(qx), sqrt(qy))));
  stat[j] = r;
  const double a = sqrt(qx), c = sqrt(qy);
  nmin[j] = a < c ? a : c;
}

// statistic of listed column pairs (a, b) of ONE mapping matrix: the group statistics of the
// candidates analysis (AbstractMinimumStatistic::getValueForGroup, Statistics.h:118-131).  Same
// operation order as k2_paired; one thread per pair.
__global__ void k2_pair_list(int stat_id, double thr, int B, int64_t n_pad, const double* __restrict__ o, const double* __restrict__ mv,
                             const int2* __restrict__ pairs, int64_t n_pairs, double* __restrict__ stat) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n_pairs) return;
  const int64_t ja = pairs[t].x, jb = pairs[t].y;
  const double nb = (double)B;
  double sx = 0., sy = 0., qx = 0., qy = 0., sxy = 0., s3 = 0., cnt = 0.;
  for (int b = 0; b < B; b++) {
    const double x = o[(size_t)b * n_pad + ja], y = o[(size_t)b * n_pad + jb];
    if (mv) {
      sx = add_(sx, add_(x, -mv[b]));
      sy = add_(sy, add_(y, -mv[b]));
    } else {
      sx = add_(sx, x);
      sy = add_(sy, y);
    }
    qx = add_(qx, mul_(x, x));
    qy = add_(qy, mul_(y, y));
    if (stat_id == 2) sxy = add_(sxy, mul_(x, y));
    if (stat_id == 3 && x >= 1. && y >= 1.) cnt += 1.;
    if (stat_id == 4) { double u = add_(x, y); s3 = add_(s3, mul_(u, u)); }
    if (stat_id == 6) { cnt += (x >= thr && y >= thr) ? 1. : 0.; sxy += x >= thr ? 1. : 0.; s3 += y >= thr ? 1. : 0.; }
  }
  double r;
  if (stat_id == 6) r = mi_binary(nb, sxy, s3, cnt);
  else if (stat_id == 7) r = mi_labels(o + ja, (size_t)n_pad, o + jb, (size_t)n_pad, B);
  else if (stat_id == 0 || stat_id == 1) {
    const double mx = sx / nb, my = sy / nb;
    double cxy = 0., cxx = 0., cyy = 0.;
    for (int b = 0; b < B; b++) {
      double x = o[(size_t)b * n_pad + ja], y = o[(size_t)b * n_pad + jb];
      if (mv) { x = add_(x, -mv[b]); y = add_(y, -mv[b]); }
      x = add_(x, -mx);
      y = add_(y, -my);
      cxy = add_(cxy, mul_(x, y));
      cxx = add_(cxx, mul_(x, x));
      cyy = add_(cyy, mul_(y, y));
    }
    cxy = cxy / nb * nb / (nb - 1.);
    cxx = cxx / nb * nb / (nb - 1.);
    cyy = cyy / nb * nb / (nb - 1.);
    r = stat_id == 0 ? cxy / mul_(sqrt(cxx), sqrt(cyy)) : cxy;
  } else if (stat_id == 2) r = sxy / mul_(sqrt(qx), sqrt(qy));
  else if (stat_id == 3) r = cnt;
  else r = add_(1., -(sqrt(s3) / add_(sqrt(qx), sqrt(qy))));
  stat[t] = r;
}

__global__ void k2_raw_rows(int64_t n, const double* stat, const double* nmin, const int32_t* rc1,
                            const int32_t* rc2, const double* pr1, const double* pr2, double* raw, const int32_t* col1,
                            const int32_t* col2) {
  const int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= n) return;
  const int64_t a = col1 ? col1[j] : j, b = col2 ? col2[j] : j;
  raw[j * 4 + 0] = stat[j];
  raw[j * 4 + 1] = (double)(rc1[a] < rc2[b] ? rc1[a] : rc2[b]);
  raw[j * 4 + 2] = pr1[a] < pr2[b] ? pr1[a] : pr2[b];
  raw[j * 4 + 3] = nmin[j];
}

// ---------------------------------------------------------------------------- pattern compression
// launch_compress_patterns.  Entry k of the keys belongs to column k of the first batch, or to column half + k - n
__device__ __forceinline__ int64_t key_column(int64_t k, int64_t n, int64_t half) { return k < n ? k : half + k - n; }
__device__ __forceinline__ bool batch_column(int64_t s, int64_t n, int64_t half) { return s < n || (s >= half && s < half + n); }

// The key of every column of a batch the simulator did not key (host alignments, continuous rates): the same words
// and hash as k3_simulate, the rows taken in its walk order (loads coalesced across the warp)
__global__ void k2_column_keys(int T, int64_t n, int64_t half, int64_t n_pad, const uint8_t* __restrict__ tips,
                               const int32_t* __restrict__ leaf_rows, uint64_t* __restrict__ hash, int32_t* __restrict__ col,
                               uint32_t* __restrict__ packed) {
  const int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= 2 * n) return;
  const int64_t s = key_column(k, n, half);
  uint64_t h = kColumnHashInit;
  for (int w = 0; 16 * w < T; w++) {
    const int m = min(16, T - 16 * w);
    uint32_t word = 0;
#pragma unroll 16
    for (int j = 0; j < m; j++) word |= (uint32_t)tips[(size_t)__ldg(leaf_rows + 16 * w + j) * n_pad + s] << (2 * j);
    packed[(size_t)w * n_pad + s] = word;
    h = column_hash_step(h, word);
  }
  hash[k] = column_hash_final(h);
  col[k] = (int32_t)s;
}
// sorted entry i opens a run of equal (masked) hashes: i, else 0 -- a max-scan then gives every entry its run's start
__global__ void k2_run_starts(int64_t m, const uint64_t* __restrict__ hs, uint64_t mask, int32_t* __restrict__ start) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= m) return;
  start[i] = (i == 0 || ((hs[i] ^ hs[i - 1]) & mask) != 0) ? (int32_t)i : 0;
}
// rep[column] = the column heading its run (the stable sort put the lowest column first), stored as ~head for the
// head itself; the columns of runs shorter than min_run represent themselves
__global__ void k2_run_heads(int64_t m, int min_run, const int32_t* __restrict__ run_start, const int32_t* __restrict__ cs,
                             int32_t* __restrict__ rep) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= m) return;
  const int64_t st = run_start[i];
  const bool merged = st + min_run - 1 < m && run_start[st + min_run - 1] == st;
  const int32_t h = cs[st];
  rep[cs[i]] = !merged ? cs[i] : st == i ? ~h : h;
}
// A column joins its run's head only if their packed tips are equal; otherwise it represents itself.  Scan value
// of a representative: 1 << 32 for the head of a run with other members, 1 for any other.
__global__ void k2_pick_representatives(int W, int64_t n, int64_t half, int64_t n_pad, const uint32_t* __restrict__ packed,
                                        int32_t* __restrict__ rep, int64_t* __restrict__ val) {
  const int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= n_pad) return;
  int64_t v = 0;
  if (batch_column(s, n, half)) {
    const int32_t h = rep[s];
    if (h < 0) {
      rep[s] = ~h;
      v = (int64_t)1 << 32;
    } else if (h != s) {
      bool joins = true;
#pragma unroll 8
      for (int w = 0; w < W; w++) joins &= packed[(size_t)w * n_pad + s] == packed[(size_t)w * n_pad + h];
      if (!joins) { rep[s] = (int32_t)s; v = 1; }
    } else v = 1;
  }
  val[s] = v;
}
// packed column of representative r: the columns mapped for themselves alone first, the heads of runs behind them
__device__ __forceinline__ int32_t packed_column(int64_t r, const int64_t* __restrict__ val, const int64_t* __restrict__ pos,
                                                 int32_t n_alone) {
  return val[r] == 1 ? (int32_t)pos[r] : n_alone + (int32_t)(pos[r] >> 32);
}
// The heads of merged runs sit together behind the other representatives: k2_paired reads a shared vector for every
// member, and a narrow band of columns keeps those reads in fewer pages and in L2 (B200, config 4, every repeated
// column merged: k2_paired 7.8 ms with the band, 10.7 ms with the heads in column order, 4.3 ms uncompressed).
__global__ void k2_compact_columns(int T, int64_t n, int64_t half, int64_t n_pad, const uint8_t* __restrict__ tips,
                                   const int32_t* __restrict__ rep, const int64_t* __restrict__ val,
                                   const int64_t* __restrict__ pos, uint8_t* __restrict__ tips_c, int32_t* __restrict__ col,
                                   int32_t* __restrict__ count) {
  const int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= n_pad) return;
  const int64_t tot = pos[n_pad - 1] + val[n_pad - 1];
  const int32_t n_alone = (int32_t)(tot & 0xffffffff), nr = n_alone + (int32_t)(tot >> 32);
  if (s == 0) *count = nr;
  if (batch_column(s, n, half)) {
    const int32_t r = rep[s], d = packed_column(r, val, pos, n_alone);
    if (r == s) {
#pragma unroll 16
      for (int t = 0; t < T; t++) tips_c[(size_t)t * n_pad + d] = tips[(size_t)t * n_pad + s];
    }
    col[s] = d;
  } else col[s] = 0;
  // one CTA's worth of valid filler behind the representatives
  if (s < 256 && nr + s < n_pad)
    for (int t = 0; t < T; t++) tips_c[(size_t)t * n_pad + nr + s] = 0;
}

// ---------------------------------------------------------------------------- binning
__global__ void k2_bin_keys(int64_t n, const double* nmin, double nmax, int K, uint32_t* cat) {
  const int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= n) return;
  int c = domain_index(nmax, K, nmin[j]);
  cat[j] = c < 0 ? (uint32_t)K : (uint32_t)c;
}
__global__ void k2_bin_offsets(int64_t n, const uint32_t* cat_sorted, int K, int64_t* off) {
  int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k > K) return;
  int64_t lo = 0, hi = n; // first index with cat >= k
  while (lo < hi) {
    int64_t mid = (lo + hi) >> 1;
    if (cat_sorted[mid] < (uint32_t)k) lo = mid + 1; else hi = mid;
  }
  off[k] = lo;
}

// ---------------------------------------------------------------------------- per-site prep
// mean, sd (unbiased, as VectorTools::sd) and norm per site from the [B][n_pad] matrix,
// summed over branches in id order without fused operations (see k2_paired)
__global__ void k2_prep(int B, int64_t n, int64_t n_pad, const double* __restrict__ out,
                        const double* __restrict__ mv, double* mean, double* sd, double* norm) {
  const int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= n) return;
  const double nb = (double)B;
  double sx = 0., qx = 0.;
  for (int b = 0; b < B; b++) {
    const double x = out[(size_t)b * n_pad + s];
    sx = add_(sx, mv ? add_(x, -mv[b]) : x);
    qx = add_(qx, mul_(x, x));
  }
  const double m = sx / nb;
  double css = 0.;
  for (int b = 0; b < B; b++) {
    double x = out[(size_t)b * n_pad + s];
    if (mv) x = add_(x, -mv[b]);
    x = add_(x, -m);
    css = add_(css, mul_(x, x));
  }
  mean[s] = m;
  sd[s] = sqrt(css / nb * nb / (nb - 1.));
  norm[s] = sqrt(qx);
}

// branches of each site whose entry reaches the MI threshold (category 1)
__global__ void k2_count_ge(int B, int64_t n, int64_t n_pad, const double* __restrict__ out, double thr, double* cnt) {
  const int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= n) return;
  double c = 0.;
  for (int b = 0; b < B; b++) c += out[(size_t)b * n_pad + s] >= thr ? 1. : 0.;
  cnt[s] = c;
}

// mean vector of the mapped alignment: mv[b] = (sum over sites, in site order, of n_b(site)) / S
// (CoMap.cpp:350-359), one thread per branch
__global__ void k2_mean_vector(int B, int64_t S, int64_t n_pad, const double* __restrict__ out, double* mv) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  double t = 0.;
  for (int64_t s = 0; s < S; s++) t = add_(t, out[(size_t)b * n_pad + s]);
  mv[b] = t / (double)S;
}

// ---------------------------------------------------------------------------- tiles
constexpr int TS = 64;  // tile edge (sites)
constexpr int BK = 16;  // branches per smem stage
enum { MODE_PAIRS = 0, MODE_DIST = 1, MODE_RECT = 2 };

struct TileParams {
  int stat_id, mode, B;
  int64_t S, S_pad;
  const double* out;          // [B][S_pad]
  const double *mean, *sd, *norm, *post_rate;
  const double* mv;           // mean vector subtracted before centring (corrected correlation) or nullptr
  const int32_t* rate_class;
  // MODE_RECT (two data sets, CoETools.cpp:732-840): the column operand, its per-site arrays
  // and the second data set's own rate filters; in the other modes these alias the first
  int64_t S2, S2_pad;
  const double *out2, *mean2, *sd2, *norm2, *post_rate2, *mv2;
  const int32_t* rate_class2;
  int min_rate_class2;
  double min_rate2;
  double thr;                 // MI threshold
  int nmin_by_row;            // upstream quirk: min(Nmin) pairs norms1[i] with norms2[i] (CoETools.cpp:803)
  const int2* tiles;          // (ti, tj) with tj >= ti
  const int32_t* rows;        // owned row list (gathered i-dimension) or nullptr = identity
  int64_t n_rows;             // number of owned rows
  const int64_t* row_off;     // [n_rows] start of each owned row in the dense output
  // filters (CoETools.cpp:420-481)
  int min_rate_class, max_rate_class_diff;
  double min_rate, max_rate_diff, min_stat;
  int any_filter;
  // null
  int K;
  double nmax;
  const int64_t* bin_off;
  const double* sorted;
  // outputs (dense upper triangle of the owned rows), all nullable
  int32_t *o_i, *o_j, *o_rcmin;
  double *o_stat, *o_prmin, *o_nmin, *o_pvalue;
  int32_t* o_nsim;
  uint8_t* o_keep;
  double* mat;                // MODE_DIST: [S][S]
  double dist_comp;           // distance = comp - stat (Distance.h:334-337), or stat itself
  int dist_is_stat;
};

template <int STAT>
__device__ __forceinline__ double tile_load(double x, double mean, double thr = 0.) {
  if (STAT == 0 || STAT == 1) return add_(x, -mean);
  if (STAT == 3) return x >= 1. ? 1. : 0.;
  if (STAT == 6) return x >= thr ? 1. : 0.;
  if (STAT == 7) return 0.; // the label statistic reads its two columns in the epilogue (mi_labels)
  return x;
}

// One pair (row ri of the owned rows = site i, column site j) from its accumulated sum: statistic, filters,
// Domain bin, p-value, stores.  Shared by the unfused and the tensor-core tile kernels.
// #{sim < stat} in the pair's Nmin bin for NV pairs at once: the binary searches advance in lock step so that their
// loads -- dependent L2 round trips, 17 per pair at 10^5 samples per bin -- overlap instead of queueing behind each
// other (ncu r2m: 29 % of the tile kernel's stalls were these loads).  Same counts as one search after the other.
template <int NV>
__device__ __forceinline__ void pvalues_interleaved(const TileParams& p, const bool (&valid)[NV], const int64_t (&idx)[NV],
                                                    const double (&stat)[NV], const double (&nm)[NV]) {
  const double* sim[NV];
  int32_t lo[NV], hi[NV], nsim[NV];
  bool any = false;
#pragma unroll
  for (int v = 0; v < NV; v++) {
    sim[v] = p.sorted; lo[v] = hi[v] = nsim[v] = 0;
    if (!valid[v]) continue;
    const int cat = domain_index(p.nmax, p.K, nm[v]);
    if (cat >= 0) {
      sim[v] = p.sorted + p.bin_off[cat];
      nsim[v] = (int32_t)(p.bin_off[cat + 1] - p.bin_off[cat]);
      hi[v] = nsim[v];
      any |= nsim[v] > 0;
    } else nsim[v] = -1; // outside [0, nmax): "NA\t0"
  }
  while (any) {
    double x[NV];
    int32_t mid[NV];
#pragma unroll
    for (int v = 0; v < NV; v++) {
      mid[v] = (int32_t)(((int64_t)lo[v] + hi[v]) >> 1);
      x[v] = lo[v] < hi[v] ? sim[v][mid[v]] : 0.;
    }
    any = false;
#pragma unroll
    for (int v = 0; v < NV; v++) {
      if (lo[v] < hi[v]) {
        if (x[v] < stat[v]) lo[v] = mid[v] + 1; else hi[v] = mid[v];
      }
      any |= lo[v] < hi[v];
    }
  }
#pragma unroll
  for (int v = 0; v < NV; v++) {
    if (!valid[v]) continue;
    const bool in = nsim[v] >= 0;
    const int32_t ns = in ? nsim[v] : 0;
    if (p.o_pvalue) p.o_pvalue[idx[v]] = in ? (double)(ns - lo[v] + 1) / (double)(ns + 1) : nan("");
    if (p.o_nsim) p.o_nsim[idx[v]] = ns;
  }
}

// One pair (row ri of the owned rows = site i, column site j) from its accumulated sum: statistic, filters,
// stores; the p-value either here (one search) or deferred to pvalues_interleaved (idx / stat / Nmin returned).
// Shared by the unfused and the tensor-core tile kernels.
template <int STAT>
__device__ __forceinline__ double pair_stat(const TileParams& p, int64_t i, int64_t j, double a) {
  const double nb = (double)p.B;
  if (STAT == 0) return (a / nb * nb / (nb - 1.)) / mul_(p.sd[i], p.sd2[j]);
  else if (STAT == 1) return a / nb * nb / (nb - 1.);
  else if (STAT == 2) return a / mul_(p.norm[i], p.norm2[j]);
  else if (STAT == 3) return a;
  else if (STAT == 4) return add_(1., -(sqrt(a) / add_(p.norm[i], p.norm2[j])));
  else if (STAT == 6) return mi_binary(nb, p.mean[i], p.mean2[j], a); // mean arrays hold the category-1 counts
  else if (STAT == 7) return mi_labels(p.out + i, (size_t)p.S_pad, p.out2 + j, (size_t)p.S2_pad, p.B); // from the columns themselves
  else return sqrt(a);
}
template <int STAT, bool DEFER = false>
__device__ __forceinline__ void pair_epilogue(const TileParams& p, int64_t ri, int64_t i, int64_t j, double a,
                                              int64_t* idx_out = nullptr, double* stat_out = nullptr, double* nm_out = nullptr) {
  const double stat = pair_stat<STAT>(p, i, j, a);
  if (p.mode == MODE_DIST) {
    double d = p.dist_is_stat ? stat : p.dist_comp - stat;
    p.mat[(size_t)i * p.S + j] = d;
    p.mat[(size_t)j * p.S + i] = d;
    return;
  }
  const int64_t idx = p.mode == MODE_RECT ? i * p.S2 + j : p.row_off[ri] + (j - i - 1);
  const int ci = p.rate_class[i], cj = p.rate_class2[j];
  const double pi_ = p.post_rate[i], pj = p.post_rate2[j];
  const double ni = p.norm[i], nj = p.norm2[p.nmin_by_row && i < p.S2 ? i : j];
  if (p.any_filter) {
    bool keep = ci >= p.min_rate_class && cj >= p.min_rate_class2 && !(pi_ < p.min_rate) && !(pj < p.min_rate2);
    if (p.max_rate_class_diff >= 0 && abs(cj - ci) > p.max_rate_class_diff) keep = false;
    if (p.max_rate_diff >= 0. && fabs(pj - pi_) > p.max_rate_diff) keep = false;
    if (fabs(stat) < p.min_stat) keep = false;
    p.o_keep[idx] = keep ? 1 : 0;
  }
  const double nm = ni < nj ? ni : nj;
  if (p.o_i) p.o_i[idx] = (int32_t)i;
  if (p.o_j) p.o_j[idx] = (int32_t)j;
  if (p.o_stat) p.o_stat[idx] = stat;
  if (p.o_rcmin) p.o_rcmin[idx] = ci < cj ? ci : cj;
  if (p.o_prmin) p.o_prmin[idx] = pi_ < pj ? pi_ : pj;
  if (p.o_nmin) p.o_nmin[idx] = nm;
  if constexpr (DEFER) {
    *idx_out = idx; *stat_out = stat; *nm_out = nm;
    return;
  }
  if (p.K > 0 && (p.o_pvalue || p.o_nsim)) {
    int cat = domain_index(p.nmax, p.K, nm);
    double pv = nan("");
    int64_t nsim = 0;
    if (cat >= 0) {
      const double* sim = p.sorted + p.bin_off[cat];
      nsim = p.bin_off[cat + 1] - p.bin_off[cat];
      int64_t lo = 0, hi = nsim; // count = #{sim < stat} on the ascending bin
      while (lo < hi) {
        int64_t mid = (lo + hi) >> 1;
        if (sim[mid] < stat) lo = mid + 1; else hi = mid;
      }
      pv = (double)(nsim - lo + 1) / (double)(nsim + 1);
    }
    if (p.o_pvalue) p.o_pvalue[idx] = pv;
    if (p.o_nsim) p.o_nsim[idx] = (int32_t)nsim;
  }
}

template <int STAT>
__global__ void __launch_bounds__(256) k2_tiles(TileParams p) {
  __shared__ __align__(16) double stage[2][BK][TS];
  double (*As)[TS] = stage[0];
  double (*Bs)[TS] = stage[1];
  const int2 t = p.tiles[blockIdx.x];
  const int64_t i0 = (int64_t)t.x * TS, j0 = (int64_t)t.y * TS;
  const int tid = threadIdx.x;
  const int tx = tid & 15, ty = tid >> 4; // thread tile: rows u*16+ty, cols v*16+tx (u, v < 4)
  // loader mapping: 4 elements per thread per operand: k = tid / 16, cols (tid % 16) * 4 ..
  const int lk = tid >> 4, lc = (tid & 15) * 4;
  int64_t ai[4], bj[4];
  double am[4], bm[4];
#pragma unroll
  for (int u = 0; u < 4; u++) {
    int64_t ri = i0 + lc + u;
    ai[u] = ri < p.n_rows ? (p.rows ? p.rows[ri] : ri) : -1;
    int64_t cj = j0 + lc + u;
    bj[u] = cj < p.S2 ? cj : -1;
    am[u] = ai[u] >= 0 ? p.mean[ai[u]] : 0.;
    bm[u] = bj[u] >= 0 ? p.mean2[bj[u]] : 0.;
  }
  double acc[4][4];
#pragma unroll
  for (int u = 0; u < 4; u++)
#pragma unroll
    for (int v = 0; v < 4; v++) acc[u][v] = 0.;

  // stage = BK branches of both operands; the global loads of stage n + 1 are issued before the products of
  // stage n (register double buffering): without it 32 % of the warp stalls were on the loads of the next stage
  double ra[4], rb[4];
  auto fetch = [&](int k0) {
    const int k = k0 + lk;
    const double* rowp = p.out + (size_t)k * p.S_pad;
    const double* colp = p.out2 + (size_t)k * p.S2_pad;
    const double mvk = (STAT == 0 && p.mv && k < p.B) ? p.mv[k] : 0.;
    const double mvk2 = (STAT == 0 && p.mv && k < p.B) ? p.mv2[k] : 0.;
#pragma unroll
    for (int u = 0; u < 4; u++) {
      double a = 0., b = 0.;
      if (k < p.B) {
        if (STAT == 0 && p.mv) {
          if (ai[u] >= 0) a = tile_load<STAT>(add_(rowp[ai[u]], -mvk), am[u]);
          if (bj[u] >= 0) b = tile_load<STAT>(add_(colp[bj[u]], -mvk2), bm[u]);
        } else {
          if (ai[u] >= 0) a = tile_load<STAT>(rowp[ai[u]], am[u], p.thr);
          if (bj[u] >= 0) b = tile_load<STAT>(colp[bj[u]], bm[u], p.thr);
        }
      }
      ra[u] = a; rb[u] = b;
    }
  };
  fetch(0);
  for (int k0 = 0; k0 < p.B; k0 += BK) {
#pragma unroll
    for (int u = 0; u < 4; u += 2) {
      *reinterpret_cast<double2*>(&As[lk][lc + u]) = make_double2(ra[u], ra[u + 1]);
      *reinterpret_cast<double2*>(&Bs[lk][lc + u]) = make_double2(rb[u], rb[u + 1]);
    }
    __syncthreads();
    if (k0 + BK < p.B) fetch(k0 + BK);
#pragma unroll
    for (int kk = 0; kk < BK; kk++) {
      // rows u*16+ty, columns v*16+tx: every operand read is one 64-bit LDS whose 32 lanes touch one 128-byte
      // line (a: two addresses, b: sixteen, the other half-warp broadcast) = 1 wavefront.  The 4x4 blocked
      // mapping (rows ty*4.., cols tx*4.. as 128-bit loads) cost 24 wavefronts per kk against 16 cycles of
      // FP64 issue (ncu r2m: l1tex 81 %, FP64 pipe 45 %); this one costs 8.  Three CTAs per SM instead of two
      // (__launch_bounds__(256, 3): 80 registers, ~150 B of spills) measured slower: pairs 3.3 vs 2.95 ms, the
      // 20 000-site distance matrix 15.9 vs 13.9 ms.
      double a[4], b[4];
#pragma unroll
      for (int u = 0; u < 4; u++) { a[u] = As[kk][u * 16 + ty]; b[u] = Bs[kk][u * 16 + tx]; }
#pragma unroll
      for (int u = 0; u < 4; u++)
#pragma unroll
        for (int v = 0; v < 4; v++) {
          if (STAT == 4) { double s = add_(a[u], b[v]); acc[u][v] = add_(acc[u][v], mul_(s, s)); }
          else if (STAT == 5) { double s = add_(b[v], -a[u]); acc[u][v] = add_(acc[u][v], mul_(s, s)); }
          else acc[u][v] = add_(acc[u][v], mul_(a[u], b[v]));
        }
    }
    __syncthreads();
  }

  if (p.mode == MODE_DIST) {
    // d(i,j) goes to both triangles.  The upper one is written from the registers (16 lanes = 128 contiguous
    // bytes); the mirror image is transposed through the (now free) stage memory, 16 tile rows at a time, so that
    // it leaves as 128-byte row segments too instead of one 8-byte store per matrix row.
    static_assert(sizeof(stage) >= TS * 17 * sizeof(double), "transpose buffer");
    double (*T)[17] = reinterpret_cast<double (*)[17]>(&stage[0][0][0]);
    const int c = tid & 15, r = tid >> 4;
#pragma unroll
    for (int u = 0; u < 4; u++) {
      const int64_t ri = i0 + u * 16 + ty;
      const int64_t i = ri < p.n_rows ? (p.rows ? p.rows[ri] : ri) : -1;
#pragma unroll
      for (int v = 0; v < 4; v++) {
        const int64_t j = j0 + v * 16 + tx;
        double d = 0.;
        if (i >= 0 && j < p.S2 && j > i) {
          const double stat = pair_stat<STAT>(p, i, j, acc[u][v]);
          d = p.dist_is_stat ? stat : p.dist_comp - stat;
          p.mat[(size_t)i * p.S + j] = d;
        }
        T[v * 16 + tx][ty] = d;
      }
      __syncthreads();
      const int64_t mri = i0 + u * 16 + c;
      const int64_t mi = mri < p.n_rows ? (p.rows ? p.rows[mri] : mri) : -1;
#pragma unroll
      for (int rr = 0; rr < 4; rr++) {
        const int64_t j = j0 + rr * 16 + r;
        if (mi >= 0 && j < p.S2 && j > mi) p.mat[(size_t)j * p.S + mi] = T[rr * 16 + r][c];
      }
      __syncthreads();
    }
    if (t.x == t.y) { // zero diagonal
      for (int d = tid; d < TS; d += blockDim.x) {
        int64_t i = i0 + d;
        if (i < p.S) p.mat[(size_t)i * p.S + i] = 0.;
      }
    }
    return;
  }
  const bool want_pv = p.K > 0 && (p.o_pvalue || p.o_nsim);
#pragma unroll
  for (int u = 0; u < 4; u++) {
    const int64_t ri = i0 + u * 16 + ty;
    if (ri >= p.n_rows) continue;
    const int64_t i = p.rows ? p.rows[ri] : ri;
    bool valid[4];
    int64_t idx[4];
    double st[4], nm[4];
#pragma unroll
    for (int v = 0; v < 4; v++) {
      const int64_t j = j0 + v * 16 + tx;
      valid[v] = !(j >= p.S2 || (p.mode != MODE_RECT && j <= i));
      idx[v] = 0; st[v] = nm[v] = 0.;
      if (valid[v]) pair_epilogue<STAT, true>(p, ri, i, j, acc[u][v], &idx[v], &st[v], &nm[v]);
    }
    if (want_pv) pvalues_interleaved<4>(p, valid, idx, st, nm);
  }
}

// independant comparisons (CoETools.cpp:795-796): row i pairs site i of data set 1 with site i of
// data set 2; statistic and Nmin come from k2_paired, this fills the other columns and the filters
__global__ void k2_diag_rows(TileParams p) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= p.S) return;
  const int ci = p.rate_class[i], cj = p.rate_class2[i];
  const double pi_ = p.post_rate[i], pj = p.post_rate2[i];
  const double stat = p.o_stat[i];
  if (p.any_filter) {
    bool keep = ci >= p.min_rate_class && cj >= p.min_rate_class2 && !(pi_ < p.min_rate) && !(pj < p.min_rate2);
    if (p.max_rate_class_diff >= 0 && abs(cj - ci) > p.max_rate_class_diff) keep = false;
    if (p.max_rate_diff >= 0. && fabs(pj - pi_) > p.max_rate_diff) keep = false;
    if (fabs(stat) < p.min_stat) keep = false;
    p.o_keep[i] = keep ? 1 : 0;
  }
  p.o_i[i] = (int32_t)i;
  p.o_j[i] = (int32_t)i;
  p.o_rcmin[i] = ci < cj ? ci : cj;
  p.o_prmin[i] = pi_ < pj ? pi_ : pj;
}

// p-value columns from the resident Stat / Nmin columns (same epilogue as k2_tiles): used when
// the null-independent columns were scored before the null existed, so the Gram tiles are not
// recomputed for PValue / Nsim
__global__ void k2_pvalues(int64_t n, const double* __restrict__ stat, const double* __restrict__ nmin, int K, double nmax,
                           const int64_t* __restrict__ bin_off, const double* __restrict__ sorted, double* __restrict__ pvalue,
                           int32_t* __restrict__ nsim_out) {
  const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= n) return;
  const double st = stat[r];
  const int cat = domain_index(nmax, K, nmin[r]);
  double pv = nan("");
  int64_t nsim = 0;
  if (cat >= 0) {
    const double* sim = sorted + bin_off[cat];
    nsim = bin_off[cat + 1] - bin_off[cat];
    int64_t lo = 0, hi = nsim; // count = #{sim < stat} on the ascending bin
    while (lo < hi) {
      int64_t mid = (lo + hi) >> 1;
      if (sim[mid] < st) lo = mid + 1; else hi = mid;
    }
    pv = (double)(nsim - lo + 1) / (double)(nsim + 1);
  }
  if (pvalue) pvalue[r] = pv;
  if (nsim_out) nsim_out[r] = (int32_t)nsim;
}

template <class T>
__global__ void k2_compact(int64_t n, const uint8_t* keep, const int64_t* pos, const T* src, T* dst) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n && keep[i]) dst[pos[i]] = src[i];
}
__global__ void k2_keep_to_i64(int64_t n, const uint8_t* keep, int64_t* out) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = keep[i];
}

} // namespace

void launch_paired(int stat_id, double thr, int B, int64_t n, int64_t n_pad, int64_t n_pad2, const double* o1, const double* o2,
                   const double* mv, const double* mv2, double* stat, double* nmin, cudaStream_t st, const int32_t* col1,
                   const int32_t* col2) {
  const unsigned g = (unsigned)((n + 127) / 128);
  switch (stat_id) { // the statistic is a template parameter: no per-branch dispatch in the inner loops
    case 0: k2_paired<0><<<g, 128, 0, st>>>(thr, B, n, n_pad, n_pad2, o1, o2, mv, mv2, stat, nmin, col1, col2); break;
    case 1: k2_paired<1><<<g, 128, 0, st>>>(thr, B, n, n_pad, n_pad2, o1, o2, mv, mv2, stat, nmin, col1, col2); break;
    case 2: k2_paired<2><<<g, 128, 0, st>>>(thr, B, n, n_pad, n_pad2, o1, o2, mv, mv2, stat, nmin, col1, col2); break;
    case 3: k2_paired<3><<<g, 128, 0, st>>>(thr, B, n, n_pad, n_pad2, o1, o2, mv, mv2, stat, nmin, col1, col2); break;
    case 4: k2_paired<4><<<g, 128, 0, st>>>(thr, B, n, n_pad, n_pad2, o1, o2, mv, mv2, stat, nmin, col1, col2); break;
    case 6: k2_paired<6><<<g, 128, 0, st>>>(thr, B, n, n_pad, n_pad2, o1, o2, mv, mv2, stat, nmin, col1, col2); break;
    case 7: k2_paired<7><<<g, 128, 0, st>>>(thr, B, n, n_pad, n_pad2, o1, o2, mv, mv2, stat, nmin, col1, col2); break;
    default: fail("unknown statistic id %d", stat_id);
  }
  CMB_CUDA(cudaGetLastError());
}
void launch_pair_list(int stat_id, double thr, int B, int64_t n_pad, const double* out, const double* mv, const int2* pairs,
                      int64_t n_pairs, double* stat, cudaStream_t st) {
  if (n_pairs == 0) return;
  k2_pair_list<<<(unsigned)((n_pairs + 127) / 128), 128, 0, st>>>(stat_id, thr, B, n_pad, out, mv, pairs, n_pairs, stat);
  CMB_CUDA(cudaGetLastError());
}
ColumnKeys column_key_buffers(int T, int64_t n, int64_t n_pad, DevBuf& tmp) {
  if (n_pad > 0x7fffffff) fail("internal: batch too large for 32-bit column indices");
  const int m = (int)(2 * n);
  size_t sort_bytes = 0, max_bytes = 0, sum_bytes = 0;
  cub::DeviceRadixSort::SortPairs(nullptr, sort_bytes, (const uint64_t*)nullptr, (uint64_t*)nullptr, (const int32_t*)nullptr,
                                  (int32_t*)nullptr, m, 0, 64);
  cub::DeviceScan::InclusiveScan(nullptr, max_bytes, (const int32_t*)nullptr, (int32_t*)nullptr, cuda::maximum<int32_t>(), m);
  cub::DeviceScan::ExclusiveSum(nullptr, sum_bytes, (const int64_t*)nullptr, (int64_t*)nullptr, (int)n_pad);
  const size_t a8 = align256(8 * (size_t)m), a4 = align256(4 * (size_t)m), c4 = align256(4 * (size_t)n_pad);
  const size_t c8 = align256(8 * (size_t)n_pad);
  const size_t pk = align256(4 * (size_t)((T + 15) / 16) * n_pad);
  ColumnKeys k;
  k.cub_bytes = std::max(sort_bytes, std::max(max_bytes, sum_bytes));
  tmp.reserve(2 * a8 + 2 * a4 + pk + c4 + 2 * c8 + k.cub_bytes);
  unsigned char* p = tmp.as<unsigned char>();
  k.hash = (uint64_t*)p; p += a8;
  k.hash_sorted = (uint64_t*)p; p += a8;
  k.col = (int32_t*)p; p += a4;
  k.col_sorted = (int32_t*)p; p += a4;
  k.packed = (uint32_t*)p; p += pk;
  k.rep = (int32_t*)p; p += c4;
  k.val = (int64_t*)p; p += c8;
  k.pos = (int64_t*)p; p += c8;
  k.cub_tmp = p;
  return k;
}
int launch_compress_patterns(int T, int64_t n, int64_t half, int64_t n_pad, const uint8_t* tips, const int32_t* leaf_rows,
                             bool keyed, int hash_bits, int min_run, const ColumnKeys& k, uint8_t* tips_c, int32_t* col,
                             int32_t* count, cudaStream_t st) {
  if (hash_bits < 1 || hash_bits > 64) fail("internal: %d hash bits", hash_bits);
  if (min_run < 2) fail("internal: runs of %d columns", min_run);
  const int64_t m = 2 * n;
  const unsigned gm = (unsigned)((m + 255) / 256), g = (unsigned)((n_pad + 255) / 256);
  int nl = 7; // the sort and the scans counted once each
  if (!keyed) {
    k2_column_keys<<<gm, 256, 0, st>>>(T, n, half, n_pad, tips, leaf_rows, k.hash, k.col, k.packed);
    nl++;
  }
  size_t bytes = k.cub_bytes;
  CMB_CUDA(cub::DeviceRadixSort::SortPairs(k.cub_tmp, bytes, k.hash, k.hash_sorted, k.col, k.col_sorted, (int)m, 0, hash_bits, st));
  int32_t* start = reinterpret_cast<int32_t*>(k.hash); // the unsorted hashes are spent
  k2_run_starts<<<gm, 256, 0, st>>>(m, k.hash_sorted, hash_bits == 64 ? ~0ull : (1ull << hash_bits) - 1, start);
  bytes = k.cub_bytes;
  int32_t* run_start = reinterpret_cast<int32_t*>(k.pos);
  CMB_CUDA(cub::DeviceScan::InclusiveScan(k.cub_tmp, bytes, start, run_start, cuda::maximum<int32_t>(), (int)m, st));
  k2_run_heads<<<gm, 256, 0, st>>>(m, min_run, run_start, k.col_sorted, k.rep);
  k2_pick_representatives<<<g, 256, 0, st>>>((T + 15) / 16, n, half, n_pad, k.packed, k.rep, k.val);
  bytes = k.cub_bytes;
  CMB_CUDA(cub::DeviceScan::ExclusiveSum(k.cub_tmp, bytes, k.val, k.pos, (int)n_pad, st));
  k2_compact_columns<<<g, 256, 0, st>>>(T, n, half, n_pad, tips, k.rep, k.val, k.pos, tips_c, col, count);
  CMB_CUDA(cudaGetLastError());
  return nl;
}

void launch_raw_rows(int64_t n, const double* stat, const double* nmin, const int32_t* rc1, const int32_t* rc2,
                     const double* pr1, const double* pr2, double* raw, cudaStream_t st, const int32_t* col1,
                     const int32_t* col2) {
  k2_raw_rows<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(n, stat, nmin, rc1, rc2, pr1, pr2, raw, col1, col2);
  CMB_CUDA(cudaGetLastError());
}
void launch_prep(int B, int64_t n, int64_t n_pad, const double* out, const double* mv, double* mean, double* sd,
                 double* norm, cudaStream_t st) {
  k2_prep<<<(unsigned)((n + 127) / 128), 128, 0, st>>>(B, n, n_pad, out, mv, mean, sd, norm);
  CMB_CUDA(cudaGetLastError());
}
void launch_count_ge(int B, int64_t n, int64_t n_pad, const double* out, double thr, double* cnt, cudaStream_t st) {
  k2_count_ge<<<(unsigned)((n + 127) / 128), 128, 0, st>>>(B, n, n_pad, out, thr, cnt);
  CMB_CUDA(cudaGetLastError());
}
void launch_mean_vector(int B, int64_t S, int64_t n_pad, const double* out, double* mv, cudaStream_t st) {
  k2_mean_vector<<<(unsigned)((B + 127) / 128), 128, 0, st>>>(B, S, n_pad, out, mv);
  CMB_CUDA(cudaGetLastError());
}

// Bins the n samples by Nmin and sorts each bin ascending.  sorted gets the retained
// samples grouped by bin; off (K+1 int64, device) the bin boundaries.  Returns launches.
int bin_and_sort(int64_t n, const double* stat, const double* nmin, int K, double nmax, DevBuf& tmp,
                 double* sorted, int64_t* off_dev, cudaStream_t st) {
  if (n == 0) {
    CMB_CUDA(cudaMemsetAsync(off_dev, 0, sizeof(int64_t) * (K + 1), st));
    return 0;
  }
  // layout of tmp: cat[n] u32 | cat2[n] u32 | stat1[n] f64 | cub temp
  size_t need1 = 0, need2 = 0;
  cub::DeviceRadixSort::SortPairs(nullptr, need1, (const double*)nullptr, (double*)nullptr, (const uint32_t*)nullptr,
                                  (uint32_t*)nullptr, (int)n, 0, 64, st);
  cub::DeviceRadixSort::SortPairs(nullptr, need2, (const uint32_t*)nullptr, (uint32_t*)nullptr, (const double*)nullptr,
                                  (double*)nullptr, (int)n, 0, 32, st);
  size_t need = need1 > need2 ? need1 : need2;
  size_t a = align256((size_t)n * 4), d = align256((size_t)n * 8);
  tmp.reserve(2 * a + d + need + 256);
  unsigned char* base = tmp.as<unsigned char>();
  uint32_t* cat = (uint32_t*)base;
  uint32_t* cat2 = (uint32_t*)(base + a);
  double* stat1 = (double*)(base + 2 * a);
  void* ctemp = base + 2 * a + d;
  k2_bin_keys<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(n, nmin, nmax, K, cat);
  CMB_CUDA(cudaGetLastError());
  // sort by statistic, then stable sort by bin
  CMB_CUDA(cub::DeviceRadixSort::SortPairs(ctemp, need, stat, stat1, cat, cat2, (int)n, 0, 64, st));
  int bits = 1;
  while ((1 << bits) <= K) bits++;
  CMB_CUDA(cub::DeviceRadixSort::SortPairs(ctemp, need, cat2, cat, stat1, sorted, (int)n, 0, bits, st));
  k2_bin_offsets<<<(unsigned)((K + 1 + 63) / 64), 64, 0, st>>>(n, cat, K, off_dev);
  CMB_CUDA(cudaGetLastError());
  return 6;
}

int launch_tiles(const TilesLaunch& L, cudaStream_t st) {
  TileParams p{};
  p.stat_id = L.stat_id; p.mode = L.dist_mode ? MODE_DIST : MODE_PAIRS; p.B = L.B; p.S = L.S; p.S_pad = L.S_pad;
  p.out = L.out; p.mean = L.mean; p.sd = L.sd; p.norm = L.norm; p.post_rate = L.post_rate; p.rate_class = L.rate_class;
  p.mv = L.mv;
  const bool rect = L.out2 != nullptr;
  if (rect) p.mode = MODE_RECT;
  p.S2 = rect ? L.S2 : L.S; p.S2_pad = rect ? L.S2_pad : L.S_pad; p.out2 = rect ? L.out2 : L.out;
  p.mean2 = rect ? L.mean2 : L.mean; p.sd2 = rect ? L.sd2 : L.sd; p.norm2 = rect ? L.norm2 : L.norm;
  p.post_rate2 = rect ? L.post_rate2 : L.post_rate; p.rate_class2 = rect ? L.rate_class2 : L.rate_class;
  p.mv2 = rect ? L.mv2 : L.mv;
  p.min_rate_class2 = rect ? L.min_rate_class2 : L.min_rate_class; p.min_rate2 = rect ? L.min_rate2 : L.min_rate;
  p.nmin_by_row = rect ? L.nmin_by_row : 0;
  p.thr = L.thr;
  p.tiles = L.tiles; p.rows = L.rows; p.n_rows = L.n_rows; p.row_off = L.row_off;
  p.min_rate_class = L.min_rate_class; p.max_rate_class_diff = L.max_rate_class_diff; p.min_rate = L.min_rate;
  p.max_rate_diff = L.max_rate_diff; p.min_stat = L.min_stat; p.any_filter = L.any_filter;
  p.K = L.K; p.nmax = L.nmax; p.bin_off = L.bin_off; p.sorted = L.sorted;
  p.o_i = L.o_i; p.o_j = L.o_j; p.o_rcmin = L.o_rcmin; p.o_stat = L.o_stat; p.o_prmin = L.o_prmin; p.o_nmin = L.o_nmin;
  p.o_pvalue = L.o_pvalue; p.o_nsim = L.o_nsim; p.o_keep = L.o_keep; p.mat = L.mat; p.dist_comp = L.dist_comp;
  p.dist_is_stat = L.dist_is_stat;
  if (L.n_tiles == 0) return 0;
  unsigned g = (unsigned)L.n_tiles;
  switch (L.stat_id) {
    case 0: k2_tiles<0><<<g, 256, 0, st>>>(p); break;
    case 1: k2_tiles<1><<<g, 256, 0, st>>>(p); break;
    case 2: k2_tiles<2><<<g, 256, 0, st>>>(p); break;
    case 3: k2_tiles<3><<<g, 256, 0, st>>>(p); break;
    case 4: k2_tiles<4><<<g, 256, 0, st>>>(p); break;
    case 5: k2_tiles<5><<<g, 256, 0, st>>>(p); break;
    case 6: k2_tiles<6><<<g, 256, 0, st>>>(p); break;
    case 7: k2_tiles<7><<<g, 256, 0, st>>>(p); break;
    default: fail("unknown statistic id %d", L.stat_id);
  }
  CMB_CUDA(cudaGetLastError());
  return 1;
}

void launch_pvalues(int64_t n, const double* stat, const double* nmin, int K, double nmax, const int64_t* bin_off,
                    const double* sorted, double* pvalue, int32_t* nsim, cudaStream_t st) {
  if (n == 0) return;
  k2_pvalues<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(n, stat, nmin, K, nmax, bin_off, sorted, pvalue, nsim);
  CMB_CUDA(cudaGetLastError());
}

int launch_inter_diagonal(const TilesLaunch& L, cudaStream_t st) {
  if (!L.out2 || L.S != L.S2) fail("internal: diagonal comparison needs two data sets of the same length");
  if (L.S == 0) return 0;
  TileParams p{};
  p.S = L.S; p.rate_class = L.rate_class; p.rate_class2 = L.rate_class2; p.post_rate = L.post_rate; p.post_rate2 = L.post_rate2;
  p.min_rate_class = L.min_rate_class; p.min_rate_class2 = L.min_rate_class2; p.min_rate = L.min_rate; p.min_rate2 = L.min_rate2;
  p.max_rate_class_diff = L.max_rate_class_diff; p.max_rate_diff = L.max_rate_diff; p.min_stat = L.min_stat;
  p.any_filter = L.any_filter;
  p.o_i = L.o_i; p.o_j = L.o_j; p.o_stat = L.o_stat; p.o_rcmin = L.o_rcmin; p.o_prmin = L.o_prmin; p.o_keep = L.o_keep;
  launch_paired(L.stat_id, L.thr, L.B, L.S, L.S_pad, L.S2_pad, L.out, L.out2, L.mv, L.mv2, L.o_stat, L.o_nmin, st);
  k2_diag_rows<<<(unsigned)((L.S + 127) / 128), 128, 0, st>>>(p);
  CMB_CUDA(cudaGetLastError());
  return 2;
}

// exclusive scan of the keep flags -> positions; returns number kept (synchronises)
int64_t compact_positions(int64_t n, const uint8_t* keep, DevBuf& tmp, int64_t** pos_out, cudaStream_t st) {
  size_t need = 0;
  cub::DeviceScan::ExclusiveSum(nullptr, need, (const int64_t*)nullptr, (int64_t*)nullptr, (int)n, st);
  size_t a = align256((size_t)n * 8);
  tmp.reserve(2 * a + need + 256);
  int64_t* flags = tmp.as<int64_t>();
  int64_t* pos = (int64_t*)(tmp.as<unsigned char>() + a);
  void* ctemp = tmp.as<unsigned char>() + 2 * a;
  k2_keep_to_i64<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(n, keep, flags);
  CMB_CUDA(cub::DeviceScan::ExclusiveSum(ctemp, need, flags, pos, (int)n, st));
  int64_t last_pos = 0, last_flag = 0;
  CMB_CUDA(cudaMemcpyAsync(&last_pos, pos + n - 1, 8, cudaMemcpyDeviceToHost, st));
  CMB_CUDA(cudaMemcpyAsync(&last_flag, flags + n - 1, 8, cudaMemcpyDeviceToHost, st));
  CMB_CUDA(cudaStreamSynchronize(st));
  *pos_out = pos;
  return last_pos + last_flag;
}
template <class T>
void compact_column(int64_t n, const uint8_t* keep, const int64_t* pos, const T* src, T* dst, cudaStream_t st) {
  k2_compact<T><<<(unsigned)((n + 255) / 256), 256, 0, st>>>(n, keep, pos, src, dst);
  CMB_CUDA(cudaGetLastError());
}
template void compact_column<int32_t>(int64_t, const uint8_t*, const int64_t*, const int32_t*, int32_t*, cudaStream_t);
template void compact_column<int64_t>(int64_t, const uint8_t*, const int64_t*, const int64_t*, int64_t*, cudaStream_t);
template void compact_column<double>(int64_t, const uint8_t*, const int64_t*, const double*, double*, cudaStream_t);

} // namespace cmb
