// Launch interfaces of the CUDA kernels (implemented in k*.cu).
#pragma once
#include "common.h"

namespace cmb {

struct DevStream {           // an OpStream uploaded to the device
  DevBuf bytes, off, nbytes, nrec, aux;
  uint32_t n_chunks = 0, cap = 0, n_records = 0;
  int stack_depth = 0;
  uint32_t stage_bytes = 0;
  uint32_t blk_off_max[3] = {0, 0, 0};
  void upload(const OpStream& s, cudaStream_t st);
};

struct ChunkMeta {           // kernel-side view of a DevStream
  const unsigned char* src;
  const uint32_t *off, *bytes, *nrec;
  uint32_t n_chunks, cap;
};
inline ChunkMeta meta_of(const DevStream& s) {
  return ChunkMeta{s.bytes.as<unsigned char>(), s.off.as<uint32_t>(), s.nbytes.as<uint32_t>(),
                   s.nrec.as<uint32_t>(), s.n_chunks, s.cap};
}

struct MapBuffers {          // per-batch device arrays, n_pad sites (multiple of 256)
  int64_t n = 0, n_pad = 0;
  const uint8_t* tips = nullptr;   // [T][n_pad]
  double* D = nullptr;             // A = 20: [n_pad/256][n_slots][C*A][256] (k1_map.cu d_block);
                                   // A = 4:  [n_pad/128][n_slots][C][128][4] (k1_mma.cu d_chunk)
  double* Lc = nullptr;            // [C][n_pad]
  double* invL = nullptr;          // [n_pad]
  double* loglik = nullptr;        // [n_pad]
  double* post_rate = nullptr;     // [n_pad]
  int32_t* rate_class = nullptr;   // [n_pad]
  double* out = nullptr;           // [B][n_pad]
  const int32_t* n_active = nullptr; // device scalar: only sites [0, *n_active) are mapped (nullptr: all n_pad); A = 4 kernels
};

struct MapModel {            // device-resident model constants
  int A = 0, C = 0, B = 0, n_slots = 0, T = 0; // T = leaves (rows of the alignment)
  const uint32_t* code_mask = nullptr; // [256]
  int states_only = 0;                 // tips hold resolved state indices 0..A-1 (device simulator output)
  const double* pi = nullptr;          // [A]
  const double* rates = nullptr;       // [C]
  const double* probs = nullptr;       // [C]
  // continuous-rate simulation (cmb_set_continuous_rates): 0 = discrete classes
  int cont_kind = 0;
  double cont_alpha = 1., cont_pinv = 0.;
  const double* spec = nullptr;        // device: ev[A] | R[A][A] | L[A][A] | brlen[n_nodes]  (Q = R diag(ev) L)
};

void check_map_support(int A, int C); // throws when no kernel is built for (A, C)
void launch_map_down(const MapModel& m, const MapBuffers& b, const DevStream& s, cudaStream_t st);
void launch_map_finish(const MapModel& m, const MapBuffers& b, cudaStream_t st);
// cb > 0: only classes [c0, c0 + cb) of the m.C, from an up stream built for them (build_up_stream(.., c0, cb));
// the first block writes b.out, later ones add to it.  Scalar protein kernels only, cb <= kScalarUpClasses.
constexpr int kScalarUpClasses = 4;
void launch_map_up(const MapModel& m, const MapBuffers& b, const DevStream& s, cudaStream_t st, int c0 = 0, int cb = 0);
// A = 4: tensor-core up pass (k1_mma.cu); the stream is build_up_mma_stream's
void launch_map_up_mma(const MapModel& m, const MapBuffers& b, const DevStream& s, cudaStream_t st);
void launch_map_down_mma(const MapModel& m, const MapBuffers& b, const DevStream& s, cudaStream_t st);
// A = 20: tensor-core passes (k1_mma20.cu); the streams are build_*_mma20_stream's; part: [C][B][n_pad] scratch.
// false = no launch shape fits (the caller reports it)
bool launch_map_down_mma20(const MapModel& m, const MapBuffers& b, const DevStream& s, cudaStream_t st);
bool launch_map_up_mma20(const MapModel& m, const MapBuffers& b, const DevStream& s, double* part, cudaStream_t st);
// nijt.average = no / nijt.joint = no (k1_variants.cu): thread-per-site walk of the original tree
struct VariantTables {
  int n_nodes = 0;
  const int32_t *parent = nullptr, *ch_off = nullptr, *ch = nullptr, *leaf_row = nullptr;
  const double *P = nullptr, *N = nullptr; // [branch][C][A][A]
};
// mode 1 marginal, 2 no averaging, 3 no averaging + marginal states; overwrites b.out for sites [0, b.n); returns launches
// mode 4: only the marginal state of every node into states_out [n_nodes][n_pad] (asr.method = marginal); b.out untouched
int launch_map_variant(const MapModel& m, const MapBuffers& b, const VariantTables& vt, int mode, DevBuf& scratch, cudaStream_t st,
                       uint8_t* states_out = nullptr);
// A = 4 partial layout: 128-site chunks (common.h kChunkSites), [chunk][slot][class][site][state]
__host__ __device__ inline size_t d_chunk(int64_t chunk, int slot, int n_slots, int C) {
  return ((size_t)chunk * n_slots + slot) * ((size_t)C * kChunkSites * 4);
}

// site id of thread idx = base + (idx / group) * stride + idx % group
void launch_simulate(const MapModel& m, const DevStream& s, uint64_t seed, int64_t base, int64_t group,
                     int64_t stride, int64_t n, int64_t n_pad, int weighted, int root_node, uint8_t* tips,
                     int32_t* classes, cudaStream_t st, int64_t half_n = 0, int64_t half_col = 0, int64_t half_shift = 0,
                     int32_t* col_class = nullptr, int32_t* col_varied = nullptr);

// ---- K5: Mica's column statistics (k5_mica.cu)
void launch_mica_entropy(int A, int T, int64_t n, int64_t n_pad, const uint8_t* tips, const uint32_t* cmask, double* entropy,
                         cudaStream_t st);
void launch_mica_pairs(int A, int T, int64_t S, int64_t n_pad, const uint8_t* tips, const uint32_t* cmask, double* mi, double* hj,
                       cudaStream_t st);
// site a[r] of tip matrix t1 against site b[r] of t2 (a / b nullptr: r itself)
void launch_mica_listed(int A, int T, int64_t n, const uint8_t* t1, int64_t np1, const uint8_t* t2, int64_t np2, const int32_t* a,
                        const int32_t* b, const uint32_t* cmask, double* mi, double* hj, cudaStream_t st);
void launch_mica_permutations(int A, int T, int64_t S, int64_t n_pad, const uint8_t* tips, const uint32_t* cmask, uint64_t seed,
                              int max_perm, unsigned long long* next, double* pvalue, int32_t* nperm, cudaStream_t st);
void launch_mica_average(int64_t S, const double* mi, double* avg, cudaStream_t st);
void launch_mica_rows(int64_t S, const double* entropy, const double* norm, int32_t* oi, int32_t* oj, double* hmin, double* nmin,
                      cudaStream_t st);
void launch_min2(int64_t n, const double* a, const double* b, double* out, cudaStream_t st);

// ---- K2
// mv: mean vector subtracted before a correlation (corrected correlation) or nullptr
// col1 / col2 (nullable): column of pair j's first / second site in o1 / o2 (pattern-compressed mappings); else j
void launch_paired(int stat_id, double thr, int B, int64_t n, int64_t n_pad, int64_t n_pad2, const double* o1, const double* o2,
                   const double* mv, const double* mv2, double* stat, double* nmin, cudaStream_t st,
                   const int32_t* col1 = nullptr, const int32_t* col2 = nullptr);
// Pattern compression of a simulated alignment (what Bio++ does through its distinct-site patterns): columns whose
// tips all carry the same state are mapped ONCE per state.  cls[site] = state or -1 (varied) for the sites of
// the two batches [0, n) and [half, half + n); tips_c receives the varied columns packed from 0 and the A constant
// patterns after them; col[site] = where the site's vector will be; counts[0] = sites to map (varied + A),
// counts[1] = varied sites.  tmp: scan scratch.
// classified: the simulator already wrote the class / varied flag of every simulated column (compress_class_buffers of
// the same tmp and n_pad handed to launch_simulate); only the columns outside the two batches are filled in here
int launch_compress_constant(int A, int T, int64_t n, int64_t half, int64_t n_pad, const uint8_t* tips, uint8_t* tips_c,
                             int32_t* col, int32_t* counts, DevBuf& tmp, cudaStream_t st, bool classified = false);
void compress_class_buffers(int64_t n_pad, DevBuf& tmp, int32_t** col_class, int32_t** col_varied);
// statistic of listed column pairs of one [B][n_pad] matrix (candidate-group statistics)
void launch_pair_list(int stat_id, double thr, int B, int64_t n_pad, const double* out, const double* mv, const int2* pairs,
                      int64_t n_pairs, double* stat, cudaStream_t st);
void launch_count_ge(int B, int64_t n, int64_t n_pad, const double* out, double thr, double* cnt, cudaStream_t st);
void launch_mean_vector(int B, int64_t S, int64_t n_pad, const double* out, double* mv, cudaStream_t st);
void launch_raw_rows(int64_t n, const double* stat, const double* nmin, const int32_t* rc1, const int32_t* rc2,
                     const double* pr1, const double* pr2, double* raw, cudaStream_t st,
                     const int32_t* col1 = nullptr, const int32_t* col2 = nullptr);
void launch_prep(int B, int64_t n, int64_t n_pad, const double* out, const double* mv, double* mean, double* sd,
                 double* norm, cudaStream_t st);
int bin_and_sort(int64_t n, const double* stat, const double* nmin, int K, double nmax, DevBuf& tmp,
                 double* sorted, int64_t* off_dev, cudaStream_t st);

struct TilesLaunch {
  int stat_id = 0, B = 0;       // stat ids 0..4 as in the C ABI, 5 = euclidian distance
  bool dist_mode = false;
  int64_t S = 0, S_pad = 0;
  const double* out = nullptr;
  const double *mean = nullptr, *sd = nullptr, *norm = nullptr, *post_rate = nullptr;
  const double* mv = nullptr;   // mean vector (corrected correlation)
  // two data sets (rectangle S x S2): column operand and its per-site arrays; nullptr = one data set
  const double *out2 = nullptr, *mean2 = nullptr, *sd2 = nullptr, *norm2 = nullptr, *post_rate2 = nullptr, *mv2 = nullptr;
  const int32_t* rate_class2 = nullptr;
  int64_t S2 = 0, S2_pad = 0;
  int min_rate_class2 = 0, nmin_by_row = 0;
  double thr = 0.;              // MI threshold (stat 6; `mean` / `mean2` then hold the category-1 counts)
  double min_rate2 = 0.;
  const int32_t* rate_class = nullptr;
  const int2* tiles = nullptr;
  int64_t n_tiles = 0;
  const int32_t* rows = nullptr;
  int64_t n_rows = 0;
  const int64_t* row_off = nullptr;
  int min_rate_class = 0, max_rate_class_diff = -1;
  double min_rate = 0., max_rate_diff = -1., min_stat = 0.;
  int any_filter = 0;
  int K = 0;
  double nmax = 0.;
  const int64_t* bin_off = nullptr;
  const double* sorted = nullptr;
  int32_t *o_i = nullptr, *o_j = nullptr, *o_rcmin = nullptr;
  double *o_stat = nullptr, *o_prmin = nullptr, *o_nmin = nullptr, *o_pvalue = nullptr;
  int32_t* o_nsim = nullptr;
  uint8_t* o_keep = nullptr;
  double* mat = nullptr;
  double dist_comp = 1.;
  int dist_is_stat = 0;
};
int launch_tiles(const TilesLaunch& L, cudaStream_t st);
// PValue / Nsim of rows whose Stat / Nmin columns are already resident (no tile recomputation)
void launch_pvalues(int64_t n, const double* stat, const double* nmin, int K, double nmax, const int64_t* bin_off,
                    const double* sorted, double* pvalue, int32_t* nsim, cudaStream_t st);
int launch_inter_diagonal(const TilesLaunch& L, cudaStream_t st); // site i of data set 1 with site i of data set 2
int64_t compact_positions(int64_t n, const uint8_t* keep, DevBuf& tmp, int64_t** pos_out, cudaStream_t st);
template <class T>
void compact_column(int64_t n, const uint8_t* keep, const int64_t* pos, const T* src, T* dst, cudaStream_t st);

// [B][n_pad] -> [n][B] for the host-facing site-major output
// (dst_stride: row stride of dst, default B; the same kernel loads a site-major matrix into the
// [B][n_pad] layout by swapping the roles of the two dimensions)
void launch_transpose_out(const double* out, int B, int64_t n, int64_t n_pad, double* dst, cudaStream_t st,
                          int64_t dst_stride = 0);


// ---- K4
int launch_cluster_batch(int np, int64_t S, int linkage, double* const* mats, DevBuf* works, int32_t* const* left_dev,
                         int32_t* const* right_dev, double* const* height_dev, cudaStream_t st);
int launch_cluster(int64_t S, int linkage, double* mat, DevBuf& work, int32_t* left_dev, int32_t* right_dev,
                   double* height_dev, cudaStream_t st);
// large matrices, complete / average linkage: rounds of reciprocal nearest neighbours (k4_rnn.cu)
bool cluster_rnn_selected(int64_t S, int linkage);
int launch_cluster_rnn(int64_t S, int linkage, double* mat, DevBuf& work, int32_t* left_dev, int32_t* right_dev,
                       double* height_dev, cudaStream_t st);
void launch_group_compensation(int64_t n_groups, const int32_t* members, const int64_t* offsets, int B,
                               int64_t S_pad, const double* out, double* stat, cudaStream_t st);

} // namespace cmb
