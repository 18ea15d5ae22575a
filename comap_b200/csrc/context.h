// The context object behind cmb_ctx: one GPU, one stream, device arenas; and the scaffolding every C ABI
// entry point shares (error capture, statistic ids).
#pragma once
#include "../../include/comap_b200.h"
#include "kernels.h"
#include <algorithm>
#include <memory>

namespace cmb {

struct Profile {
  struct Entry { double ms = 0.; int64_t launches = 0; };
  std::map<std::string, Entry> entries;
  std::vector<std::tuple<std::string, cudaEvent_t, cudaEvent_t, int>> pending;
  bool enabled = false;
  int64_t total_launches = 0;
  int64_t sites_simulated = 0;   // simulated sites handed to the null's mapping
};

struct NullState {            // binned, sorted null distribution (device + host mirror)
  int K = 0;
  double nmax = 0.;
  int64_t n_samples = 0;      // unbinned samples held in stat/nmin
  DevBuf stat, nmin;          // [n_samples] raw samples of this shard
  DevBuf sorted;              // [bin_off[K]] ascending within each bin
  DevBuf bin_off_dev;         // int64 [K+1]
  std::vector<int64_t> bin_off;
  bool ready = false;
  bool nmax_from_map = false;  // nmax was taken from the mapped alignment's max(norm) (nmax < 0 at load time)
  void begin(int64_t n) {     // a new arena of n raw samples; the binned distribution is stale
    ready = false;
    stat.reserve(sizeof(double) * (size_t)std::max<int64_t>(n, 1));
    nmin.reserve(sizeof(double) * (size_t)std::max<int64_t>(n, 1));
    n_samples = n;
  }
};

struct Context {
  int device = 0;
  cudaStream_t stream = nullptr;
  bool own_stream = false;

  Tree tree;
  bool have_tree = false;
  ModelTables tables;
  bool have_model = false;
  // model inputs kept to rebuild tables when the tree changes
  std::vector<double> Q, pi, rates, probs, weights;
  int A = 0, C = 0, count_method = 0;
  bool have_weights = false;

  // device-resident model + op streams
  DevBuf d_code_mask, d_pi, d_rates, d_probs;
  DevStream down_stream, up_stream, sim_stream;
  DevBuf d_leaf_walk;            // int32 [T]: alignment row of the j-th leaf the simulation walk reaches (column keys)
  DevStream up_stream_hi; // scalar protein up pass above kScalarUpClasses classes: classes [kScalarUpClasses, C)
  int cont_kind = 0;             // continuous-rate simulation (cmb_set_continuous_rates)
  double cont_alpha = 1., cont_pinv = 0.;
  DevBuf d_spec;                 // ev | R | L | brlen for it
  bool streams_ready = false;
  bool protein_mma = false;      // A = 20 on the tensor-core kernels (k1_mma20.cu); else the thread-per-site ones
  DevBuf k1_part;                // their per-class partial outputs [C][B][n_pad]
  // nijt.average / nijt.joint (cmb_set_map_mode): 0 = average + joint (default), 1 marginal, 2 no averaging, 3 neither
  int map_mode = 0;
  DevBuf var_tree, var_tabs, var_scratch, var_scratch_obs;
  bool var_ready = false;
  VariantTables variant_tables(); // device copies of the original tree and of the P / count tables, built on first use

  // observed alignment + its mapping
  int64_t S = 0, S_pad = 0;
  DevBuf d_tips;                 // [T][S_pad]
  std::vector<uint32_t> code_mask;
  bool have_alignment = false, mapped = false;
  DevBuf d_D, d_Lc, d_invL, d_loglik, d_pr, d_rc, d_out;
  double *h_norm = nullptr, *h_loglik = nullptr; // pinned host copies [S] used by null / pairs / the saturation check
  size_t h_cap = 0;
  // cmb_map without host outputs is deferred: enqueued on a side stream so that what the caller enqueues next
  // (the null replicates) overlaps it -- a 5000-site mapping is one latency-bound tree walk on a few SMs
  cudaStream_t map_stream = nullptr;
  cudaEvent_t map_begin = nullptr, map_done = nullptr;
  bool map_pending = false;
  DevBuf k1_part_obs;            // per-class partial outputs of the observed alignment's protein mapping
  void cancel_map();             // block until a deferred mapping has left the device and drop it (no checks)
  void finish_map();             // ... and complete it: max norm, saturated sites (throws), ordering of the main stream
  void finalize_map_host();
  double max_norm = 0.;

  // scratch for simulated batches
  DevBuf s_tips[2], s_D, s_Lc, s_invL, s_loglik, s_pr[2], s_rc[2], s_out[2], s_cls;
  DevBuf d_identity_mask;
  DevBuf s_cols, s_counts;       // pattern compression of simulated batches: column of every site, columns to map per batch
  int s_batches = 0;
  int64_t null_budget_sites = 0;  // simulated sites the null may hold at once (from free memory, cached)
  const void* s_tips_ptr = nullptr;
  int64_t s_tips_pad = -1, s_tips_n = -1; // geometry the simulated tip buffer's padding columns were cleared for
  MapBuffers sim_buffers(int k, int64_t n, int64_t n_pad); // mapping buffers of n simulated sites, tips in s_tips[k]
  // s_tips[0] holds two batches of n sites at columns [0, n) and [half, half + n); the columns between and after them
  // are mapped too (their results are never read): give them a valid state once per buffer geometry
  void clear_sim_tip_padding(int64_t n, int64_t n_pad);

  NullState null;

  // clustering
  DevBuf d_dist;                 // [S][S]
  DevBuf dist_tiles;             // upper-triangle tile list of the distance kernel, cached per site count
  int64_t dist_tiles_S = -1, dist_tiles_n = 0;
  // clustering null: per-replicate matrices / vectors / work areas, kept between calls (a 20 000-site replicate
  // holds 3.2 GB; allocating and freeing four of them per call cost tens of ms)
  DevBuf cn_dists[4], cn_works[4], cn_outs[4], cn_mean, cn_sd, cn_norm, cn_staging;
  bool have_dist = false;
  int dist_id = 0;
  std::vector<int32_t> h_left, h_right;
  std::vector<double> h_height;
  bool have_dendro = false;

  DevBuf scratch, scratch2, staging;
  // Mica (capi_mica.cu): entropy [S_pad] | average MI [S_pad] | dense MI / Hjoint / Hmin / Nmin / PValue columns, i, j, Nsim
  DevBuf mica_sites, mica_table;
  bool mica_ready = false;       // the dense MI / Hjoint columns belong to the current alignment
  DevBuf pair_table;            // resident pair columns (fixed layout, see cmb_pairs_resident)
  cudaStream_t copy_stream = nullptr; // D2H of pair columns overlaps later kernels
  cudaEvent_t copy_event = nullptr;
  int64_t pairs_col_off[8] = {-1, -1, -1, -1, -1, -1, -1, -1}; // resident pair columns in `pair_table`
  int64_t pairs_rows = -1;
  void drop_pair_table() { pairs_rows = -1; for (auto& o : pairs_col_off) o = -1; }
  int pairs_stat_id = -1, pairs_shard_index = -1, pairs_shard_count = -1; // what the resident columns belong to
  DevBuf pairs_mean, pairs_sd, pairs_norm; // per-site mean / sd / norm for the tile kernels
  // corrected correlation (Statistics.h:176-205): mean vector of the mapped alignment and the
  // per-site mean / sd of the corrected vectors; built on first use after cmb_map
  DevBuf d_meanvec, corr_mean, corr_sd;
  bool have_meanvec = false;
  const double* mean_vector();  // device pointer [B]; computes it (and corr_mean / corr_sd) when stale
  // statistic=MI(threshold=..): per-site number of branches whose entry reaches the threshold
  double mi_threshold = 0.99;
  DevBuf mi_count;
  bool have_mi_count = false;
  const double* mi_counts();    // device pointer [S_pad] of the mapped alignment; built on first use
  // multi-GPU: NCCL communicator of this context's rank (comm.cpp); comm_size = 1 without one
  void* comm = nullptr;
  int comm_rank = 0, comm_size = 1;
  bool own_comm = false;
  DevBuf gather_send, gather_recv; // padded [stat | nmin] blocks of the null all-gather
  Profile prof;
  bool async_null = false; // cmb_set_async: cmb_null_intra with K = 0 returns without waiting for the device

  void require_tree_model() const;
  void ensure_streams();
  MapModel map_model() const;
  // maps n sites whose tips are at `tips` ([T][n_pad]); buffers given explicitly
  // simulated: codes are state indices (identity mask); states_only: ... and known to be < A
  // variants: honour map_mode (everything but the clustering null, ClusterTools.cpp:227)
  void run_map(const MapBuffers& b, bool simulated, bool states_only = false, bool variants = true);
  void prof_begin(const char* name);
  void prof_end(int launches);
  void prof_collect();
};

int64_t pad_sites(int64_t n);
void comm_all_gather(Context& c, const double* send, double* recv, size_t count);
// bins and sorts n device-resident samples into c.null (nmax < 0: the mapped alignment's max(norm))
void null_load(Context& c, const double* stat_dev, const double* nmin_dev, int64_t n, int K, double nmax);
// bytes of device memory one simulated site needs through simulate -> map x2 -> paired
size_t null_bytes_per_site(const Context& c);
// This rank's share of rep_cpu outer replicates: contiguous ranges, the first rep_cpu % n_ranks ranks get one more.
void replicate_range(int rep_cpu, int n_ranks, int rank, int& begin, int& end);
// The exchange of a sharded null: this rank's c.null samples (its replicate_range) are all-gathered over the
// communicator in blocks padded with Nmin = NaN, and every rank bins and sorts the union into c.null.
void gather_null_shards(Context& c, int rep_cpu, int rep_ram, int K, double nmax);

inline void check_stat(int stat_id) {
  if (stat_id < 0 || stat_id > CMB_STAT_MI_LABEL) fail("unknown statistic id %d", stat_id);
}
// whether any of the pair filters can drop a row
inline bool any_filter(const cmb_filters* f) {
  return f && (f->min_rate_class > 0 || f->min_rate > 0. || f->max_rate_class_diff >= 0 || f->max_rate_diff >= 0. ||
               f->min_stat > 0.);
}

extern thread_local std::string g_last_error; // defined in capi.cu

} // namespace cmb

struct cmb_ctx { cmb::Context c; };

// Every C ABI entry point returns 0, or 1 with the message for cmb_last_error.
#define CMB_TRY try {
#define CMB_CATCH                                   \
  }                                                 \
  catch (const std::exception& e) {                 \
    ::cmb::g_last_error = e.what();                 \
    return 1;                                       \
  }                                                 \
  catch (...) {                                     \
    ::cmb::g_last_error = "unknown error";          \
    return 1;                                       \
  }                                                 \
  return 0;
