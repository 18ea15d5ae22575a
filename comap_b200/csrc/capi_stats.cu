// C ABI, part 2: simulation, null distribution, pair statistics, clustering.
#include "../../include/comap_b200.h"
#include "context.h"
#include <algorithm>
#include <cmath>
#include <cstring>

using namespace cmb;

namespace cmb {

size_t null_bytes_per_site(const Context& c) {
  size_t D = (size_t)c.tree.n_slots * c.C * c.A * 8;
  size_t out = (size_t)c.tree.B * 8 * 2;
  size_t tips = (size_t)c.tree.n_leaves * 2;
  const size_t part = c.protein_mma ? (size_t)c.C * c.tree.B * 8 : 0; // per-class partial outputs of k1_mma20.cu
  return D + out + tips + part + (size_t)c.C * 8 + 16 * 8;
}

void null_load(Context& c, const double* stat_dev, const double* nmin_dev, int64_t n, int K, double nmax) {
  if (K < 1) fail("statistic.null.nb_rate_classes must be > 0 (Domain.cpp:49)");
  if (K > 4096) fail("too many null bins (%d)", K);
  const bool from_map = nmax < 0.;
  if (from_map) {
    c.finish_map();
    if (!c.mapped) fail("null binning with nmax < 0 needs a mapped alignment (cmb_map)");
    nmax = c.max_norm;
  }
  if (n > 0x7fffffff) fail("null distribution too large (%lld samples)", (long long)n);
  NullState& ns = c.null;
  ns.K = K; ns.nmax = nmax; ns.nmax_from_map = from_map;
  ns.sorted.reserve(sizeof(double) * (size_t)std::max<int64_t>(n, 1));
  ns.bin_off_dev.reserve(sizeof(int64_t) * (K + 2));
  c.prof_begin("sort");
  int l = bin_and_sort(n, stat_dev, nmin_dev, K, nmax, c.scratch2, ns.sorted.as<double>(),
                       ns.bin_off_dev.as<int64_t>(), c.stream);
  c.prof_end(l);
  ns.bin_off.assign(K + 1, 0);
  CMB_CUDA(cudaMemcpyAsync(ns.bin_off.data(), ns.bin_off_dev.p, sizeof(int64_t) * (K + 1), cudaMemcpyDeviceToHost,
                           c.stream));
  CMB_CUDA(cudaStreamSynchronize(c.stream));
  ns.ready = true;
}

} // namespace cmb

namespace {

// The two simulated alignments of a batch of outer replicates (AnalysisTools.cpp:591-611) live side by side in
// ONE set of mapping buffers -- columns [0, n) hold batch 1, [half, half + n) batch 2 -- so one down / up launch
// pair maps both (twice the CTAs per launch: a 125-replicate shard of an 8-GPU run fills 6.6 waves of the grid
// instead of 2 x 3.3), and the paired statistic reads the two halves of the same output matrix.
void null_core(Context& c, int stat_id, uint64_t seed, int rep_cpu, int rep_ram, int rep_begin, int rep_end,
               int weighted, int K, double nmax, double* raw, const uint8_t* sim1, const uint8_t* sim2) {
  check_stat(stat_id);
  if (rep_ram < 1 || rep_cpu < 0) fail("null: bad replicate counts");
  if (rep_begin < 0 || rep_end > rep_cpu || rep_begin > rep_end) fail("null: bad replicate range");
  CMB_CUDA(cudaSetDevice(c.device));
  c.ensure_streams();
  const int B = c.tree.B, T = c.tree.n_leaves;
  const int64_t R = rep_ram, nreps = rep_end - rep_begin, total = nreps * R;
  NullState& ns = c.null;
  ns.begin(total);
  // batch as many outer replicates as fit comfortably in free HBM (the answer is cached: cudaMemGetInfo
  // costs a host round trip per call)
  if (c.null_budget_sites <= 0) {
    size_t freeb = 0, totalb = 0;
    CMB_CUDA(cudaMemGetInfo(&freeb, &totalb));
    size_t held = c.s_D.cap + c.s_out[0].cap + c.s_tips[0].cap;
    size_t budget = (size_t)((freeb + held) * 0.6);
    c.null_budget_sites = std::max<int64_t>(1, (int64_t)(budget / null_bytes_per_site(c)));
  }
  int64_t max_sites = std::max<int64_t>(R, std::min<int64_t>(c.null_budget_sites, (int64_t)1 << 20));
  int64_t rpb = std::max<int64_t>(1, max_sites / R);
  MapModel m = c.map_model();
  // the corrected correlation scores simulated pairs with the OBSERVED alignment's mean vector
  // (one statistic object serves both loops upstream, CoMap.cpp:350-359)
  const bool corrected = stat_id == CMB_STAT_CORRECTED_CORRELATION;
  const double* mv = corrected ? c.mean_vector() : nullptr;
  int64_t off = 0;
  for (int64_t r0 = rep_begin; r0 < rep_end; r0 += rpb) {
    const int64_t nb = std::min<int64_t>(rpb, rep_end - r0), n = nb * R;
    const int64_t half = (n + 255) / 256 * 256, n_pad = pad_sites(half + n);
    MapBuffers bb = c.sim_buffers(0, half + n, n_pad);
    uint8_t* tips = c.s_tips[0].as<uint8_t>();
    c.clear_sim_tip_padding(n, n_pad);
    const bool dedup_on = !(getenv("CMB_NULL_DEDUP") && atoi(getenv("CMB_NULL_DEDUP")) == 0);
    const bool dedup = dedup_on && c.A == 4 && !c.map_mode; // the variant kernels walk every column
    int32_t *col_class = nullptr, *col_varied = nullptr;
    bool classified = false;
    if (sim1) {
      for (int k = 0; k < 2; k++) {
        const uint8_t* src = k == 0 ? sim1 : sim2;
        for (int64_t r = 0; r < nb; r++)
          CMB_CUDA(cudaMemcpy2DAsync(tips + k * half + r * R, n_pad, src + (size_t)(r0 + r) * T * R, R, R, T,
                                     cudaMemcpyHostToDevice, c.stream));
      }
    } else { // both batches in one launch: threads >= n simulate the second alignment's sites into the columns from `half`
      if (dedup && m.cont_kind == 0) { // the simulator classifies its columns while it writes them
        compress_class_buffers(n_pad, c.scratch2, &col_class, &col_varied);
        classified = true;
      }
      c.prof_begin("simulate");
      launch_simulate(m, c.sim_stream, seed, 2 * r0 * R, R, 2 * R, 2 * n, n_pad, weighted, c.tree.n_nodes - 1, tips, nullptr,
                      c.stream, n, half, R, col_class, col_varied);
      c.prof_end(1);
    }
    // Pattern compression (nucleotides): columns whose tips all carry the same state -- 16 % of the simulated
    // sites of config 4 -- are mapped once per state, as Bio++ maps distinct site patterns and copies
    // (LegacySubstitutionMappingTools::computeSubstitutionVectors over getNumberOfDistinctSites()).  The varied
    // columns are packed to the front of a second tip buffer with the A constant patterns behind them, the
    // mapping kernels stop at the packed count (a device scalar: no host round trip), and the paired statistic
    // reads each site's vector through a column index.
    const int32_t *col1 = nullptr, *col2 = nullptr;
    if (dedup) {
      c.s_tips[1].reserve((size_t)T * n_pad);
      c.s_cols.reserve(sizeof(int32_t) * (size_t)n_pad + 256);
      c.s_counts.reserve(sizeof(int32_t) * 2 * 4096);
      if (c.s_batches >= 4096) c.s_batches = 0;
      int32_t* counts = c.s_counts.as<int32_t>() + 2 * c.s_batches;
      c.prof_begin("compress");
      const int nl = launch_compress_constant(c.A, T, n, half, n_pad, tips, c.s_tips[1].as<uint8_t>(), c.s_cols.as<int32_t>(), counts,
                                              c.scratch2, c.stream, classified);
      c.prof_end(nl);
      bb.tips = c.s_tips[1].as<uint8_t>();
      bb.n_active = counts;
      col1 = c.s_cols.as<int32_t>(); col2 = col1 + half;
      c.s_batches++;
    }
    c.run_map(bb, true, sim1 == nullptr);
    c.prof_begin("null_pairs");
    launch_paired(corrected ? 0 : stat_id, c.mi_threshold, B, n, n_pad, n_pad, bb.out, dedup ? bb.out : bb.out + half, mv, mv,
                  ns.stat.as<double>() + off, ns.nmin.as<double>() + off, c.stream, col1, col2);
    c.prof_end(1);
    if (raw) {
      c.scratch.reserve(sizeof(double) * 4 * (size_t)n);
      launch_raw_rows(n, ns.stat.as<double>() + off, ns.nmin.as<double>() + off, bb.rate_class, dedup ? bb.rate_class : bb.rate_class + half,
                      bb.post_rate, dedup ? bb.post_rate : bb.post_rate + half, c.scratch.as<double>(), c.stream, col1, col2);
      c.prof.total_launches += 1;
      CMB_CUDA(cudaMemcpyAsync(raw + off * 4, c.scratch.p, sizeof(double) * 4 * (size_t)n, cudaMemcpyDeviceToHost,
                               c.stream));
      CMB_CUDA(cudaStreamSynchronize(c.stream));
    }
    off += n;
    c.prof.sites_simulated += 2 * n;
  }
  if (K > 0) null_load(c, ns.stat.as<double>(), ns.nmin.as<double>(), total, K, nmax);
  else if (!c.async_null) CMB_CUDA(cudaStreamSynchronize(c.stream));
}

// This rank's share of the outer replicates: contiguous ranges, the first rep_cpu % n_ranks ranks get one more.
void replicate_range(int rep_cpu, int n_ranks, int rank, int& begin, int& end) {
  const int q = rep_cpu / n_ranks, r = rep_cpu % n_ranks;
  begin = rank * q + std::min(rank, r);
  end = begin + q + (rank < r ? 1 : 0);
}

__global__ void k_fill_nan(double* p, int64_t n) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) p[i] = nan("");
}

struct GroupTable {
  std::vector<int32_t> members;
  std::vector<int64_t> offsets{0};
  std::vector<double> height, stat, nmin;
};

// distance matrix of the [B][n_pad] vectors into c.d_dist (CoMap.cpp:432-440)
void distance_on_device(Context& c, int dist_id, const double* out, int64_t S, int64_t S_pad, const double* mean,
                        const double* sd, const double* norm) {
  if (dist_id < 0 || dist_id > 2) fail("unknown distance id %d", dist_id);
  constexpr int TS = 64;
  const int64_t nt = (S + TS - 1) / TS;
  if (c.dist_tiles_S != S) { // the tile list depends on the site count only
    std::vector<int2> tiles;
    for (int64_t ti = 0; ti < nt; ti++)
      for (int64_t tj = ti; tj < nt; tj++) tiles.push_back(make_int2((int)ti, (int)tj));
    c.dist_tiles.reserve(tiles.size() * 8 + 256);
    CMB_CUDA(cudaMemcpyAsync(c.dist_tiles.p, tiles.data(), tiles.size() * 8, cudaMemcpyHostToDevice, c.stream));
    CMB_CUDA(cudaStreamSynchronize(c.stream)); // the host vector goes out of scope
    c.dist_tiles_S = S; c.dist_tiles_n = (int64_t)tiles.size();
  }
  c.d_dist.reserve(sizeof(double) * (size_t)S * S);
  TilesLaunch L;
  L.dist_mode = true;
  L.stat_id = dist_id == 0 ? 0 : dist_id == 1 ? 4 : 5;
  L.dist_is_stat = dist_id == 2;
  L.dist_comp = 1.; // StatisticBasedDistance(cor, 1.) (CoMap.cpp:410); CompensationDistance = 1 - stat
  L.B = c.tree.B; L.S = S; L.S_pad = S_pad; L.out = out; L.mean = mean; L.sd = sd; L.norm = norm;
  L.tiles = c.dist_tiles.as<int2>(); L.n_tiles = c.dist_tiles_n; L.n_rows = S; L.mat = c.d_dist.as<double>();
  c.prof_begin("distance");
  int nl = launch_tiles(L, c.stream);
  c.prof_end(nl);
}

void cluster_on_device(Context& c, int linkage, int64_t S) {
  if (linkage < 0 || linkage > 2) fail("unknown clustering method %d", linkage);
  if (S < 2) fail("clustering needs at least 2 sites");
  size_t o_l = 0, o_r = align256(4 * S), o_h = align256(o_r + 4 * S);
  c.staging.reserve(align256(o_h + 8 * S));
  unsigned char* sb = c.staging.as<unsigned char>();
  c.prof_begin("cluster");
  int nl = launch_cluster(S, linkage, c.d_dist.as<double>(), c.scratch2, (int32_t*)(sb + o_l), (int32_t*)(sb + o_r),
                          (double*)(sb + o_h), c.stream);
  c.prof_end(nl);
  c.h_left.resize(S - 1); c.h_right.resize(S - 1); c.h_height.resize(S - 1);
  CMB_CUDA(cudaMemcpyAsync(c.h_left.data(), sb + o_l, 4 * (S - 1), cudaMemcpyDeviceToHost, c.stream));
  CMB_CUDA(cudaMemcpyAsync(c.h_right.data(), sb + o_r, 4 * (S - 1), cudaMemcpyDeviceToHost, c.stream));
  CMB_CUDA(cudaMemcpyAsync(c.h_height.data(), sb + o_h, 8 * (S - 1), cudaMemcpyDeviceToHost, c.stream));
  CMB_CUDA(cudaStreamSynchronize(c.stream));
  for (int64_t k = 0; k + 1 < S; k++)
    if (c.h_left[k] < 0) fail("clustering stopped early: the distance matrix holds NaN");
}

// nb dendrograms (replicates of the clustering null) in one cooperative launch; results per problem
struct DendroHost { std::vector<int32_t> left, right; std::vector<double> height; };
void cluster_batch_on_device(Context& c, int linkage, int64_t S, int nb, DevBuf* dists, DevBuf* works, DevBuf& staging,
                             DendroHost* out) {
  if (linkage < 0 || linkage > 2) fail("unknown clustering method %d", linkage);
  if (S < 2) fail("clustering needs at least 2 sites");
  const size_t o_r = align256(4 * S), o_h = align256(o_r + 4 * S), per = align256(o_h + 8 * S);
  staging.reserve(per * nb);
  unsigned char* sb = staging.as<unsigned char>();
  double* mats[4]; int32_t* l[4]; int32_t* r[4]; double* h[4];
  for (int q = 0; q < nb; q++) {
    mats[q] = dists[q].as<double>();
    l[q] = (int32_t*)(sb + per * q); r[q] = (int32_t*)(sb + per * q + o_r); h[q] = (double*)(sb + per * q + o_h);
  }
  c.prof_begin("cluster");
  int nl = launch_cluster_batch(nb, S, linkage, mats, works, l, r, h, c.stream);
  c.prof_end(nl);
  for (int q = 0; q < nb; q++) {
    out[q].left.resize(S - 1); out[q].right.resize(S - 1); out[q].height.resize(S - 1);
    CMB_CUDA(cudaMemcpyAsync(out[q].left.data(), l[q], 4 * (S - 1), cudaMemcpyDeviceToHost, c.stream));
    CMB_CUDA(cudaMemcpyAsync(out[q].right.data(), r[q], 4 * (S - 1), cudaMemcpyDeviceToHost, c.stream));
    CMB_CUDA(cudaMemcpyAsync(out[q].height.data(), h[q], 8 * (S - 1), cudaMemcpyDeviceToHost, c.stream));
  }
  CMB_CUDA(cudaStreamSynchronize(c.stream));
  for (int q = 0; q < nb; q++)
    for (int64_t k = 0; k + 1 < S; k++)
      if (out[q].left[k] < 0) fail("clustering stopped early: the distance matrix holds NaN");
}

// One group per inner node of the dendrogram, emitted in post-order with members in DFS
// leaf order (ClusterTools::getGroups, ClusterTools.cpp:59-113), Nmin = min leaf norm
// (:296-319), Stat per Distance::setStatisticAsProperty (Distance.h:109-129,346-368,
// 390-422), size filter of CoMap.cpp:517.
void groups_of_dendrogram(Context& c, int dist_id, int max_size, int64_t S, int64_t S_pad, const double* out_dev,
                          const double* h_norm, GroupTable& g) {
  if (max_size < 1) fail("clustering.maximum_group_size must be positive");
  const std::vector<int32_t>&left = c.h_left, &right = c.h_right;
  const int32_t root = (int32_t)(2 * S - 2);
  std::vector<int32_t> stack{root}, dfs;
  std::vector<char> state(2 * S, 0);
  std::vector<int64_t> first(2 * S, 0);
  dfs.reserve(S);
  while (!stack.empty()) {
    int32_t v = stack.back();
    if (v < S) { first[v] = (int64_t)dfs.size(); dfs.push_back(v); stack.pop_back(); continue; }
    if (state[v] == 0) { first[v] = (int64_t)dfs.size(); state[v] = 1; stack.push_back(left[v - S]); continue; }
    if (state[v] == 1) { state[v] = 2; stack.push_back(right[v - S]); continue; }
    stack.pop_back();
    const int64_t cnt = (int64_t)dfs.size() - first[v];
    if (cnt > max_size) continue;
    double nmin = INFINITY;
    for (int64_t k = 0; k < cnt; k++) {
      int32_t mmb = dfs[first[v] + k];
      g.members.push_back(mmb);
      if (h_norm[mmb] < nmin) nmin = h_norm[mmb];
    }
    g.offsets.push_back((int64_t)g.members.size());
    const double h = c.h_height[v - S];
    g.height.push_back(h);
    g.nmin.push_back(nmin);
    g.stat.push_back(dist_id == 0 ? 1. - 2 * h : 2 * h); // compensation filled below
  }
  if (dist_id == 1 && !g.height.empty()) {
    const size_t ng = g.height.size();
    size_t o_m = 0, o_o = align256(4 * g.members.size()), o_s = align256(o_o + 8 * (ng + 1));
    c.scratch.reserve(align256(o_s + 8 * ng));
    unsigned char* sb = c.scratch.as<unsigned char>();
    CMB_CUDA(cudaMemcpyAsync(sb + o_m, g.members.data(), 4 * g.members.size(), cudaMemcpyHostToDevice, c.stream));
    CMB_CUDA(cudaMemcpyAsync(sb + o_o, g.offsets.data(), 8 * (ng + 1), cudaMemcpyHostToDevice, c.stream));
    launch_group_compensation((int64_t)ng, (const int32_t*)(sb + o_m), (const int64_t*)(sb + o_o), c.tree.B, S_pad,
                              out_dev, (double*)(sb + o_s), c.stream);
    c.prof.total_launches += 1;
    CMB_CUDA(cudaMemcpyAsync(g.stat.data(), sb + o_s, 8 * ng, cudaMemcpyDeviceToHost, c.stream));
    CMB_CUDA(cudaStreamSynchronize(c.stream));
  }
}

} // namespace

extern "C" {

int cmb_simulate(cmb_ctx* ctx, uint64_t seed, int64_t first_site, int64_t n, int32_t weighted_classes,
                 uint8_t* states, int32_t* classes) {
  CMB_TRY
  Context& c = ctx->c;
  CMB_CUDA(cudaSetDevice(c.device));
  c.ensure_streams();
  if (n < 1) fail("cmb_simulate: n must be positive");
  const int T = c.tree.n_leaves;
  const int64_t n_pad = pad_sites(n);
  c.s_tips[0].reserve((size_t)T * n_pad);
  c.s_cls.reserve(sizeof(int32_t) * n_pad);
  MapModel m = c.map_model();
  c.prof_begin("simulate");
  launch_simulate(m, c.sim_stream, seed, first_site, n, 0, n, n_pad, weighted_classes, c.tree.n_nodes - 1,
                  c.s_tips[0].as<uint8_t>(), c.s_cls.as<int32_t>(), c.stream);
  c.prof_end(1);
  CMB_CUDA(cudaMemcpy2DAsync(states, n, c.s_tips[0].p, n_pad, n, T, cudaMemcpyDeviceToHost, c.stream));
  if (classes) CMB_CUDA(cudaMemcpyAsync(classes, c.s_cls.p, sizeof(int32_t) * n, cudaMemcpyDeviceToHost, c.stream));
  CMB_CUDA(cudaStreamSynchronize(c.stream));
  CMB_CATCH
}

int cmb_null_intra(cmb_ctx* ctx, int32_t stat_id, uint64_t seed, int32_t rep_cpu, int32_t rep_ram, int32_t rep_begin,
                   int32_t rep_end, int32_t weighted_classes, int32_t K, double nmax, double* raw) {
  CMB_TRY
  null_core(ctx->c, stat_id, seed, rep_cpu, rep_ram, rep_begin, rep_end, weighted_classes, K, nmax, raw, nullptr, nullptr);
  CMB_CATCH
}

int cmb_null_intra_sharded(cmb_ctx* ctx, int32_t stat_id, uint64_t seed, int32_t rep_cpu, int32_t rep_ram,
                           int32_t weighted_classes, int32_t K, double nmax, double* raw) {
  CMB_TRY
  Context& c = ctx->c;
  if (K < 1) fail("cmb_null_intra_sharded: K must be positive");
  if (c.comm_size == 1) { // no communicator: the whole null on this GPU
    null_core(c, stat_id, seed, rep_cpu, rep_ram, 0, rep_cpu, weighted_classes, K, nmax, raw, nullptr, nullptr);
    return 0;
  }
  int r0, r1;
  replicate_range(rep_cpu, c.comm_size, c.comm_rank, r0, r1);
  const bool was_async = c.async_null;
  c.async_null = true; // no host wait between the last null kernel and the exchange
  struct Restore { Context& c; bool v; ~Restore() { c.async_null = v; } } restore{c, was_async};
  null_core(c, stat_id, seed, rep_cpu, rep_ram, r0, r1, weighted_classes, 0, 0., raw, nullptr, nullptr);
  // every rank contributes one block [stat (cap) | nmin (cap)], cap = the largest shard; unused entries carry
  // Nmin = NaN, which Domain::getIndex rejects, so they fall out of the binning like out-of-range samples
  const int64_t R = rep_ram, n = (int64_t)(r1 - r0) * R;
  const int64_t cap = ((int64_t)(rep_cpu + c.comm_size - 1) / c.comm_size) * R;
  c.gather_send.reserve(sizeof(double) * 2 * (size_t)cap);
  c.gather_recv.reserve(sizeof(double) * 2 * (size_t)cap * c.comm_size);
  double* send = c.gather_send.as<double>();
  if (n < cap) {
    k_fill_nan<<<(unsigned)((2 * cap + 255) / 256), 256, 0, c.stream>>>(send, 2 * cap);
    CMB_CUDA(cudaGetLastError());
    c.prof.total_launches += 1;
  }
  if (n > 0) {
    CMB_CUDA(cudaMemcpyAsync(send, c.null.stat.p, sizeof(double) * n, cudaMemcpyDeviceToDevice, c.stream));
    CMB_CUDA(cudaMemcpyAsync(send + cap, c.null.nmin.p, sizeof(double) * n, cudaMemcpyDeviceToDevice, c.stream));
  }
  comm_all_gather(c, send, c.gather_recv.as<double>(), 2 * (size_t)cap);
  // blocks [stat | nmin] per rank -> two contiguous arrays of comm_size * cap samples
  const int64_t tot = cap * c.comm_size;
  c.null.stat.reserve(sizeof(double) * (size_t)tot);
  c.null.nmin.reserve(sizeof(double) * (size_t)tot);
  CMB_CUDA(cudaMemcpy2DAsync(c.null.stat.p, sizeof(double) * cap, c.gather_recv.p, sizeof(double) * 2 * cap,
                             sizeof(double) * cap, c.comm_size, cudaMemcpyDeviceToDevice, c.stream));
  CMB_CUDA(cudaMemcpy2DAsync(c.null.nmin.p, sizeof(double) * cap, c.gather_recv.as<double>() + cap, sizeof(double) * 2 * cap,
                             sizeof(double) * cap, c.comm_size, cudaMemcpyDeviceToDevice, c.stream));
  c.null.n_samples = tot;
  null_load(c, c.null.stat.as<double>(), c.null.nmin.as<double>(), tot, K, nmax);
  CMB_CATCH
}

int cmb_null_intra_from_alignments(cmb_ctx* ctx, int32_t stat_id, int32_t rep_cpu, int32_t rep_ram, const uint8_t* sim1,
                                   const uint8_t* sim2, int32_t K, double nmax, double* raw) {
  CMB_TRY
  if (!sim1 || !sim2) fail("cmb_null_intra_from_alignments: alignments missing");
  const int64_t tot = (int64_t)rep_cpu * ctx->c.tree.n_leaves * rep_ram;
  for (int64_t i = 0; i < tot; i++)
    if (sim1[i] >= ctx->c.A || sim2[i] >= ctx->c.A) fail("cmb_null_intra_from_alignments: state out of range");
  null_core(ctx->c, stat_id, 0, rep_cpu, rep_ram, 0, rep_cpu, 0, K, nmax, raw, sim1, sim2);
  CMB_CATCH
}

int cmb_null_samples_dev(cmb_ctx* ctx, const double** stat_dev, const double** nmin_dev, int64_t* n) {
  CMB_TRY
  *stat_dev = ctx->c.null.stat.as<double>();
  *nmin_dev = ctx->c.null.nmin.as<double>();
  *n = ctx->c.null.n_samples;
  CMB_CATCH
}

int cmb_null_load_dev(cmb_ctx* ctx, const double* stat_dev, const double* nmin_dev, int64_t n, int32_t K, double nmax) {
  CMB_TRY
  CMB_CUDA(cudaSetDevice(ctx->c.device));
  null_load(ctx->c, stat_dev, nmin_dev, n, K, nmax);
  CMB_CATCH
}

int cmb_null_get(cmb_ctx* ctx, int32_t* K, double* nmax, int64_t* bin_offsets, double* sorted, int64_t capacity) {
  CMB_TRY
  Context& c = ctx->c;
  if (!c.null.ready) fail("cmb_null_get: no null distribution loaded");
  if (K) *K = c.null.K;
  if (nmax) *nmax = c.null.nmax;
  if (bin_offsets) std::memcpy(bin_offsets, c.null.bin_off.data(), sizeof(int64_t) * (c.null.K + 1));
  if (sorted) {
    int64_t n = c.null.bin_off[c.null.K];
    if (capacity < n) fail("cmb_null_get: capacity %lld < %lld", (long long)capacity, (long long)n);
    CMB_CUDA(cudaMemcpyAsync(sorted, c.null.sorted.p, sizeof(double) * n, cudaMemcpyDeviceToHost, c.stream));
    CMB_CUDA(cudaStreamSynchronize(c.stream));
  }
  CMB_CATCH
}

// column ids: 0 i, 1 j, 2 stat, 3 rcmin, 4 prmin, 5 nmin, 6 pvalue, 7 nsim
static const size_t kColElt[8] = {4, 4, 8, 4, 8, 8, 8, 4}; // Nsim <= 2^31 null samples: int32 (half the D2H)

int cmb_pairs_resident(cmb_ctx* ctx, int32_t stat_id, const cmb_filters* f, int32_t use_null, int32_t shard_index,
                       int32_t shard_count, uint32_t columns, int64_t* n_rows) {
  CMB_TRY
  Context& c = ctx->c;
  CMB_CUDA(cudaSetDevice(c.device));
  check_stat(stat_id);
  c.finish_map();
  if (!c.mapped) fail("cmb_pairs: call cmb_map first");
  if (use_null && !c.null.ready) fail("cmb_pairs: no null distribution (cmb_null_intra / cmb_null_load_dev)");
  if (shard_count < 1 || shard_index < 0 || shard_index >= shard_count) fail("cmb_pairs: bad shard");
  if (!use_null) columns &= ~(uint32_t)0xC0;
  const int64_t S = c.S;
  constexpr int TS = 64;
  // owned rows, dense offsets, tile list
  std::vector<int32_t> rows;
  std::vector<int64_t> row_off;
  int64_t total = 0;
  const int64_t period = 2 * (int64_t)shard_count;
  for (int64_t i = 0; i < S; i++) {
    int64_t r = i % period;
    if (shard_count == 1 || r == shard_index || r == period - 1 - shard_index) {
      rows.push_back((int32_t)i);
      row_off.push_back(total);
      total += S - 1 - i;
    }
  }
  std::vector<int2> tiles;
  const int64_t n_rows_owned = (int64_t)rows.size();
  for (int64_t ti = 0; ti * TS < n_rows_owned; ti++) {
    int64_t imin = rows[ti * TS];
    for (int64_t tj = (imin + 1) / TS; tj * TS < S; tj++) tiles.push_back(make_int2((int)ti, (int)tj));
  }
  const bool filtered = any_filter(f);
  const size_t nT = std::max<size_t>(total, 1);
  size_t o_rows = 0, o_roff = align256(o_rows + rows.size() * 4), o_tiles = align256(o_roff + row_off.size() * 8),
         o_end = align256(o_tiles + tiles.size() * 8);
  DevBuf& meta = c.scratch;
  meta.reserve(o_end + 256);
  unsigned char* mb = meta.as<unsigned char>();
  if (!rows.empty()) {
    CMB_CUDA(cudaMemcpyAsync(mb + o_rows, rows.data(), rows.size() * 4, cudaMemcpyHostToDevice, c.stream));
    CMB_CUDA(cudaMemcpyAsync(mb + o_roff, row_off.data(), row_off.size() * 8, cudaMemcpyHostToDevice, c.stream));
  }
  if (!tiles.empty())
    CMB_CUDA(cudaMemcpyAsync(mb + o_tiles, tiles.data(), tiles.size() * 8, cudaMemcpyHostToDevice, c.stream));
  // dense columns and, when filtering, compacted copies.  The layout is the same for every
  // column mask, so columns can be produced by separate calls (the null-independent ones
  // first, PValue / Nsim once the null exists) while earlier ones are still being copied out.
  size_t off[8] = {0}, off2[8] = {0}, cur = 0;
  for (int k = 0; k < 8; k++) {
    off[k] = cur; cur = align256(cur + kColElt[k] * nT);
    if (filtered) { off2[k] = cur; cur = align256(cur + kColElt[k] * nT); }
  }
  size_t o_keep = cur;
  cur = align256(cur + nT);
  if (c.copy_stream && cur + 256 > c.pair_table.cap) CMB_CUDA(cudaStreamSynchronize(c.copy_stream)); // growing frees the old table
  c.pair_table.reserve(cur + 256);
  unsigned char* sb = c.pair_table.as<unsigned char>();
  if (total > 0x7fffffff) fail("cmb_pairs: %lld pairs in one shard exceed the 2^31 - 1 rows one call scores; use more shards", (long long)total);

  TilesLaunch L;
  L.stat_id = stat_id; L.B = c.tree.B; L.S = S; L.S_pad = c.S_pad; L.out = c.d_out.as<double>();
  L.mean = c.pairs_mean.as<double>(); L.sd = c.pairs_sd.as<double>(); L.norm = c.pairs_norm.as<double>();
  if (stat_id == CMB_STAT_MI) { // the tile kernel reads the per-site category-1 counts through `mean`
    L.thr = c.mi_threshold;
    L.mean = c.mi_counts();
  }
  if (stat_id == CMB_STAT_CORRECTED_CORRELATION) { // correlation of the mean-vector-corrected rows
    L.mv = c.mean_vector();
    L.stat_id = CMB_STAT_CORRELATION;
    L.mean = c.corr_mean.as<double>(); L.sd = c.corr_sd.as<double>();
  }
  L.post_rate = c.d_pr.as<double>(); L.rate_class = c.d_rc.as<int32_t>();
  L.tiles = (const int2*)(mb + o_tiles); L.n_tiles = (int64_t)tiles.size();
  L.rows = shard_count == 1 ? nullptr : (const int32_t*)(mb + o_rows);
  L.n_rows = n_rows_owned; L.row_off = (const int64_t*)(mb + o_roff);
  if (f) {
    L.min_rate_class = f->min_rate_class; L.max_rate_class_diff = f->max_rate_class_diff;
    L.min_rate = f->min_rate; L.max_rate_diff = f->max_rate_diff; L.min_stat = f->min_stat;
  }
  L.any_filter = filtered;
  if (use_null) {
    L.K = c.null.K; L.nmax = c.null.nmax;
    L.bin_off = c.null.bin_off_dev.as<int64_t>(); L.sorted = c.null.sorted.as<double>();
  }
  auto dp = [&](int k) -> void* { return (columns >> k & 1) ? sb + off[k] : nullptr; };
  L.o_i = (int32_t*)dp(0); L.o_j = (int32_t*)dp(1); L.o_stat = (double*)dp(2); L.o_rcmin = (int32_t*)dp(3);
  L.o_prmin = (double*)dp(4); L.o_nmin = (double*)dp(5); L.o_pvalue = (double*)dp(6); L.o_nsim = (int32_t*)dp(7);
  L.o_keep = sb + o_keep;
  c.prof_begin("pairs");
  int nl = 0;
  // only PValue / Nsim asked for and Stat / Nmin of the same table are resident: no Gram tiles
  const bool pv_only = use_null && !filtered && (columns & 0x3Fu) == 0 && c.pairs_rows == total &&
                       c.pairs_col_off[2] == (int64_t)off[2] && c.pairs_col_off[5] == (int64_t)off[5] &&
                       c.pairs_stat_id == stat_id && c.pairs_shard_index == shard_index && c.pairs_shard_count == shard_count;
  if (pv_only) {
    launch_pvalues(total, (const double*)(sb + off[2]), (const double*)(sb + off[5]), L.K, L.nmax, L.bin_off, L.sorted,
                   L.o_pvalue, L.o_nsim, c.stream);
    nl = 1;
  } else nl = launch_tiles(L, c.stream);
  c.prof_end(nl);
  int64_t kept = total;
  if (filtered && total > 0) {
    int64_t* pos = nullptr;
    kept = compact_positions(total, L.o_keep, c.scratch2, &pos, c.stream);
    for (int k = 0; k < 8; k++) {
      if (!(columns >> k & 1)) continue;
      if (kColElt[k] == 4) compact_column<int32_t>(total, L.o_keep, pos, (int32_t*)(sb + off[k]), (int32_t*)(sb + off2[k]), c.stream);
      else compact_column<double>(total, L.o_keep, pos, (double*)(sb + off[k]), (double*)(sb + off2[k]), c.stream);
      off[k] = off2[k];
      c.prof.total_launches += 1;
    }
  }
  if (filtered || c.pairs_rows != kept) c.drop_pair_table(); // filtered tables are only valid as one consistent call
  for (int k = 0; k < 8; k++)
    if (columns >> k & 1) c.pairs_col_off[k] = (int64_t)off[k];
  c.pairs_rows = kept;
  c.pairs_stat_id = stat_id; c.pairs_shard_index = shard_index; c.pairs_shard_count = shard_count;
  if (n_rows) *n_rows = kept;
  CMB_CATCH
}

int cmb_pairs_fetch(cmb_ctx* ctx, int32_t column, void* host, int64_t capacity) {
  CMB_TRY
  Context& c = ctx->c;
  if (column < 0 || column > 7) fail("cmb_pairs_fetch: bad column %d", column);
  if (c.pairs_rows < 0 || c.pairs_col_off[column] < 0) fail("cmb_pairs_fetch: column %d is not resident", column);
  if (capacity < c.pairs_rows) fail("cmb_pairs_fetch: capacity %lld < %lld rows", (long long)capacity, (long long)c.pairs_rows);
  if (c.pairs_rows > 0) {
    // copies run on their own stream behind an event, so kernels enqueued later on the
    // compute stream (the null distribution) overlap the transfer
    if (!c.copy_stream) {
      CMB_CUDA(cudaStreamCreateWithFlags(&c.copy_stream, cudaStreamNonBlocking));
      CMB_CUDA(cudaEventCreateWithFlags(&c.copy_event, cudaEventDisableTiming));
    }
    CMB_CUDA(cudaEventRecord(c.copy_event, c.stream));
    CMB_CUDA(cudaStreamWaitEvent(c.copy_stream, c.copy_event, 0));
    CMB_CUDA(cudaMemcpyAsync(host, c.pair_table.as<unsigned char>() + c.pairs_col_off[column],
                             kColElt[column] * (size_t)c.pairs_rows, cudaMemcpyDeviceToHost, c.copy_stream));
  }
  CMB_CATCH
}

int cmb_pairs(cmb_ctx* ctx, int32_t stat_id, const cmb_filters* f, int32_t use_null, int32_t shard_index,
              int32_t shard_count, int64_t capacity, int32_t* out_i, int32_t* out_j, double* out_stat, int32_t* out_rcmin,
              double* out_prmin, double* out_nmin, double* out_pvalue, int32_t* out_nsim, int64_t* n_rows) {
  void* host[8] = {out_i, out_j, out_stat, out_rcmin, out_prmin, out_nmin, out_pvalue, out_nsim};
  uint32_t columns = 0;
  for (int k = 0; k < 8; k++) if (host[k]) columns |= 1u << k;
  int64_t kept = 0;
  int rc = cmb_pairs_resident(ctx, stat_id, f, use_null, shard_index, shard_count, columns, &kept);
  if (rc) return rc;
  CMB_TRY
  if (kept > capacity) fail("cmb_pairs: capacity %lld < %lld rows", (long long)capacity, (long long)kept);
  if (!use_null) columns &= ~(uint32_t)0xC0;
  for (int k = 0; k < 8; k++)
    if (columns >> k & 1) { if (cmb_pairs_fetch(ctx, k, host[k], capacity)) return 1; }
  CMB_CUDA(cudaStreamSynchronize(ctx->c.stream));
  if (ctx->c.copy_stream) CMB_CUDA(cudaStreamSynchronize(ctx->c.copy_stream));
  if (n_rows) *n_rows = kept;
  CMB_CATCH
}

int cmb_distance_matrix(cmb_ctx* ctx, int32_t dist_id, double* mat) {
  CMB_TRY
  Context& c = ctx->c;
  CMB_CUDA(cudaSetDevice(c.device));
  c.finish_map();
  if (!c.mapped) fail("cmb_distance_matrix: call cmb_map first");
  distance_on_device(c, dist_id, c.d_out.as<double>(), c.S, c.S_pad, c.pairs_mean.as<double>(),
                     c.pairs_sd.as<double>(), c.pairs_norm.as<double>());
  c.have_dist = true;
  c.dist_id = dist_id;
  if (mat) {
    CMB_CUDA(cudaMemcpyAsync(mat, c.d_dist.p, sizeof(double) * (size_t)c.S * c.S, cudaMemcpyDeviceToHost, c.stream));
    CMB_CUDA(cudaStreamSynchronize(c.stream));
  }
  CMB_CATCH
}

int cmb_cluster(cmb_ctx* ctx, int32_t linkage, int32_t* left, int32_t* right, double* height) {
  CMB_TRY
  Context& c = ctx->c;
  CMB_CUDA(cudaSetDevice(c.device));
  if (!c.have_dist) fail("cmb_cluster: call cmb_distance_matrix first");
  cluster_on_device(c, linkage, c.S);
  c.have_dist = false; // the matrix is consumed
  c.have_dendro = true;
  const int64_t n = c.S - 1;
  if (left) std::memcpy(left, c.h_left.data(), sizeof(int32_t) * n);
  if (right) std::memcpy(right, c.h_right.data(), sizeof(int32_t) * n);
  if (height) std::memcpy(height, c.h_height.data(), sizeof(double) * n);
  CMB_CATCH
}

int cmb_groups(cmb_ctx* ctx, int32_t dist_id, int32_t max_size, int32_t* members, int64_t* offsets, double* g_height,
               double* g_stat, double* g_nmin, int64_t* n_groups) {
  CMB_TRY
  Context& c = ctx->c;
  CMB_CUDA(cudaSetDevice(c.device));
  if (!c.have_dendro) fail("cmb_groups: call cmb_cluster first");
  GroupTable g;
  groups_of_dendrogram(c, dist_id, max_size, c.S, c.S_pad, c.d_out.as<double>(), c.h_norm, g);
  const int64_t ng = (int64_t)g.height.size();
  if (members && !g.members.empty()) std::memcpy(members, g.members.data(), sizeof(int32_t) * g.members.size());
  if (offsets) std::memcpy(offsets, g.offsets.data(), sizeof(int64_t) * (ng + 1));
  if (g_height && ng) std::memcpy(g_height, g.height.data(), sizeof(double) * ng);
  if (g_stat && ng) std::memcpy(g_stat, g.stat.data(), sizeof(double) * ng);
  if (g_nmin && ng) std::memcpy(g_nmin, g.nmin.data(), sizeof(double) * ng);
  if (n_groups) *n_groups = ng;
  CMB_CATCH
}

int cmb_cluster_null(cmb_ctx* ctx, int32_t dist_id, int32_t linkage, uint64_t seed, int32_t rep_begin, int32_t rep_end,
                     int32_t weighted_classes, int32_t max_size, int64_t capacity_rows, int64_t capacity_members,
                     int32_t* row_rep, int32_t* row_size, double* row_dmax, double* row_stat, double* row_nmin,
                     int32_t* members, int64_t* offsets, int64_t* n_rows) {
  CMB_TRY
  Context& c = ctx->c;
  CMB_CUDA(cudaSetDevice(c.device));
  if (!c.have_alignment) fail("cmb_cluster_null: the data set size comes from the alignment (cmb_set_alignment)");
  if (rep_begin < 0 || rep_end < rep_begin) fail("cmb_cluster_null: bad replicate range");
  c.ensure_streams();
  const int64_t S = c.S, S_pad = c.S_pad;
  const int B = c.tree.B;
  MapModel m = c.map_model();
  int64_t rows = 0, mem = 0;
  if (offsets) offsets[0] = 0;
  DevBuf &mean = c.cn_mean, &sd = c.cn_sd, &norm = c.cn_norm, &staging = c.cn_staging;
  // Replicates are clustered in batches: the exact merge loop is a chain of barrier latencies, so up to four
  // dendrograms advance through the same barriers (k4_cluster<NP>).  Each needs its own matrix and vectors.
  size_t free_b = 0, total_b = 0;
  CMB_CUDA(cudaMemGetInfo(&free_b, &total_b));
  size_t held = 0;
  for (int q = 0; q < 4; q++) held += c.cn_dists[q].cap + c.cn_outs[q].cap + c.cn_works[q].cap;
  const size_t per_rep = sizeof(double) * ((size_t)S * S + (size_t)B * S_pad) + ((size_t)64 << 20);
  int NB = (int)std::min<size_t>(4, std::max<size_t>(1, (size_t)(0.6 * (double)(free_b + held)) / per_rep));
  if (const char* e = std::getenv("CMB_K4_BATCH")) NB = std::max(1, std::min(4, atoi(e)));
  DevBuf *dists = c.cn_dists, *works = c.cn_works, *outs = c.cn_outs;
  std::vector<double> h_norms[4];
  DendroHost dendro[4];
  for (int rep0 = rep_begin; rep0 < rep_end; rep0 += NB) {
    const int nb = std::min(NB, rep_end - rep0);
    for (int q = 0; q < nb; q++) {
      const int rep = rep0 + q;
      // ClusterTools.cpp:224-227: simulate sizeOfDataSet sites, re-initialise, map
      MapBuffers b = c.sim_buffers(0, S, S_pad);
      c.prof_begin("simulate");
      launch_simulate(m, c.sim_stream, seed, (int64_t)rep * S, S, 0, S, S_pad, weighted_classes, c.tree.n_nodes - 1,
                      c.s_tips[0].as<uint8_t>(), nullptr, c.stream);
      c.prof_end(1);
      c.run_map(b, true, false, false); // ClusterTools.cpp:227: always computeSubstitutionVectors
      mean.reserve(sizeof(double) * S_pad); sd.reserve(sizeof(double) * S_pad); norm.reserve(sizeof(double) * S_pad);
      launch_prep(B, S, S_pad, b.out, nullptr, mean.as<double>(), sd.as<double>(), norm.as<double>(), c.stream);
      c.prof.total_launches += 1;
      h_norms[q].resize(S);
      CMB_CUDA(cudaMemcpyAsync(h_norms[q].data(), norm.p, sizeof(double) * S, cudaMemcpyDeviceToHost, c.stream));
      distance_on_device(c, dist_id, b.out, S, S_pad, mean.as<double>(), sd.as<double>(), norm.as<double>());
      std::swap(c.d_dist, dists[q]); // the matrix stays with this replicate; the next one gets (or allocates) another
      outs[q].reserve(sizeof(double) * (size_t)B * S_pad); // the group statistics need this replicate's vectors
      CMB_CUDA(cudaMemcpyAsync(outs[q].p, b.out, sizeof(double) * (size_t)B * S_pad, cudaMemcpyDeviceToDevice, c.stream));
    }
    cluster_batch_on_device(c, linkage, S, nb, dists, works, staging, dendro);
    for (int q = 0; q < nb; q++) {
      const int rep = rep0 + q;
      c.h_left.swap(dendro[q].left); c.h_right.swap(dendro[q].right); c.h_height.swap(dendro[q].height);
      GroupTable g;
      groups_of_dendrogram(c, dist_id, max_size, S, S_pad, outs[q].as<double>(), h_norms[q].data(), g);
      const int64_t ng = (int64_t)g.height.size();
      if (rows + ng > capacity_rows || mem + (int64_t)g.members.size() > capacity_members)
        fail("cmb_cluster_null: output capacity exceeded");
      for (int64_t k = 0; k < ng; k++) {
        if (row_rep) row_rep[rows + k] = rep;
        if (row_size) row_size[rows + k] = (int32_t)(g.offsets[k + 1] - g.offsets[k]);
        if (row_dmax) row_dmax[rows + k] = g.height[k] * 2.; // ClusterTools.cpp:286
        if (row_stat) row_stat[rows + k] = g.stat[k];
        if (row_nmin) row_nmin[rows + k] = g.nmin[k];
        if (offsets) offsets[rows + k + 1] = mem + g.offsets[k + 1];
      }
      if (members && !g.members.empty()) std::memcpy(members + mem, g.members.data(), sizeof(int32_t) * g.members.size());
      rows += ng;
      mem += (int64_t)g.members.size();
    }
  }
  c.have_dist = false; // the matrices were consumed
  c.have_dendro = false;
  if (n_rows) *n_rows = rows;
  CMB_CATCH
}

} // extern "C"
