// C ABI, part 3: two data sets ("inter-gene" analysis, SURVEY.md s8f-1).
//
//   cmb_pairs_inter  replaces CoETools::computeInterStats (CoETools.cpp:732-840): the statistic of
//                    every site of data set 1 with every site of data set 2 on the same tree
//                    topology (or site i with site i: independant_comparisons), the filters
//                    with per-data-set rate thresholds, rows in the reference's order.
//   cmb_null_inter   replaces AnalysisTools::getNullDistributionInterDR (AnalysisTools.cpp:662-735):
//                    rep_cpu x { simulate rep_ram sites under each data set's model, map both,
//                    paired statistic j<->j }, rows Stat RCmin PRmin Nmin; cmb_null_inter_range
//                    computes the rows of a range of outer replicates (a GPU's share).
// Each data set lives in its own context (tree, model, alignment, mapping); both must be on the
// same device.  The kernels are K2's (rectangle mode of k2_tiles, k2_paired) and K1/K3.
#include "../../include/comap_b200.h"
#include "context.h"
#include <algorithm>
#include <cmath>
#include <cstring>

using namespace cmb;

namespace {

void check_pair(const Context& a, const Context& b, const char* who) {
  if (a.device != b.device) fail("%s: both data sets must live on the same device", who);
  if (!a.have_tree || !b.have_tree || a.tree.B != b.tree.B)
    fail("%s: the two trees must have the same topology (%d vs %d branches)", who, a.tree.B, b.tree.B);
  // TreeTools::haveSameTopology (CoMap.cpp:243): same parent array
  if (a.tree.parent != b.tree.parent) fail("%s: the second tree must have the same topology as the first tree", who);
}

// second stream waits for everything queued on the first
void order_after(cudaStream_t later, cudaStream_t earlier) {
  if (later == earlier) return;
  cudaEvent_t e;
  CMB_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
  CMB_CUDA(cudaEventRecord(e, earlier));
  CMB_CUDA(cudaStreamWaitEvent(later, e, 0));
  CMB_CUDA(cudaEventDestroy(e));
}

} // namespace

extern "C" {

int cmb_pairs_inter(cmb_ctx* ctx1, cmb_ctx* ctx2, int32_t stat_id, const cmb_filters* f, int32_t min_rate_class2,
                    double min_rate2, int32_t independent, int32_t nmin_by_row, int64_t capacity, int32_t* out_i,
                    int32_t* out_j, double* out_stat, int32_t* out_rcmin, double* out_prmin, double* out_nmin,
                    int64_t* n_rows) {
  CMB_TRY
  Context& c = ctx1->c;
  Context& d = ctx2->c;
  CMB_CUDA(cudaSetDevice(c.device));
  check_stat(stat_id);
  check_pair(c, d, "cmb_pairs_inter");
  c.finish_map(); d.finish_map();
  if (!c.mapped || !d.mapped) fail("cmb_pairs_inter: call cmb_map on both data sets first");
  const int64_t S1 = c.S, S2 = d.S;
  if (independent && S1 != S2)
    fail("When performing independant comparisons, the two datasets must have the same length."); // CoETools.cpp:745-749
  const bool corrected = stat_id == CMB_STAT_CORRECTED_CORRELATION;
  const double* mv1 = corrected ? c.mean_vector() : nullptr;
  const double* mv2 = corrected ? d.mean_vector() : nullptr;
  order_after(c.stream, d.stream); // the second data set's mapping (and mean vector) is complete
  const bool filtered = any_filter(f) || min_rate_class2 > 0 || min_rate2 > 0.;
  const int64_t total = independent ? S1 : S1 * S2;
  if (total > 0x7fffffff) fail("cmb_pairs_inter: %lld pairs exceed the 2^31 - 1 rows one call scores", (long long)total);
  // dense columns i j stat rcmin prmin nmin | keep | compacted copies
  const size_t elt[6] = {4, 4, 8, 4, 8, 8};
  size_t off[6], off2[6], cur = 0;
  for (int k = 0; k < 6; k++) { off[k] = cur; cur = align256(cur + elt[k] * (size_t)total); }
  const size_t o_keep = cur;
  cur = align256(cur + (size_t)total);
  for (int k = 0; k < 6; k++) { off2[k] = cur; cur = align256(cur + (filtered ? elt[k] * (size_t)total : 0)); }
  if (c.copy_stream) CMB_CUDA(cudaStreamSynchronize(c.copy_stream));
  c.pair_table.reserve(cur + 256);
  c.drop_pair_table(); // the resident intra table is gone
  unsigned char* sb = c.pair_table.as<unsigned char>();
  int32_t* o_i = (int32_t*)(sb + off[0]); int32_t* o_j = (int32_t*)(sb + off[1]); double* o_stat = (double*)(sb + off[2]);
  int32_t* o_rc = (int32_t*)(sb + off[3]); double* o_pr = (double*)(sb + off[4]); double* o_nm = (double*)(sb + off[5]);
  uint8_t* o_keep_p = sb + o_keep;

  TilesLaunch L;
  L.stat_id = corrected ? CMB_STAT_CORRELATION : stat_id;
  L.B = c.tree.B; L.S = S1; L.S_pad = c.S_pad; L.out = c.d_out.as<double>();
  L.mean = corrected ? c.corr_mean.as<double>() : c.pairs_mean.as<double>();
  L.sd = corrected ? c.corr_sd.as<double>() : c.pairs_sd.as<double>();
  L.norm = c.pairs_norm.as<double>(); L.post_rate = c.d_pr.as<double>(); L.rate_class = c.d_rc.as<int32_t>();
  L.mv = mv1;
  L.out2 = d.d_out.as<double>(); L.S2 = S2; L.S2_pad = d.S_pad;
  L.mean2 = corrected ? d.corr_mean.as<double>() : d.pairs_mean.as<double>();
  L.sd2 = corrected ? d.corr_sd.as<double>() : d.pairs_sd.as<double>();
  L.norm2 = d.pairs_norm.as<double>(); L.post_rate2 = d.d_pr.as<double>(); L.rate_class2 = d.d_rc.as<int32_t>();
  L.mv2 = mv2;
  if (stat_id == CMB_STAT_MI) {
    d.mi_threshold = c.mi_threshold; d.have_mi_count = false; // one statistic object upstream: one threshold
    L.thr = c.mi_threshold; L.mean = c.mi_counts(); L.mean2 = d.mi_counts();
    order_after(c.stream, d.stream);
  }
  if (f) {
    L.min_rate_class = f->min_rate_class; L.max_rate_class_diff = f->max_rate_class_diff;
    L.min_rate = f->min_rate; L.max_rate_diff = f->max_rate_diff; L.min_stat = f->min_stat;
  }
  L.min_rate_class2 = min_rate_class2; L.min_rate2 = min_rate2;
  L.any_filter = filtered; L.nmin_by_row = nmin_by_row;
  L.o_i = o_i; L.o_j = o_j; L.o_stat = o_stat; L.o_rcmin = o_rc; L.o_prmin = o_pr; L.o_nmin = o_nm; L.o_keep = o_keep_p;
  c.prof_begin("pairs");
  int nl = 0;
  if (!independent) {
    constexpr int TS = 64;
    std::vector<int2> tiles;
    for (int64_t ti = 0; ti * TS < S1; ti++)
      for (int64_t tj = 0; tj * TS < S2; tj++) tiles.push_back(make_int2((int)ti, (int)tj));
    c.scratch.reserve(tiles.size() * sizeof(int2) + 256);
    CMB_CUDA(cudaMemcpyAsync(c.scratch.p, tiles.data(), tiles.size() * sizeof(int2), cudaMemcpyHostToDevice, c.stream));
    L.tiles = c.scratch.as<int2>(); L.n_tiles = (int64_t)tiles.size();
    L.rows = nullptr; L.n_rows = S1; L.row_off = nullptr;
    nl = launch_tiles(L, c.stream);
  } else {
    // site i with site i: the paired kernel on the two observed mappings, then the row columns
    nl = launch_inter_diagonal(L, c.stream);
  }
  c.prof_end(nl);
  int64_t kept = total;
  if (filtered && total > 0) {
    int64_t* pos = nullptr;
    kept = compact_positions(total, o_keep_p, c.scratch2, &pos, c.stream);
    for (int k = 0; k < 6; k++) {
      if (elt[k] == 4) compact_column<int32_t>(total, o_keep_p, pos, (int32_t*)(sb + off[k]), (int32_t*)(sb + off2[k]), c.stream);
      else compact_column<double>(total, o_keep_p, pos, (double*)(sb + off[k]), (double*)(sb + off2[k]), c.stream);
      off[k] = off2[k];
      c.prof.total_launches += 1;
    }
  }
  if (kept > capacity) fail("cmb_pairs_inter: capacity %lld < %lld rows", (long long)capacity, (long long)kept);
  void* host[6] = {out_i, out_j, out_stat, out_rcmin, out_prmin, out_nmin};
  for (int k = 0; k < 6; k++)
    if (host[k] && kept > 0)
      CMB_CUDA(cudaMemcpyAsync(host[k], sb + off[k], elt[k] * (size_t)kept, cudaMemcpyDeviceToHost, c.stream));
  CMB_CUDA(cudaStreamSynchronize(c.stream));
  if (n_rows) *n_rows = kept;
  CMB_CATCH
}

int cmb_null_inter_range(cmb_ctx* ctx1, cmb_ctx* ctx2, int32_t stat_id, uint64_t seed, int32_t rep_cpu, int32_t rep_ram,
                         int32_t rep_begin, int32_t rep_end, int32_t weighted_classes, double* raw) {
  CMB_TRY
  Context& c = ctx1->c;
  Context& d = ctx2->c;
  CMB_CUDA(cudaSetDevice(c.device));
  check_stat(stat_id);
  if (rep_ram < 1 || rep_cpu < 0) fail("cmb_null_inter: bad replicate counts");
  if (rep_begin < 0 || rep_end > rep_cpu || rep_begin > rep_end) fail("cmb_null_inter: bad replicate range");
  if (!raw) fail("cmb_null_inter: raw output buffer required");
  check_pair(c, d, "cmb_null_inter");
  c.ensure_streams();
  d.ensure_streams();
  const bool corrected = stat_id == CMB_STAT_CORRECTED_CORRELATION;
  const double* mv1 = corrected ? c.mean_vector() : nullptr;
  const double* mv2 = corrected ? d.mean_vector() : nullptr;
  const int B = c.tree.B;
  const int64_t R = rep_ram, total = (int64_t)(rep_end - rep_begin) * R;
  c.null.begin(total);
  // batch outer replicates: the two data sets' partials are alive at the same time
  size_t freeb = 0, totalb = 0;
  CMB_CUDA(cudaMemGetInfo(&freeb, &totalb));
  const size_t held = c.s_D.cap + c.s_out[0].cap + d.s_D.cap + d.s_out[0].cap;
  int64_t max_sites = (int64_t)((double)(freeb + held) * 0.6 / (double)(null_bytes_per_site(c) + null_bytes_per_site(d)));
  max_sites = std::min<int64_t>(std::max<int64_t>(max_sites, R), (int64_t)1 << 20);
  const int64_t rpb = std::max<int64_t>(1, max_sites / R);
  // the second simulator draws from its own stream of the same counter-based generator
  const uint64_t seed2 = seed ^ 0x9E3779B97F4A7C15ull;
  MapModel m1 = c.map_model(), m2 = d.map_model();
  int64_t off = 0;
  for (int64_t r0 = rep_begin; r0 < rep_end; r0 += rpb) {
    const int64_t nb = std::min<int64_t>(rpb, rep_end - r0), n = nb * R;
    const int64_t np1 = pad_sites(n), np2 = pad_sites(n);
    MapBuffers b1 = c.sim_buffers(0, n, np1), b2 = d.sim_buffers(0, n, np2);
    c.prof_begin("simulate");
    launch_simulate(m1, c.sim_stream, seed, r0 * R, R, R, n, np1, weighted_classes, c.tree.n_nodes - 1,
                    c.s_tips[0].as<uint8_t>(), nullptr, c.stream);
    c.prof_end(1);
    c.run_map(b1, true, true);
    order_after(d.stream, c.stream); // keeps the second data set's buffers ordered behind earlier readers
    launch_simulate(m2, d.sim_stream, seed2, r0 * R, R, R, n, np2, weighted_classes, d.tree.n_nodes - 1,
                    d.s_tips[0].as<uint8_t>(), nullptr, d.stream);
    d.prof.total_launches += 1;
    d.run_map(b2, true, true);
    order_after(c.stream, d.stream);
    c.prof_begin("null_pairs");
    launch_paired(corrected ? 0 : stat_id, c.mi_threshold, B, n, np1, np2, b1.out, b2.out, mv1, mv2, c.null.stat.as<double>() + off,
                  c.null.nmin.as<double>() + off, c.stream);
    c.prof_end(1);
    c.scratch.reserve(sizeof(double) * 4 * (size_t)n);
    launch_raw_rows(n, c.null.stat.as<double>() + off, c.null.nmin.as<double>() + off, b1.rate_class, b2.rate_class,
                    b1.post_rate, b2.post_rate, c.scratch.as<double>(), c.stream);
    c.prof.total_launches += 1;
    CMB_CUDA(cudaMemcpyAsync(raw + off * 4, c.scratch.p, sizeof(double) * 4 * (size_t)n, cudaMemcpyDeviceToHost, c.stream));
    CMB_CUDA(cudaStreamSynchronize(c.stream));
    off += n;
  }
  CMB_CATCH
}

int cmb_null_inter(cmb_ctx* ctx1, cmb_ctx* ctx2, int32_t stat_id, uint64_t seed, int32_t rep_cpu, int32_t rep_ram,
                   int32_t weighted_classes, double* raw) {
  return cmb_null_inter_range(ctx1, ctx2, stat_id, seed, rep_cpu, rep_ram, 0, rep_cpu, weighted_classes, raw);
}

} // extern "C"

// ------------------------------------------------------------------------------------------------
// Candidate groups (SURVEY.md s8f-3): CoMap.cpp:592-711, CandidateGroupSet (CoETools.h:139-300,
// CoETools.cpp:901-1038), computePValuesForCandidateGroups (CoETools.cpp:1042-1087).
// The sampler is the reference's sequential state machine, driven by the NORMS of the simulated
// sites; simulate / map / every statistic run on the device (K3, K1, k2_pair_list or the
// compensation group kernel).  Like upstream, simulated sites a group has not completed when a
// batch ends are dropped (CoETools.cpp:990-991).
namespace {

struct CandidateSet {
  int n_groups = 0;
  const int64_t* off = nullptr;      // [n_groups + 1] into sites
  const int32_t* sites = nullptr;    // site indices of the mapped alignment
  std::vector<char> analysable;
  std::vector<double> lo, hi;        // norm range per candidate site (flat, as `sites`)
  std::vector<int64_t> n1, n2;
  int64_t min_sim = 0;
  int64_t n_completed = 0, n_analysable = 0, n_trials = 0;
  int64_t group_pos = 0, site_pos = 0;
  std::vector<std::vector<int64_t>> pending; // per candidate site (flat): simulated columns waiting, FIFO
  std::vector<size_t> pending_head;
  int64_t size_of(int64_t g) const { return off[g + 1] - off[g]; }

  // CandidateGroupSet::nextCandidateSite, CoETools.cpp:901-933
  void next_site() {
    if (n2[group_pos] < min_sim) {
      site_pos++;
      if (site_pos >= size_of(group_pos)) {
        group_pos++;
        if (group_pos >= n_groups) group_pos = 0;
        site_pos = 0;
      }
    }
    const int64_t start = group_pos;
    if (n2[group_pos] >= min_sim || !analysable[group_pos]) {
      while (n2[group_pos] >= min_sim || !analysable[group_pos]) {
        group_pos++;
        if (group_pos >= n_groups) group_pos = 0;
        if (group_pos == start) fail("DEBUG: something wrong happened, this message should never appear!");
      }
      site_pos = 0;
    }
  }
};

struct GroupJob { int64_t group; std::vector<int64_t> cols; };

// group statistics on the device: min over the pairs (i > j) of the pair statistic, or the
// compensation group formula (Statistics.h:118-131, 267-295); `cols` index columns of `out`
void group_stats(Context& c, int stat_id, const double* out, int64_t n_pad, const double* mv,
                 const std::vector<GroupJob>& jobs, std::vector<double>& result) {
  result.assign(jobs.size(), 0.);
  if (jobs.empty()) return;
  const int B = c.tree.B;
  if (stat_id == CMB_STAT_COMPENSATION) {
    std::vector<int32_t> members;
    std::vector<int64_t> offsets{0};
    for (const auto& j : jobs) {
      for (int64_t col : j.cols) members.push_back((int32_t)col);
      offsets.push_back((int64_t)members.size());
    }
    const size_t o_off = align256(members.size() * 4), o_stat = align256(o_off + offsets.size() * 8);
    c.scratch2.reserve(o_stat + jobs.size() * 8 + 256);
    unsigned char* sb = c.scratch2.as<unsigned char>();
    CMB_CUDA(cudaMemcpyAsync(sb, members.data(), members.size() * 4, cudaMemcpyHostToDevice, c.stream));
    CMB_CUDA(cudaMemcpyAsync(sb + o_off, offsets.data(), offsets.size() * 8, cudaMemcpyHostToDevice, c.stream));
    launch_group_compensation((int64_t)jobs.size(), (const int32_t*)sb, (const int64_t*)(sb + o_off), B, n_pad, out,
                              (double*)(sb + o_stat), c.stream);
    c.prof.total_launches += 1;
    CMB_CUDA(cudaMemcpyAsync(result.data(), sb + o_stat, jobs.size() * 8, cudaMemcpyDeviceToHost, c.stream));
    CMB_CUDA(cudaStreamSynchronize(c.stream));
    return;
  }
  std::vector<int2> pairs;
  for (const auto& j : jobs)
    for (size_t a = 1; a < j.cols.size(); a++)
      for (size_t b = 0; b < a; b++) pairs.push_back(make_int2((int)j.cols[a], (int)j.cols[b])); // getValueForPair(v[i], v[j])
  std::vector<double> vals(pairs.size());
  const size_t o_stat = align256(pairs.size() * sizeof(int2));
  c.scratch2.reserve(o_stat + pairs.size() * 8 + 256);
  unsigned char* sb = c.scratch2.as<unsigned char>();
  if (!pairs.empty()) {
    CMB_CUDA(cudaMemcpyAsync(sb, pairs.data(), pairs.size() * sizeof(int2), cudaMemcpyHostToDevice, c.stream));
    const bool corrected = stat_id == CMB_STAT_CORRECTED_CORRELATION;
    launch_pair_list(corrected ? 0 : stat_id, c.mi_threshold, B, n_pad, out, corrected ? mv : nullptr, (const int2*)sb, (int64_t)pairs.size(),
                     (double*)(sb + o_stat), c.stream);
    c.prof.total_launches += 1;
    CMB_CUDA(cudaMemcpyAsync(vals.data(), sb + o_stat, pairs.size() * 8, cudaMemcpyDeviceToHost, c.stream));
    CMB_CUDA(cudaStreamSynchronize(c.stream));
  }
  size_t k = 0;
  for (size_t g = 0; g < jobs.size(); g++) {
    double mini = INFINITY; // -log(0)
    const size_t n = jobs[g].cols.size();
    for (size_t a = 1; a < n; a++)
      for (size_t b = 0; b < a; b++) {
        const double val = vals[k++];
        if (val < mini) mini = val;
      }
    result[g] = mini;
  }
}

} // namespace

extern "C" int cmb_candidates(cmb_ctx* ctx, int32_t stat_id, int32_t n_groups, const int64_t* group_off,
                              const int32_t* group_sites, const uint8_t* analysable, double omega, int64_t min_sim,
                              int32_t max_trials, int32_t rep_ram, uint64_t seed, int32_t weighted_classes,
                              double* out_stat, double* out_pvalue, int64_t* out_n1, int64_t* out_n2, int64_t* n_simulated) {
  CMB_TRY
  Context& c = ctx->c;
  CMB_CUDA(cudaSetDevice(c.device));
  check_stat(stat_id);
  c.finish_map();
  if (!c.mapped) fail("cmb_candidates: call cmb_map first");
  if (n_groups < 1) fail("ERROR!!! No group can be tested!"); // CoMap.cpp:679-680
  if (rep_ram < 1 || min_sim < 1) fail("cmb_candidates: bad simulation counts");
  c.ensure_streams();
  const double* mv = stat_id == CMB_STAT_CORRECTED_CORRELATION ? c.mean_vector() : nullptr;
  CandidateSet cs;
  cs.n_groups = n_groups; cs.off = group_off; cs.sites = group_sites; cs.min_sim = min_sim;
  cs.analysable.assign(n_groups, 1);
  cs.n1.assign(n_groups, 0); cs.n2.assign(n_groups, 0);
  const int64_t n_sites = group_off[n_groups];
  cs.lo.resize(n_sites); cs.hi.resize(n_sites);
  cs.pending.assign(n_sites, {}); cs.pending_head.assign(n_sites, 0);
  std::vector<GroupJob> obs;
  for (int g = 0; g < n_groups; g++) {
    cs.analysable[g] = analysable ? (analysable[g] != 0) : 1;
    if (!cs.analysable[g]) continue;
    cs.n_analysable++;
    if (cs.size_of(g) < 2) fail("Error, group %d has %lld sites.", g, (long long)cs.size_of(g)); // CoMap.cpp:645-648
    GroupJob j; j.group = g;
    for (int64_t k = group_off[g]; k < group_off[g + 1]; k++) {
      const int32_t s = group_sites[k];
      if (s < 0 || s >= c.S) fail("cmb_candidates: site index %d out of range", s);
      j.cols.push_back(s);
      cs.lo[k] = c.h_norm[s] - omega; // CandidateGroup::computeNormRanges, CoETools.h:118-128
      cs.hi[k] = c.h_norm[s] + omega;
    }
    obs.push_back(std::move(j));
  }
  if (cs.n_analysable == 0) fail("ERROR!!! No group can be tested!");
  std::vector<double> observed(n_groups, NAN), tmp;
  group_stats(c, stat_id, c.d_out.as<double>(), c.S_pad, mv, obs, tmp);
  for (size_t k = 0; k < obs.size(); k++) observed[obs[k].group] = tmp[k];

  MapModel m = c.map_model();
  const int64_t R = rep_ram, n_pad = pad_sites(R);
  std::vector<double> norms(R);
  int64_t batch = 0;
  bool test = true;
  while (test) { // CoETools::computePValuesForCandidateGroups, CoETools.cpp:1053-1086
    MapBuffers b = c.sim_buffers(0, R, n_pad);
    c.prof_begin("simulate");
    launch_simulate(m, c.sim_stream, seed, batch * R, R, R, R, n_pad, weighted_classes, c.tree.n_nodes - 1,
                    c.s_tips[0].as<uint8_t>(), nullptr, c.stream);
    c.prof_end(1);
    c.run_map(b, true, true);
    c.scratch.reserve(sizeof(double) * 3 * (size_t)n_pad);
    double* dmean = c.scratch.as<double>();
    launch_prep(c.tree.B, R, n_pad, b.out, nullptr, dmean, dmean + n_pad, dmean + 2 * n_pad, c.stream);
    c.prof.total_launches += 1;
    CMB_CUDA(cudaMemcpyAsync(norms.data(), dmean + 2 * n_pad, sizeof(double) * R, cudaMemcpyDeviceToHost, c.stream));
    CMB_CUDA(cudaStreamSynchronize(c.stream));
    batch++;
    // ---- CandidateGroupSet::analyseSimulations, CoETools.cpp:948-995
    std::vector<GroupJob> jobs;
    bool test_free = true;
    for (int64_t i = 0; test && i < R; i++) {
      bool first = true, test_norm = false;
      int64_t start_g = 0, start_s = 0;
      while (test && !test_norm) {
        cs.next_site();
        if (first) { start_g = cs.group_pos; start_s = cs.site_pos; first = false; }
        else if (cs.group_pos == start_g && cs.site_pos == start_s) break; // looped over the whole set: drop this site
        const int64_t k = group_off[cs.group_pos] + cs.site_pos;
        test_norm = norms[i] >= cs.lo[k] && norms[i] <= cs.hi[k];
        if (test_norm) {
          // addSimulatedSite, CoETools.cpp:999-1038
          const int64_t g = cs.group_pos;
          cs.pending[k].push_back(i);
          bool complete = true;
          for (int64_t q = group_off[g]; complete && q < group_off[g + 1]; q++)
            if (cs.pending_head[q] >= cs.pending[q].size()) complete = false;
          if (complete) {
            GroupJob j; j.group = g;
            for (int64_t q = group_off[g]; q < group_off[g + 1]; q++) j.cols.push_back(cs.pending[q][cs.pending_head[q]++]);
            jobs.push_back(std::move(j));
            cs.n2[g]++;
            if (cs.n2[g] == min_sim) cs.n_completed++;
            test_free = false;
          }
          if (cs.n_completed == cs.n_analysable) test = false;
        }
      }
    }
    if (test_free) cs.n_trials++;
    for (auto& p : cs.pending) p.clear(); // resetSimulations: unfinished groups lose their sites
    std::fill(cs.pending_head.begin(), cs.pending_head.end(), 0);
    group_stats(c, stat_id, b.out, n_pad, mv, jobs, tmp);
    for (size_t k = 0; k < jobs.size(); k++)
      if (tmp[k] >= observed[jobs[k].group]) cs.n1[jobs[k].group]++;
    test = test && cs.n_trials < max_trials;
  }
  for (int g = 0; g < n_groups; g++) {
    if (out_stat) out_stat[g] = observed[g];
    if (out_pvalue) out_pvalue[g] = cs.analysable[g] ? ((double)cs.n1[g] + 1.) / ((double)cs.n2[g] + 1.) : NAN;
    if (out_n1) out_n1[g] = cs.n1[g];
    if (out_n2) out_n2[g] = cs.n2[g];
  }
  if (n_simulated) *n_simulated = batch * R;
  CMB_CATCH
}
