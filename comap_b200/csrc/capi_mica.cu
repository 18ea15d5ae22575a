// C ABI, part 4: Mica (CoMap/Mica.cpp) -- mutual information between alignment columns with the p-value epilogue of
// the pairwise analysis.  The entry points follow the program's phases: site statistics (Mica.cpp:341-361), the null
// distribution (parametric bootstrap :470-545 on the device; the other methods build their samples from
// cmb_mica_pairs / cmb_mica_pair_list on the host and hand them to cmb_null_load), the table (:646-689).
#include "context.h"
#include "../../include/comap_b200.h"
#include <algorithm>
#include <cstring>

using namespace cmb;

namespace {

// dense columns of the pair table in c.mica_table: MI | Hjoint | Hmin | Nmin | PValue | i | j | Nsim
struct MicaTable {
  int64_t n;
  double *mi, *hj, *hmin, *nmin, *pv;
  int32_t *i, *j, *nsim;
};
MicaTable mica_table(Context& c) {
  const int64_t n = c.S * (c.S - 1) / 2;
  const size_t d = align256(sizeof(double) * (size_t)std::max<int64_t>(n, 1)), w = align256(sizeof(int32_t) * (size_t)std::max<int64_t>(n, 1));
  c.mica_table.reserve(5 * d + 3 * w);
  unsigned char* b = c.mica_table.as<unsigned char>();
  MicaTable t;
  t.n = n;
  t.mi = (double*)b; t.hj = (double*)(b + d); t.hmin = (double*)(b + 2 * d); t.nmin = (double*)(b + 3 * d); t.pv = (double*)(b + 4 * d);
  t.i = (int32_t*)(b + 5 * d); t.j = (int32_t*)(b + 5 * d + w); t.nsim = (int32_t*)(b + 5 * d + 2 * w);
  return t;
}

// entropy and dense MI / Hjoint of the current alignment, computed once per alignment
void ensure_mica(Context& c) {
  if (!c.have_alignment) fail("mica: call cmb_set_alignment first");
  if (c.S < 2) fail("mica: at least two sites are needed");
  if (c.mica_ready) return;
  const int T = c.tree.n_leaves;
  c.mica_sites.reserve(2 * sizeof(double) * (size_t)c.S_pad);
  MicaTable t = mica_table(c);
  const uint32_t* cm = c.d_code_mask.as<uint32_t>();
  c.prof_begin("mica_pairs");
  launch_mica_entropy(c.A, T, c.S, c.S_pad, c.d_tips.as<uint8_t>(), cm, c.mica_sites.as<double>(), c.stream);
  launch_mica_pairs(c.A, T, c.S, c.S_pad, c.d_tips.as<uint8_t>(), cm, t.mi, t.hj, c.stream);
  launch_mica_average(c.S, t.mi, c.mica_sites.as<double>() + c.S_pad, c.stream);
  c.prof_end(3);
  c.mica_ready = true;
}

// Mica.cpp:505-541 over the outer replicates [rep_begin, rep_end): two simulated alignments of rep_ram sites per
// replicate, their mappings for the norms (computeSubstitutionVectors, whatever nijt.average says), MI and joint
// entropy of site j with site j.  The simulator is keyed by the global site 2 r rep_ram, so ranges concatenate to the
// whole null; c.null holds this range's samples, raw (nullable) its rows.
void mica_null_core(Context& c, uint64_t seed, int rep_cpu, int rep_ram, int rep_begin, int rep_end, int weighted_classes, int K,
                    double nmax, double* raw) {
  CMB_CUDA(cudaSetDevice(c.device));
  c.ensure_streams();
  if (rep_cpu < 1 || rep_ram < 1) fail("cmb_mica_null_parametric: rep_cpu and rep_ram must be positive");
  if (rep_begin < 0 || rep_end > rep_cpu || rep_begin > rep_end) fail("cmb_mica_null_parametric: bad replicate range");
  const int B = c.tree.B, T = c.tree.n_leaves;
  const int64_t R = rep_ram, total = (int64_t)(rep_end - rep_begin) * R;
  NullState& ns = c.null;
  ns.begin(total);
  MapModel m = c.map_model();
  const uint32_t* ident = c.d_identity_mask.as<uint32_t>();
  const int64_t half = (R + 255) / 256 * 256, n_pad = pad_sites(half + R);
  for (int64_t r = rep_begin; r < rep_end; r++) {
    const int64_t o = (r - rep_begin) * R;              // this replicate's first sample of the range
    MapBuffers bb = c.sim_buffers(0, half + R, n_pad);
    uint8_t* tips = c.s_tips[0].as<uint8_t>();
    c.clear_sim_tip_padding(R, n_pad);
    c.prof_begin("simulate");
    launch_simulate(m, c.sim_stream, seed, 2 * r * R, R, 2 * R, 2 * R, n_pad, weighted_classes, c.tree.n_nodes - 1, tips, nullptr,
                    c.stream, R, half, R);
    c.prof_end(1);
    c.run_map(bb, true, true, false);
    c.scratch.reserve(sizeof(double) * 4 * (size_t)n_pad);
    double* prep = c.scratch.as<double>();             // mean | sd | norm of the mapped batch pair
    launch_prep(B, half + R, n_pad, bb.out, nullptr, prep, prep + n_pad, prep + 2 * n_pad, c.stream);
    double* hj = prep + 3 * n_pad;
    c.prof_begin("mica_null");
    launch_mica_listed(c.A, T, R, tips, n_pad, tips + half, n_pad, nullptr, nullptr, ident, ns.stat.as<double>() + o, hj, c.stream);
    launch_min2(R, prep + 2 * n_pad, prep + 2 * n_pad + half, ns.nmin.as<double>() + o, c.stream);
    c.prof_end(3);
    if (raw) { // rows of null.output.file: MI, Hjoint, Nmin
      std::vector<double> h_mi(R), h_hj(R), h_nm(R);
      CMB_CUDA(cudaMemcpyAsync(h_mi.data(), ns.stat.as<double>() + o, sizeof(double) * R, cudaMemcpyDeviceToHost, c.stream));
      CMB_CUDA(cudaMemcpyAsync(h_hj.data(), hj, sizeof(double) * R, cudaMemcpyDeviceToHost, c.stream));
      CMB_CUDA(cudaMemcpyAsync(h_nm.data(), ns.nmin.as<double>() + o, sizeof(double) * R, cudaMemcpyDeviceToHost, c.stream));
      CMB_CUDA(cudaStreamSynchronize(c.stream));
      for (int64_t j = 0; j < R; j++) { raw[(o + j) * 3] = h_mi[j]; raw[(o + j) * 3 + 1] = h_hj[j]; raw[(o + j) * 3 + 2] = h_nm[j]; }
    }
    c.prof.sites_simulated += 2 * R;
  }
  if (K > 0) null_load(c, ns.stat.as<double>(), ns.nmin.as<double>(), total, K, nmax);
  else CMB_CUDA(cudaStreamSynchronize(c.stream));
}

} // namespace

extern "C" {

int cmb_mica_sites(cmb_ctx* ctx, double* entropy, double* average_mi) {
  CMB_TRY
  Context& c = ctx->c;
  CMB_CUDA(cudaSetDevice(c.device));
  ensure_mica(c);
  if (entropy) CMB_CUDA(cudaMemcpyAsync(entropy, c.mica_sites.p, sizeof(double) * c.S, cudaMemcpyDeviceToHost, c.stream));
  if (average_mi)
    CMB_CUDA(cudaMemcpyAsync(average_mi, c.mica_sites.as<double>() + c.S_pad, sizeof(double) * c.S, cudaMemcpyDeviceToHost, c.stream));
  CMB_CUDA(cudaStreamSynchronize(c.stream));
  CMB_CATCH
}

int cmb_mica_pairs(cmb_ctx* ctx, int32_t key, int32_t use_null, int64_t capacity, int32_t* out_i, int32_t* out_j, double* mi,
                   double* hjoint, double* hmin, double* nmin, double* pvalue, int32_t* nsim, int64_t* n_rows) {
  CMB_TRY
  Context& c = ctx->c;
  CMB_CUDA(cudaSetDevice(c.device));
  ensure_mica(c);
  if (key != CMB_MICA_KEY_NMIN && key != CMB_MICA_KEY_HMIN) fail("cmb_mica_pairs: key must be CMB_MICA_KEY_NMIN or CMB_MICA_KEY_HMIN");
  if (use_null && !c.null.ready) fail("cmb_mica_pairs: no null distribution (cmb_mica_null_parametric / cmb_null_load)");
  c.finish_map();
  if (key == CMB_MICA_KEY_NMIN && !c.mapped) fail("cmb_mica_pairs: conditioning on Nmin needs a mapped alignment (cmb_map)");
  MicaTable t = mica_table(c);
  if (capacity < t.n) fail("cmb_mica_pairs: capacity %lld < %lld pairs", (long long)capacity, (long long)t.n);
  launch_mica_rows(c.S, c.mica_sites.as<double>(), c.mapped ? c.pairs_norm.as<double>() : nullptr, t.i, t.j, t.hmin, t.nmin, c.stream);
  c.prof.total_launches += 1;
  if (use_null) { // Mica.cpp:672-683: the pairwise analysis' count in the sorted bin of Nmin (model) or Hmin
    launch_pvalues(t.n, t.mi, key == CMB_MICA_KEY_NMIN ? t.nmin : t.hmin, c.null.K, c.null.nmax, c.null.bin_off_dev.as<int64_t>(),
                   c.null.sorted.as<double>(), t.pv, t.nsim, c.stream);
    c.prof.total_launches += 1;
  }
  auto get = [&](void* host, const void* dev, size_t elt) {
    if (host) CMB_CUDA(cudaMemcpyAsync(host, dev, elt * (size_t)t.n, cudaMemcpyDeviceToHost, c.stream));
  };
  get(out_i, t.i, 4); get(out_j, t.j, 4); get(mi, t.mi, 8); get(hjoint, t.hj, 8); get(hmin, t.hmin, 8); get(nmin, t.nmin, 8);
  if (use_null) { get(pvalue, t.pv, 8); get(nsim, t.nsim, 4); }
  CMB_CUDA(cudaStreamSynchronize(c.stream));
  if (n_rows) *n_rows = t.n;
  CMB_CATCH
}

int cmb_mica_pair_list(cmb_ctx* ctx, int64_t n, const int32_t* site1, const int32_t* site2, double* mi, double* hjoint) {
  CMB_TRY
  Context& c = ctx->c;
  CMB_CUDA(cudaSetDevice(c.device));
  if (!c.have_alignment) fail("cmb_mica_pair_list: call cmb_set_alignment first");
  if (n < 0 || !site1 || !site2 || !mi) fail("cmb_mica_pair_list: bad arguments");
  for (int64_t r = 0; r < n; r++)
    if (site1[r] < 0 || site1[r] >= c.S || site2[r] < 0 || site2[r] >= c.S) fail("cmb_mica_pair_list: site index out of range at %lld", (long long)r);
  const size_t w = align256(sizeof(int32_t) * (size_t)std::max<int64_t>(n, 1)), d = align256(sizeof(double) * (size_t)std::max<int64_t>(n, 1));
  c.scratch.reserve(2 * w + 2 * d);
  unsigned char* b = c.scratch.as<unsigned char>();
  CMB_CUDA(cudaMemcpyAsync(b, site1, sizeof(int32_t) * n, cudaMemcpyHostToDevice, c.stream));
  CMB_CUDA(cudaMemcpyAsync(b + w, site2, sizeof(int32_t) * n, cudaMemcpyHostToDevice, c.stream));
  double* dmi = (double*)(b + 2 * w);
  double* dhj = (double*)(b + 2 * w + d);
  launch_mica_listed(c.A, c.tree.n_leaves, n, c.d_tips.as<uint8_t>(), c.S_pad, c.d_tips.as<uint8_t>(), c.S_pad, (const int32_t*)b,
                     (const int32_t*)(b + w), c.d_code_mask.as<uint32_t>(), dmi, dhj, c.stream);
  c.prof.total_launches += 1;
  CMB_CUDA(cudaMemcpyAsync(mi, dmi, sizeof(double) * n, cudaMemcpyDeviceToHost, c.stream));
  if (hjoint) CMB_CUDA(cudaMemcpyAsync(hjoint, dhj, sizeof(double) * n, cudaMemcpyDeviceToHost, c.stream));
  CMB_CUDA(cudaStreamSynchronize(c.stream));
  CMB_CATCH
}

int cmb_mica_permutations_shard(cmb_ctx* ctx, uint64_t seed, int32_t max_permutations, int32_t shard_index, int32_t shard_count,
                                int64_t capacity, double* pvalue, int32_t* nperm, int64_t* n_rows) {
  CMB_TRY
  Context& c = ctx->c;
  CMB_CUDA(cudaSetDevice(c.device));
  if (!c.have_alignment) fail("cmb_mica_permutations: call cmb_set_alignment first");
  if (c.S < 2) fail("mica: at least two sites are needed");
  if (max_permutations < 1) fail("Permutation number should be greater than 0!"); // Mica.cpp:611-614
  if (shard_count < 1 || shard_index < 0 || shard_index >= shard_count)
    fail("cmb_mica_permutations: bad shard %d of %d", shard_index, shard_count);
  const int64_t n_pairs = c.S * (c.S - 1) / 2;
  const int64_t n = shard_index < n_pairs ? (n_pairs - 1 - shard_index) / shard_count + 1 : 0; // idx = shard_index + k shard_count
  if (capacity < n) fail("cmb_mica_permutations: capacity %lld < %lld pairs", (long long)capacity, (long long)n);
  const size_t d = align256(sizeof(double) * (size_t)n), w = align256(sizeof(int32_t) * (size_t)n);
  c.scratch.reserve(d + w + 256);
  double* pv = c.scratch.as<double>();
  int32_t* np = (int32_t*)(c.scratch.as<unsigned char>() + d);
  unsigned long long* next = (unsigned long long*)(c.scratch.as<unsigned char>() + d + w); // the kernel's work counter
  c.prof_begin("mica_perm");
  launch_mica_permutations(c.A, c.tree.n_leaves, c.S, c.S_pad, c.d_tips.as<uint8_t>(), c.d_code_mask.as<uint32_t>(), seed,
                           max_permutations, shard_index, shard_count, n, next, pv, np, c.stream);
  c.prof_end(n > 0 ? 2 : 0);
  if (pvalue && n > 0) CMB_CUDA(cudaMemcpyAsync(pvalue, pv, sizeof(double) * n, cudaMemcpyDeviceToHost, c.stream));
  if (nperm && n > 0) CMB_CUDA(cudaMemcpyAsync(nperm, np, sizeof(int32_t) * n, cudaMemcpyDeviceToHost, c.stream));
  CMB_CUDA(cudaStreamSynchronize(c.stream));
  if (n_rows) *n_rows = n;
  CMB_CATCH
}

int cmb_mica_permutations(cmb_ctx* ctx, uint64_t seed, int32_t max_permutations, int64_t capacity, double* pvalue, int32_t* nperm,
                          int64_t* n_rows) {
  return cmb_mica_permutations_shard(ctx, seed, max_permutations, 0, 1, capacity, pvalue, nperm, n_rows);
}

int cmb_mica_null_parametric_range(cmb_ctx* ctx, uint64_t seed, int32_t rep_cpu, int32_t rep_ram, int32_t rep_begin, int32_t rep_end,
                                   int32_t weighted_classes, int32_t K, double nmax, double* raw) {
  CMB_TRY
  mica_null_core(ctx->c, seed, rep_cpu, rep_ram, rep_begin, rep_end, weighted_classes, K, nmax, raw);
  CMB_CATCH
}

int cmb_mica_null_parametric(cmb_ctx* ctx, uint64_t seed, int32_t rep_cpu, int32_t rep_ram, int32_t weighted_classes, int32_t K,
                             double nmax, double* raw) {
  return cmb_mica_null_parametric_range(ctx, seed, rep_cpu, rep_ram, 0, rep_cpu, weighted_classes, K, nmax, raw);
}

int cmb_mica_null_parametric_sharded(cmb_ctx* ctx, uint64_t seed, int32_t rep_cpu, int32_t rep_ram, int32_t weighted_classes,
                                     int32_t K, double nmax, double* raw) {
  CMB_TRY
  Context& c = ctx->c;
  if (c.comm_size == 1) { // no communicator: the whole null on this GPU
    mica_null_core(c, seed, rep_cpu, rep_ram, 0, rep_cpu, weighted_classes, K, nmax, raw);
    return 0;
  }
  int r0, r1;
  replicate_range(rep_cpu, c.comm_size, c.comm_rank, r0, r1);
  mica_null_core(c, seed, rep_cpu, rep_ram, r0, r1, weighted_classes, 0, 0., raw);
  if (K > 0) gather_null_shards(c, rep_cpu, rep_ram, K, nmax);
  CMB_CATCH
}

int cmb_null_load(cmb_ctx* ctx, const double* stat, const double* key, int64_t n, int32_t K, double kmax) {
  CMB_TRY
  Context& c = ctx->c;
  CMB_CUDA(cudaSetDevice(c.device));
  if (n < 0 || (n > 0 && (!stat || !key))) fail("cmb_null_load: bad arguments");
  NullState& ns = c.null;
  ns.begin(n);
  CMB_CUDA(cudaMemcpyAsync(ns.stat.p, stat, sizeof(double) * n, cudaMemcpyHostToDevice, c.stream));
  CMB_CUDA(cudaMemcpyAsync(ns.nmin.p, key, sizeof(double) * n, cudaMemcpyHostToDevice, c.stream));
  null_load(c, ns.stat.as<double>(), ns.nmin.as<double>(), n, K, kmax);
  CMB_CATCH
}

} // extern "C"
