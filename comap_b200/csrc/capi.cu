// C ABI of libcomap_b200.so (include/comap_b200.h): context, tree/model/alignment setup,
// mapping.  The statistics / null / clustering entry points live in capi_stats.cu.
#include "../../include/comap_b200.h"
#include "context.h"
#include <cmath>
#include <cstring>
#include <string>

namespace cmb {

thread_local std::string g_last_error;

void DevBuf::reserve(size_t bytes) {
  if (bytes <= cap) return;
  release();
  size_t want = align256(bytes);
  cudaError_t e = cudaMalloc(&p, want);
  if (e != cudaSuccess) {
    p = nullptr;
    fail("cudaMalloc of %zu bytes failed: %s", want, cudaGetErrorString(e));
  }
  cap = want;
}
void DevBuf::release() {
  if (p) cudaFree(p);
  p = nullptr;
  cap = 0;
}

void DevStream::upload(const OpStream& s, cudaStream_t st) {
  n_chunks = (uint32_t)s.chunk_off.size();
  cap = (s.chunk_cap + 127) & ~127u;
  bytes.reserve(s.bytes.size());
  off.reserve(sizeof(uint32_t) * n_chunks);
  nbytes.reserve(sizeof(uint32_t) * n_chunks);
  nrec.reserve(sizeof(uint32_t) * n_chunks);
  CMB_CUDA(cudaMemcpyAsync(bytes.p, s.bytes.data(), s.bytes.size(), cudaMemcpyHostToDevice, st));
  CMB_CUDA(cudaMemcpyAsync(off.p, s.chunk_off.data(), sizeof(uint32_t) * n_chunks, cudaMemcpyHostToDevice, st));
  CMB_CUDA(cudaMemcpyAsync(nbytes.p, s.chunk_bytes.data(), sizeof(uint32_t) * n_chunks, cudaMemcpyHostToDevice, st));
  CMB_CUDA(cudaMemcpyAsync(nrec.p, s.chunk_nrec.data(), sizeof(uint32_t) * n_chunks, cudaMemcpyHostToDevice, st));
  n_records = s.n_records;
  stack_depth = s.stack_depth;
  stage_bytes = s.stage_bytes;
  for (int k = 0; k < 3; k++) blk_off_max[k] = s.blk_off_max[k];
  if (!s.aux.empty()) {
    aux.reserve(sizeof(int32_t) * s.aux.size());
    CMB_CUDA(cudaMemcpyAsync(aux.p, s.aux.data(), sizeof(int32_t) * s.aux.size(), cudaMemcpyHostToDevice, st));
  }
  CMB_CUDA(cudaStreamSynchronize(st)); // host vectors may go away
}

// Site counts are padded to whole 256-site blocks, and to an ODD number of them: the row stride
// of every [row][site] matrix (tips, out) is then an odd multiple of 2 KB.  With an even count
// (stride a multiple of 4-8 KB) the 997 rows a pair kernel walks per site land on few DRAM
// channels: k2_paired ran 1.88 ms instead of 1.25 ms per 517 k sites.
int64_t pad_sites(int64_t n) {
  int64_t blocks = (n + 255) / 256;
  if (blocks % 2 == 0) blocks++;
  return blocks * 256;
}

void Context::require_tree_model() const {
  if (!have_tree) fail("no tree: call cmb_set_tree first");
  if (!have_model) fail("no model: call cmb_set_model first");
}

void Context::ensure_streams() {
  require_tree_model();
  if (streams_ready) return;
  build_model_tables(tables, A, Q.data(), pi.data(), C, rates.data(), probs.data(), count_method,
                     have_weights ? weights.data() : nullptr, tree.B, tree.brlen.data());
  var_ready = false;
  check_map_support(A, C);
  // cherries are recomputed instead of stored when their two extra tables per record are
  // small (nucleotides); for A = 20 the records would outgrow the shared-memory budget
  assign_slots(tree, A <= 4);
  // proteins: tensor-core kernels (k1_mma20.cu) unless the tree is so deep that the down pass' shared-memory
  // message stack (10 KB per level) does not fit, or CMB_K1_PROTEIN=scalar asks for the thread-per-site ones
  {
    const char* e = getenv("CMB_K1_PROTEIN");
    protein_mma = A == 20 && !(e && std::string(e) == "scalar") && tree.down_depth <= 12;
  }
  {
    OpStream os;
    if (A == 4) build_down_mma_stream(os, tree, tables); // tensor-core passes (k1_mma.cu)
    else if (protein_mma) build_down_mma20_stream(os, tree, tables);
    else build_down_stream(os, tree, tables, 0, C);
    down_stream.upload(os, stream);
    if (A == 4) build_up_mma_stream(os, tree, tables); // tensor-core up pass (k1_mma.cu)
    else if (protein_mma) build_up_mma20_stream(os, tree, tables, kChunkSites20);
    else build_up_stream(os, tree, tables, 0, std::min(C, kScalarUpClasses));
    up_stream.upload(os, stream);
    if (A == 20 && !protein_mma && C > kScalarUpClasses) { // the rest of the classes, a second up launch
      build_up_stream(os, tree, tables, kScalarUpClasses, C - kScalarUpClasses);
      up_stream_hi.upload(os, stream);
    }
  }
  {
    OpStream os;
    build_sim_stream(os, tree, tables);
    sim_stream.upload(os, stream);
  }
  {
    std::vector<double> ev, R, L, spec;
    build_spectrum(A, Q.data(), pi.data(), ev, R, L);
    spec.insert(spec.end(), ev.begin(), ev.end());
    spec.insert(spec.end(), R.begin(), R.end());
    spec.insert(spec.end(), L.begin(), L.end());
    spec.insert(spec.end(), tree.brlen.begin(), tree.brlen.end());
    d_spec.reserve(sizeof(double) * spec.size());
    CMB_CUDA(cudaMemcpyAsync(d_spec.p, spec.data(), sizeof(double) * spec.size(), cudaMemcpyHostToDevice, stream));
    CMB_CUDA(cudaStreamSynchronize(stream));
  }
  d_pi.reserve(sizeof(double) * A);
  d_rates.reserve(sizeof(double) * C);
  d_probs.reserve(sizeof(double) * C);
  CMB_CUDA(cudaMemcpyAsync(d_pi.p, pi.data(), sizeof(double) * A, cudaMemcpyHostToDevice, stream));
  CMB_CUDA(cudaMemcpyAsync(d_rates.p, rates.data(), sizeof(double) * C, cudaMemcpyHostToDevice, stream));
  CMB_CUDA(cudaMemcpyAsync(d_probs.p, probs.data(), sizeof(double) * C, cudaMemcpyHostToDevice, stream));
  std::vector<uint32_t> ident(256, (A >= 32) ? 0xffffffffu : ((1u << A) - 1u));
  for (int k = 0; k < A; k++) ident[k] = 1u << k;
  d_identity_mask.reserve(sizeof(uint32_t) * 256);
  CMB_CUDA(cudaMemcpyAsync(d_identity_mask.p, ident.data(), sizeof(uint32_t) * 256, cudaMemcpyHostToDevice, stream));
  CMB_CUDA(cudaStreamSynchronize(stream));
  streams_ready = true;
}

MapModel Context::map_model() const {
  MapModel m;
  m.A = A; m.C = C; m.B = tree.B; m.n_slots = tree.n_slots; m.T = tree.n_leaves;
  m.code_mask = d_code_mask.as<uint32_t>();
  m.pi = d_pi.as<double>();
  m.rates = d_rates.as<double>();
  m.probs = d_probs.as<double>();
  m.cont_kind = cont_kind; m.cont_alpha = cont_alpha; m.cont_pinv = cont_pinv;
  m.spec = d_spec.as<double>();
  return m;
}

const double* Context::mean_vector() {
  finish_map();
  if (!mapped) fail("the corrected correlation needs a mapped alignment (cmb_map) for its mean vector");
  if (!have_meanvec) {
    const int B = tree.B;
    d_meanvec.reserve(sizeof(double) * B);
    corr_mean.reserve(sizeof(double) * S_pad);
    corr_sd.reserve(sizeof(double) * S_pad);
    scratch2.reserve(sizeof(double) * S_pad);
    launch_mean_vector(B, S, S_pad, d_out.as<double>(), d_meanvec.as<double>(), stream);
    launch_prep(B, S, S_pad, d_out.as<double>(), d_meanvec.as<double>(), corr_mean.as<double>(), corr_sd.as<double>(),
                scratch2.as<double>(), stream);
    prof.total_launches += 2;
    have_meanvec = true;
  }
  return d_meanvec.as<double>();
}

const double* Context::mi_counts() {
  finish_map();
  if (!mapped) fail("statistic MI needs a mapped alignment (cmb_map)");
  if (!have_mi_count) {
    mi_count.reserve(sizeof(double) * S_pad);
    launch_count_ge(tree.B, S, S_pad, d_out.as<double>(), mi_threshold, mi_count.as<double>(), stream);
    prof.total_launches += 1;
    have_mi_count = true;
  }
  return mi_count.as<double>();
}

void Context::prof_begin(const char* name) {
  if (!prof.enabled) return;
  cudaEvent_t a, b;
  CMB_CUDA(cudaEventCreate(&a));
  CMB_CUDA(cudaEventCreate(&b));
  CMB_CUDA(cudaEventRecord(a, stream));
  prof.pending.emplace_back(name, a, b, 0);
}
void Context::prof_end(int launches) {
  prof.total_launches += launches;
  if (!prof.enabled) return;
  auto& t = prof.pending.back();
  std::get<3>(t) = launches;
  CMB_CUDA(cudaEventRecord(std::get<2>(t), stream));
}
void Context::prof_collect() {
  if (prof.pending.empty()) return;
  CMB_CUDA(cudaStreamSynchronize(stream));
  for (auto& t : prof.pending) {
    float ms = 0.f;
    CMB_CUDA(cudaEventElapsedTime(&ms, std::get<1>(t), std::get<2>(t)));
    auto& e = prof.entries[std::get<0>(t)];
    e.ms += ms;
    e.launches += std::get<3>(t);
    cudaEventDestroy(std::get<1>(t));
    cudaEventDestroy(std::get<2>(t));
  }
  prof.pending.clear();
}

void Context::cancel_map() {
  if (map_pending) CMB_CUDA(cudaEventSynchronize(map_done));
  map_pending = false;
}

// max(norm) for the null's Domain and the saturated-site check of a finished mapping (host copies are in place)
void Context::finalize_map_host() {
  max_norm = 0.;
  for (int64_t i = 0; i < S; i++)
    if (h_norm[i] > max_norm) max_norm = h_norm[i];
  // A site whose likelihood underflowed to 0 (ln L = -inf) has 1/L = inf and NaN vectors.  The reference stops
  // there (CoETools.cpp:233-247) or drops those sites and starts over (remove_saturated_sites, :248-262); the
  // per-site outputs are filled so the caller can find them, and the mapping is refused.
  int64_t n_sat = 0, first_sat = -1;
  for (int64_t i = 0; i < S; i++)
    if (!std::isfinite(h_loglik[i])) { if (!n_sat++) first_sat = i; }
  if (n_sat) {
    mapped = false;
    fail("cmb_map: the likelihood is 0 (log = -inf) at %lld site(s), first at site index %lld: computer underflow, "
         "expected on big data sets (>~500 sequences); remove those sites (input.sequence.remove_saturated_sites = yes)",
         (long long)n_sat, (long long)first_sat);
  }
  mapped = true;
}

void Context::finish_map() {
  if (!map_pending) return;
  CMB_CUDA(cudaEventSynchronize(map_done));
  map_pending = false;
  CMB_CUDA(cudaStreamWaitEvent(stream, map_done, 0)); // later work on the main stream sees the mapping
  finalize_map_host();
}

VariantTables Context::variant_tables() {
  const int n = tree.n_nodes;
  if (!var_ready) {
    std::vector<int32_t> h((size_t)4 * n + 1, 0);
    int32_t *par = h.data(), *off = par + n, *ch = off + n + 1, *leaf = ch + n - 1;
    for (int v = 0; v < n; v++) { par[v] = tree.parent[v]; leaf[v] = tree.leaf_row[v]; }
    for (int v = 0; v < n - 1; v++) off[tree.parent[v] + 1]++;
    for (int v = 0; v < n; v++) off[v + 1] += off[v];
    std::vector<int32_t> fill(off, off + n);
    for (int v = 0; v < n - 1; v++) ch[fill[tree.parent[v]]++] = v; // children in id (= Newick) order
    var_tree.reserve(sizeof(int32_t) * h.size());
    CMB_CUDA(cudaMemcpyAsync(var_tree.p, h.data(), sizeof(int32_t) * h.size(), cudaMemcpyHostToDevice, stream));
    const size_t nt = tables.P.size();
    var_tabs.reserve(sizeof(double) * 2 * nt);
    CMB_CUDA(cudaMemcpyAsync(var_tabs.p, tables.P.data(), sizeof(double) * nt, cudaMemcpyHostToDevice, stream));
    CMB_CUDA(cudaMemcpyAsync(var_tabs.as<double>() + nt, tables.N.data(), sizeof(double) * nt, cudaMemcpyHostToDevice, stream));
    CMB_CUDA(cudaStreamSynchronize(stream)); // h goes out of scope
    var_ready = true;
  }
  VariantTables vt;
  vt.n_nodes = n;
  vt.parent = var_tree.as<int32_t>(); vt.ch_off = vt.parent + n; vt.ch = vt.ch_off + n + 1; vt.leaf_row = vt.ch + n - 1;
  vt.P = var_tabs.as<double>(); vt.N = vt.P + tables.P.size();
  return vt;
}

MapBuffers Context::sim_buffers(int k, int64_t n, int64_t n_pad) {
  const int B = tree.B, T = tree.n_leaves;
  s_tips[k].reserve((size_t)T * n_pad);
  s_D.reserve(sizeof(double) * (size_t)tree.n_slots * C * A * n_pad);
  s_Lc.reserve(sizeof(double) * (size_t)C * n_pad);
  s_invL.reserve(sizeof(double) * n_pad);
  s_loglik.reserve(sizeof(double) * n_pad);
  s_pr[k].reserve(sizeof(double) * n_pad);
  s_rc[k].reserve(sizeof(int32_t) * n_pad);
  s_out[k].reserve(sizeof(double) * (size_t)B * n_pad);
  MapBuffers b;
  b.n = n; b.n_pad = n_pad;
  b.tips = s_tips[k].as<uint8_t>();
  b.D = s_D.as<double>(); b.Lc = s_Lc.as<double>(); b.invL = s_invL.as<double>();
  b.loglik = s_loglik.as<double>(); b.post_rate = s_pr[k].as<double>(); b.rate_class = s_rc[k].as<int32_t>();
  b.out = s_out[k].as<double>();
  return b;
}

void Context::clear_sim_tip_padding(int64_t n, int64_t n_pad) {
  uint8_t* tips = s_tips[0].as<uint8_t>();
  if (s_tips_ptr == tips && s_tips_pad == n_pad && s_tips_n == n) return;
  CMB_CUDA(cudaMemsetAsync(tips, 0, (size_t)tree.n_leaves * n_pad, stream));
  s_tips_ptr = tips; s_tips_pad = n_pad; s_tips_n = n;
}

// Down pass for every class block, site likelihoods, then up pass + contraction.
void Context::run_map(const MapBuffers& b, bool simulated, bool states_only, bool variants) {
  MapModel m = map_model();
  if (simulated) m.code_mask = d_identity_mask.as<uint32_t>();
  m.states_only = simulated && states_only;
  prof_begin("map_down");
  if (protein_mma) {
    if (!launch_map_down_mma20(m, b, down_stream, stream)) fail("mapping down pass: no launch shape fits shared memory for A = 20, C = %d", m.C);
  } else launch_map_down(m, b, down_stream, stream);
  launch_map_finish(m, b, stream);
  prof_end(2);
  prof_begin("map_up");
  if (protein_mma) {
    DevBuf& part = simulated ? k1_part : k1_part_obs; // the observed mapping may run beside a simulated one
    part.reserve(sizeof(double) * (size_t)m.C * m.B * b.n_pad);
    if (!launch_map_up_mma20(m, b, up_stream, part.as<double>(), stream)) fail("mapping up pass: no launch shape fits shared memory for A = 20, C = %d", m.C);
    prof_end(2);
  } else if (m.A == 20 && m.C > kScalarUpClasses) {
    launch_map_up(m, b, up_stream, stream, 0, kScalarUpClasses);
    launch_map_up(m, b, up_stream_hi, stream, kScalarUpClasses, m.C - kScalarUpClasses);
    prof_end(2);
  } else {
    launch_map_up(m, b, up_stream, stream);
    prof_end(1);
  }
  if (variants && map_mode) { // nijt.average = no / nijt.joint = no: the vectors are replaced (k1_variants.cu)
    if (b.n_active) fail("internal: mapping variants need uncompressed batches");
    const VariantTables vt = variant_tables();
    prof_begin("map_variant");
    prof_end(launch_map_variant(m, b, vt, map_mode, simulated ? var_scratch : var_scratch_obs, stream));
  }
}

} // namespace cmb

using namespace cmb;

extern "C" {

const char* cmb_last_error(void) { return g_last_error.c_str(); }
int cmb_version(void) { return 100; }

int cmb_host_alloc(uint64_t bytes, void** out) {
  CMB_TRY
  CMB_CUDA(cudaMallocHost(out, bytes));
  CMB_CATCH
}
int cmb_host_free(void* p) {
  CMB_TRY
  CMB_CUDA(cudaFreeHost(p));
  CMB_CATCH
}

int cmb_ctx_create(int device, void* stream, cmb_ctx** out) {
  CMB_TRY
  int n = 0;
  cudaError_t e = cudaGetDeviceCount(&n);
  if (e != cudaSuccess || n == 0)
    fail("no CUDA device available (%s); comap_b200 has no CPU fallback", cudaGetErrorString(e));
  if (device < 0) CMB_CUDA(cudaGetDevice(&device));
  if (device >= n) fail("device %d out of range (%d devices)", device, n);
  CMB_CUDA(cudaSetDevice(device));
  cmb_ctx* ctx = new cmb_ctx();
  ctx->c.device = device;
  if (stream) ctx->c.stream = (cudaStream_t)stream;
  else {
    CMB_CUDA(cudaStreamCreateWithFlags(&ctx->c.stream, cudaStreamNonBlocking));
    ctx->c.own_stream = true;
  }
  *out = ctx;
  CMB_CATCH
}

int cmb_ctx_destroy(cmb_ctx* ctx) {
  CMB_TRY
  if (!ctx) return 0;
  Context& c = ctx->c;
  cudaSetDevice(c.device);
  cudaStreamSynchronize(c.stream);
  cmb_comm_destroy(ctx);
  if (c.map_stream) { cudaStreamSynchronize(c.map_stream); cudaStreamDestroy(c.map_stream); cudaEventDestroy(c.map_begin); cudaEventDestroy(c.map_done); }
  if (c.h_norm) cudaFreeHost(c.h_norm);
  if (c.h_loglik) cudaFreeHost(c.h_loglik);
  if (c.copy_stream) { cudaStreamSynchronize(c.copy_stream); cudaStreamDestroy(c.copy_stream); }
  if (c.copy_event) cudaEventDestroy(c.copy_event);
  for (auto& t : c.prof.pending) { cudaEventDestroy(std::get<1>(t)); cudaEventDestroy(std::get<2>(t)); }
  if (c.own_stream) cudaStreamDestroy(c.stream);
  delete ctx; // device buffers free themselves
  CMB_CATCH
}

int cmb_sync(cmb_ctx* ctx) {
  CMB_TRY
  CMB_CUDA(cudaStreamSynchronize(ctx->c.stream));
  if (ctx->c.copy_stream) CMB_CUDA(cudaStreamSynchronize(ctx->c.copy_stream));
  if (ctx->c.map_stream) CMB_CUDA(cudaStreamSynchronize(ctx->c.map_stream));
  CMB_CATCH
}

int cmb_set_tree(cmb_ctx* ctx, int32_t n_nodes, const int32_t* parent, const double* brlen) {
  CMB_TRY
  Context& c = ctx->c;
  CMB_CUDA(cudaSetDevice(c.device));
  c.cancel_map();
  build_tree(c.tree, n_nodes, parent, brlen);
  c.have_tree = true;
  c.streams_ready = false;
  c.mapped = false;
  c.have_alignment = false;
  c.null.ready = false;
  CMB_CATCH
}

int cmb_set_model(cmb_ctx* ctx, int32_t A, const double* Q, const double* pi, int32_t C, const double* rates,
                  const double* probs, int32_t count_method, const double* weight_xy) {
  CMB_TRY
  Context& c = ctx->c;
  CMB_CUDA(cudaSetDevice(c.device));
  if (A < 2 || A > 32) fail("cmb_set_model: A must be in 2..32 (got %d)", A);
  if (C < 1 || C > 32) fail("cmb_set_model: C must be in 1..32 (got %d)", C);
  check_map_support(A, C);
  c.cancel_map();
  c.A = A; c.C = C; c.count_method = count_method;
  c.Q.assign(Q, Q + (size_t)A * A);
  c.pi.assign(pi, pi + A);
  c.rates.assign(rates, rates + C);
  c.probs.assign(probs, probs + C);
  c.have_weights = weight_xy != nullptr;
  if (weight_xy) c.weights.assign(weight_xy, weight_xy + (size_t)A * A);
  c.have_model = true;
  c.streams_ready = false;
  c.mapped = false;
  c.null.ready = false;
  if (c.have_tree) c.ensure_streams(); // validates reversibility etc. now
  CMB_CATCH
}

int cmb_set_alignment(cmb_ctx* ctx, int64_t S, const uint8_t* codes, int32_t n_codes, const uint32_t* code_mask) {
  CMB_TRY
  Context& c = ctx->c;
  CMB_CUDA(cudaSetDevice(c.device));
  if (!c.have_tree) fail("cmb_set_alignment: call cmb_set_tree first");
  if (S < 1) fail("cmb_set_alignment: empty alignment");
  if (n_codes < 1 || n_codes > 256) fail("cmb_set_alignment: n_codes must be in 1..256");
  const int T = c.tree.n_leaves;
  c.cancel_map();
  {
    uint8_t worst = 0; // branch-free max over the T*S codes (vectorises); the slow scan only names the culprit
    for (int64_t i = 0; i < (int64_t)T * S; i++) worst = codes[i] > worst ? codes[i] : worst;
    if (worst >= n_codes)
      for (int64_t i = 0; i < (int64_t)T * S; i++)
        if (codes[i] >= n_codes) fail("cmb_set_alignment: code %d out of range at row %lld", codes[i], (long long)(i / S));
  }
  c.S = S;
  c.S_pad = pad_sites(S);
  c.code_mask.assign(256, 0);
  for (int k = 0; k < n_codes; k++) c.code_mask[k] = code_mask[k];
  for (int k = n_codes; k < 256; k++) c.code_mask[k] = code_mask[0];
  c.d_code_mask.reserve(sizeof(uint32_t) * 256);
  CMB_CUDA(cudaMemcpyAsync(c.d_code_mask.p, c.code_mask.data(), sizeof(uint32_t) * 256, cudaMemcpyHostToDevice, c.stream));
  c.d_tips.reserve((size_t)T * c.S_pad);
  CMB_CUDA(cudaMemsetAsync(c.d_tips.p, 0, (size_t)T * c.S_pad, c.stream));
  CMB_CUDA(cudaMemcpy2DAsync(c.d_tips.p, c.S_pad, codes, S, S, T, cudaMemcpyHostToDevice, c.stream));
  CMB_CUDA(cudaStreamSynchronize(c.stream));
  c.have_alignment = true;
  c.mapped = false;
  c.mica_ready = false;
  if (c.null.nmax_from_map) c.null.ready = false;
  CMB_CATCH
}

int cmb_set_map_mode(cmb_ctx* ctx, int32_t average, int32_t joint) {
  CMB_TRY
  Context& c = ctx->c;
  c.cancel_map();
  const int mode = (average ? 0 : 2) + (joint ? 0 : 1);
  if (mode != c.map_mode) { c.mapped = false; c.null.ready = false; c.drop_pair_table(); c.have_dist = false; }
  c.map_mode = mode;
  CMB_CATCH
}

int cmb_ancestral_states(cmb_ctx* ctx, uint8_t* states) {
  CMB_TRY
  Context& c = ctx->c;
  CMB_CUDA(cudaSetDevice(c.device));
  if (!c.have_alignment) fail("cmb_ancestral_states: call cmb_set_alignment first");
  if (!states) fail("cmb_ancestral_states: states is NULL");
  c.finish_map();
  c.ensure_streams();
  const int n = c.tree.n_nodes;
  MapBuffers b;
  b.n = c.S; b.n_pad = c.S_pad; b.tips = c.d_tips.as<uint8_t>();
  c.scratch2.reserve((size_t)n * c.S_pad);
  const VariantTables vt = c.variant_tables();
  c.prof.total_launches += launch_map_variant(c.map_model(), b, vt, 4, c.var_scratch_obs, c.stream, c.scratch2.as<uint8_t>());
  CMB_CUDA(cudaMemcpy2DAsync(states, (size_t)c.S, c.scratch2.p, (size_t)c.S_pad, (size_t)c.S, (size_t)n, cudaMemcpyDeviceToHost, c.stream));
  CMB_CUDA(cudaStreamSynchronize(c.stream));
  CMB_CATCH
}

int cmb_map(cmb_ctx* ctx, double* n_out, double* norm, double* post_rate, int32_t* rate_class, double* loglik) {
  CMB_TRY
  Context& c = ctx->c;
  CMB_CUDA(cudaSetDevice(c.device));
  if (!c.have_alignment) fail("cmb_map: call cmb_set_alignment first");
  c.cancel_map();
  c.mapped = false;
  c.ensure_streams();
  const int64_t S = c.S, Sp = c.S_pad;
  const int A = c.A, C = c.C, B = c.tree.B;
  c.d_D.reserve(sizeof(double) * (size_t)c.tree.n_slots * C * A * Sp);
  c.d_Lc.reserve(sizeof(double) * (size_t)C * Sp);
  c.d_invL.reserve(sizeof(double) * Sp);
  c.d_loglik.reserve(sizeof(double) * Sp);
  c.d_pr.reserve(sizeof(double) * Sp);
  c.d_rc.reserve(sizeof(int32_t) * Sp);
  c.d_out.reserve(sizeof(double) * (size_t)B * Sp);
  c.pairs_mean.reserve(sizeof(double) * Sp);
  c.pairs_sd.reserve(sizeof(double) * Sp);
  c.pairs_norm.reserve(sizeof(double) * Sp);
  if ((size_t)S > c.h_cap) {
    if (c.h_norm) cudaFreeHost(c.h_norm);
    if (c.h_loglik) cudaFreeHost(c.h_loglik);
    c.h_norm = c.h_loglik = nullptr; c.h_cap = 0;
    CMB_CUDA(cudaMallocHost((void**)&c.h_norm, sizeof(double) * S));
    CMB_CUDA(cudaMallocHost((void**)&c.h_loglik, sizeof(double) * S));
    c.h_cap = (size_t)S;
  }
  // no host output asked for: the mapping is only enqueued, on a side stream ordered after what the main
  // stream holds now; the first call that needs it completes it (Context::finish_map)
  const bool deferred = !n_out && !norm && !post_rate && !rate_class && !loglik;
  cudaStream_t main_stream = c.stream;
  struct Restore { Context& c; cudaStream_t s; ~Restore() { c.stream = s; } } restore{c, main_stream};
  if (deferred) {
    if (!c.map_stream) {
      CMB_CUDA(cudaStreamCreateWithFlags(&c.map_stream, cudaStreamNonBlocking));
      CMB_CUDA(cudaEventCreateWithFlags(&c.map_begin, cudaEventDisableTiming));
      CMB_CUDA(cudaEventCreateWithFlags(&c.map_done, cudaEventDisableTiming));
    }
    CMB_CUDA(cudaEventRecord(c.map_begin, main_stream));
    CMB_CUDA(cudaStreamWaitEvent(c.map_stream, c.map_begin, 0));
    c.stream = c.map_stream;
  }
  MapBuffers b;
  b.n = S; b.n_pad = Sp;
  b.tips = c.d_tips.as<uint8_t>();
  b.D = c.d_D.as<double>(); b.Lc = c.d_Lc.as<double>(); b.invL = c.d_invL.as<double>();
  b.loglik = c.d_loglik.as<double>(); b.post_rate = c.d_pr.as<double>(); b.rate_class = c.d_rc.as<int32_t>();
  b.out = c.d_out.as<double>();
  c.run_map(b, false);
  // per-site mean / sd / norm in the reference's summation order (k2_prep); norms are needed
  // on the host by the null (Domain upper bound) and for the caller
  launch_prep(B, S, Sp, b.out, nullptr, c.pairs_mean.as<double>(), c.pairs_sd.as<double>(), c.pairs_norm.as<double>(), c.stream);
  c.have_meanvec = false;
  c.have_mi_count = false;
  c.prof.total_launches += 1;
  CMB_CUDA(cudaMemcpyAsync(c.h_norm, c.pairs_norm.p, sizeof(double) * S, cudaMemcpyDeviceToHost, c.stream));
  if (n_out) {
    c.scratch.reserve(sizeof(double) * (size_t)S * B);
    launch_transpose_out(b.out, B, S, Sp, c.scratch.as<double>(), c.stream);
    c.prof.total_launches += 1;
    CMB_CUDA(cudaMemcpyAsync(n_out, c.scratch.p, sizeof(double) * (size_t)S * B, cudaMemcpyDeviceToHost, c.stream));
  }
  if (post_rate) CMB_CUDA(cudaMemcpyAsync(post_rate, c.d_pr.p, sizeof(double) * S, cudaMemcpyDeviceToHost, c.stream));
  if (rate_class) CMB_CUDA(cudaMemcpyAsync(rate_class, c.d_rc.p, sizeof(int32_t) * S, cudaMemcpyDeviceToHost, c.stream));
  CMB_CUDA(cudaMemcpyAsync(c.h_loglik, c.d_loglik.p, sizeof(double) * S, cudaMemcpyDeviceToHost, c.stream));
  c.have_dist = false;
  c.drop_pair_table(); // resident pair columns belong to the previous mapping
  if (c.null.nmax_from_map) c.null.ready = false; // binned with the previous mapping's max(norm)
  if (deferred) {
    CMB_CUDA(cudaEventRecord(c.map_done, c.map_stream));
    c.map_pending = true;
    return 0;
  }
  CMB_CUDA(cudaStreamSynchronize(c.stream));
  if (loglik) std::memcpy(loglik, c.h_loglik, sizeof(double) * S);
  if (norm) std::memcpy(norm, c.h_norm, sizeof(double) * S);
  c.finalize_map_host();
  CMB_CATCH
}

int cmb_load_vectors(cmb_ctx* ctx, const double* n_in, double* norm) {
  CMB_TRY
  Context& c = ctx->c;
  CMB_CUDA(cudaSetDevice(c.device));
  c.finish_map();
  if (!c.mapped) fail("cmb_load_vectors: call cmb_map first (site likelihoods and rates come from the alignment)");
  if (!n_in) fail("cmb_load_vectors: no vectors given");
  const int64_t S = c.S, Sp = c.S_pad;
  const int B = c.tree.B;
  c.scratch.reserve(sizeof(double) * (size_t)S * B);
  CMB_CUDA(cudaMemcpyAsync(c.scratch.p, n_in, sizeof(double) * (size_t)S * B, cudaMemcpyHostToDevice, c.stream));
  // [S][B] -> [B][S_pad]: the transpose kernel with the two dimensions swapped
  CMB_CUDA(cudaMemsetAsync(c.d_out.p, 0, sizeof(double) * (size_t)B * Sp, c.stream));
  launch_transpose_out(c.scratch.as<double>(), (int)S, B, B, c.d_out.as<double>(), c.stream, Sp);
  launch_prep(B, S, Sp, c.d_out.as<double>(), nullptr, c.pairs_mean.as<double>(), c.pairs_sd.as<double>(),
              c.pairs_norm.as<double>(), c.stream);
  c.prof.total_launches += 2;
  c.have_meanvec = false;
  c.have_mi_count = false;
  CMB_CUDA(cudaMemcpyAsync(c.h_norm, c.pairs_norm.p, sizeof(double) * S, cudaMemcpyDeviceToHost, c.stream));
  CMB_CUDA(cudaStreamSynchronize(c.stream));
  c.max_norm = 0.;
  for (int64_t i = 0; i < S; i++)
    if (c.h_norm[i] > c.max_norm) c.max_norm = c.h_norm[i];
  if (norm) std::memcpy(norm, c.h_norm, sizeof(double) * S);
  c.have_dist = false;
  c.null.ready = false;
  c.drop_pair_table();
  CMB_CATCH
}

int cmb_set_mi_threshold(cmb_ctx* ctx, double threshold) {
  ctx->c.mi_threshold = threshold;
  ctx->c.have_mi_count = false;
  ctx->c.drop_pair_table(); // resident Stat columns were scored with the previous threshold
  return 0;
}

int cmb_set_continuous_rates(cmb_ctx* ctx, int32_t kind, double alpha, double p_invariant) {
  CMB_TRY
  if (kind < 0 || kind > 3) fail("cmb_set_continuous_rates: kind must be 0 (off), 1 (constant), 2 (gamma) or 3 (invariant + gamma)");
  if (kind >= 2 && !(alpha > 0.)) fail("cmb_set_continuous_rates: alpha must be positive");
  if (kind == 3 && !(p_invariant >= 0. && p_invariant < 1.)) fail("cmb_set_continuous_rates: p must be in [0, 1)");
  ctx->c.cont_kind = kind; ctx->c.cont_alpha = alpha; ctx->c.cont_pinv = p_invariant;
  CMB_CATCH
}

int cmb_set_async(cmb_ctx* ctx, int32_t on) {
  ctx->c.async_null = on != 0;
  return 0;
}

int cmb_profile_enable(cmb_ctx* ctx, int32_t on) {
  ctx->c.prof.enabled = on != 0;
  return 0;
}
int cmb_profile_reset(cmb_ctx* ctx) {
  CMB_TRY
  ctx->c.prof_collect();
  ctx->c.prof.entries.clear();
  ctx->c.prof.total_launches = 0;
  ctx->c.prof.sites_simulated = 0;
  ctx->c.s_batches = 0;
  CMB_CATCH
}
int cmb_profile_get(cmb_ctx* ctx, const char* name, double* ms, int64_t* launches) {
  CMB_TRY
  ctx->c.prof_collect();
  if (std::string(name) == "sites_simulated" || std::string(name) == "sites_mapped_null") {
    // counters, returned through `ms`: simulated sites handed to the null's mapping since the reset, and how many
    // of them (varied columns + the A constant patterns per batch) the mapping kernels actually walked
    Context& c = ctx->c;
    double v = (double)c.prof.sites_simulated;
    if (std::string(name) == "sites_mapped_null") {
      if (c.s_batches > 0 && c.s_counts.p) {
        std::vector<int32_t> h(2 * (size_t)c.s_batches);
        CMB_CUDA(cudaMemcpy(h.data(), c.s_counts.p, sizeof(int32_t) * h.size(), cudaMemcpyDeviceToHost));
        v = 0.;
        for (int k = 0; k < c.s_batches; k++) v += h[2 * k];
      }
    }
    if (ms) *ms = v;
    if (launches) *launches = c.s_batches;
    return 0;
  }
  auto it = ctx->c.prof.entries.find(name);
  if (ms) *ms = it == ctx->c.prof.entries.end() ? 0. : it->second.ms;
  if (launches) *launches = it == ctx->c.prof.entries.end() ? 0 : it->second.launches;
  CMB_CATCH
}
int64_t cmb_launch_count(cmb_ctx* ctx) { return ctx->c.prof.total_launches; }

} // extern "C"
