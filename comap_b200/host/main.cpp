// comap_b200 -- CoMap's command line on top of libcomap_b200.so.
//
//   comap_b200 param=options.bpp key=value ... [--seed=N] [--dry-run]
//
// Mirrors the flow of CoMap.cpp:96-737 for the homogeneous, single data set case: same
// option keys (SURVEY.md s5.1), same messages where cheap, same output tables.  Everything
// numerical goes through the C ABI (include/comap_b200.h); there is no CPU fallback.
// --dry-run stops after the inputs are prepared and prints what would be handed to the
// device (used by the CPU tests).
#include "bpp.h"
#include "../../include/comap_b200.h"
#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <fstream>
#include <functional>
#include <iostream>
#include <random>
#include <sstream>
#include <thread>

using namespace host;

namespace {

void display_result(const std::string& what, const std::string& value) {
  std::string w = what;
  while (w.size() < 39) w += '.';
  std::cout << w << ": " << value << std::endl;
}
template <class T> void display_result(const std::string& what, const T& v) {
  std::ostringstream ss;
  ss << v;
  display_result(what, ss.str());
}
void display_message(const std::string& m) { std::cout << m << std::endl; }

void chk(int rc) {
  if (rc) throw Error(std::string("comap_b200: ") + cmb_last_error());
}

// operator<<(double) at default precision == "%g" with 6 significant digits
inline int fmt_g(char* p, double v) { return snprintf(p, 32, "%g", v); }

// Formats rows [r0, r1) with `row(r, buf)` on all host cores and writes them in order:
// 12.5 M "%g" rows are the reference's dominant wall-time term (SURVEY.md s3.1).
template <class F> void write_rows_parallel(std::ostream& out, int64_t n, size_t max_row_bytes, F row) {
  const int nt = (int)std::max(1u, std::min(std::thread::hardware_concurrency(), 32u));
  const int64_t chunk = 1 << 16;
  for (int64_t base = 0; base < n; base += chunk * nt) {
    std::vector<std::string> bufs(nt);
    std::vector<std::thread> th;
    for (int t = 0; t < nt; t++) {
      const int64_t a = base + (int64_t)t * chunk, b = std::min(n, a + chunk);
      if (a >= b) break;
      th.emplace_back([&, t, a, b]() {
        std::string& s = bufs[t];
        s.resize((size_t)(b - a) * max_row_bytes);
        char* p = &s[0];
        for (int64_t r = a; r < b; r++) p += row(r, p);
        s.resize((size_t)(p - &s[0]));
      });
    }
    for (auto& x : th) x.join();
    for (auto& s : bufs) out.write(s.data(), (std::streamsize)s.size());
  }
}

struct Inputs {
  Application app;
  Tree tree;
  Alphabet alpha;
  Alignment aln;
  std::vector<int> cols;      // kept columns (0-based)
  std::vector<int> all_cols;  // before input.remove_const
  Model model;
  RateDist rdist;
  std::vector<uint8_t> codes; // [T][S], rows in leaf order
  std::vector<uint32_t> code_mask;
  int count_method = CMB_COUNT_UNIFORMIZATION;
  bool average = true, joint = true; // nijt.average / nijt.joint (CoETools.cpp:393-394)
  std::vector<double> weights;   // weighted substitution count (nijt=...(weight=...)); empty = unweighted
  bool weights_symmetric = true;
};

std::string data_dir_of(const char* argv0) {
  if (const char* e = getenv("COMAP_B200_DATA")) return e;
  std::string p = argv0;
  size_t k = p.find_last_of('/');
  std::string dir = k == std::string::npos ? "." : p.substr(0, k);
  return dir + "/../data";
}

// Params of the second data set: the keys CoMap reads with the suffix "2" (suffix optional --
// CoETools::readData, CoETools.cpp:91-93; getVectors :374,390; writeInfos :503; the rate
// thresholds :422,435) take the value of KEY2 when it is set.  model / rate_distribution / nijt
// are read without suffix upstream, so both data sets share them.
Params second_data_set_params(const Params& P) {
  Params Q = P;
  for (const auto& kv : P) {
    const std::string& k = kv.first;
    if (k.size() < 2 || k.back() != '2') continue;
    const std::string base = k.substr(0, k.size() - 1);
    if (base == "alphabet" || base.rfind("input.sequence.", 0) == 0 || base.rfind("input.tree.", 0) == 0 ||
        base == "output.vectors.file" || base == "input.vectors.file" || base == "output.infos" ||
        base == "statistic.min_rate_class" || base == "statistic.min_rate")
      Q[base] = kv.second;
  }
  if (P.find("input.tree.file2") == P.end()) Q["input.tree.file"] = "none";            // -> copy of tree 1
  for (const char* k : {"output.vectors.file", "input.vectors.file", "output.infos"})  // never shared
    if (P.find(std::string(k) + "2") == P.end()) Q[k] = "none";
  return Q;
}

// with_model = false (mica without use_model, Mica.cpp:186-199): no tree, model or counts are read; the alignment's
// sequences hang off a star tree so that the library knows the rows
void prepare(Inputs& in, const char* argv0, const Params* override_params = nullptr, const Tree* first_tree = nullptr,
             bool with_model = true) {
  const Params& P = override_params ? *override_params : in.app.params;
  display_message(first_tree ? "\nLoading second dataset...\n" : "\n\n-*- Retrieve data and model -*-\n");
  // tree (PhylogeneticsApplicationTools::getTree, CoMap.cpp:125-129; second data set: CoMap.cpp:238-252)
  std::string tree_path = get_path(P, "input.tree.file", "none");
  if (!with_model) {
  } else if (tree_path == "none" && first_tree) in.tree = *first_tree; // "Copy tree."
  else {
    if (tree_path == "none") throw Error("input.tree.file is not set");
    std::string tfmt = get_string(P, "input.tree.format", "Newick");
    if (lower(parse_procedure(tfmt).name) != "newick") throw Error("input.tree.format '" + tfmt + "' is not supported (Newick)");
    display_result("Input tree file ", tree_path);
    in.tree = parse_newick(read_file(tree_path));
    if (first_tree && in.tree.parent != first_tree->parent)
      throw Error("The second tree must have the same topology as the first tree.");
  }
  if (with_model) {
    display_result("Number of leaves", in.tree.leaves.size());
    display_result("Number of sons at root", in.tree.n_root_children);
    if (in.tree.was_unrooted) display_message("WARNING!!! Tree has been unrooted.");
  }
  // data (CoETools::readData, CoETools.cpp:78-124)
  in.alpha = make_alphabet(get_string(P, "alphabet", "DNA"));
  display_result("Alphabet type ", in.alpha.name);
  std::string seq_path = get_path(P, "input.sequence.file", "none");
  if (seq_path == "none") throw Error("input.sequence.file is not set");
  std::string sfmt = get_string(P, "input.sequence.format", "Fasta");
  in.aln = read_alignment(seq_path, sfmt);
  display_result("Sequence file ", seq_path);
  in.cols = select_sites(in.aln, in.alpha, P, sfmt, &in.all_cols);
  if (!with_model) {
    const int T = (int)in.aln.names.size();
    if (T < 2) throw Error("at least two sequences are needed");
    in.tree = Tree();
    in.tree.parent.assign(T + 1, T); in.tree.parent[T] = -1;
    in.tree.brlen.assign(T + 1, 0.1); in.tree.brlen[T] = 0.;
    in.tree.name = in.aln.names; in.tree.name.push_back("");
    for (int v = 0; v < T; v++) in.tree.leaves.push_back(v);
    in.tree.n_root_children = T;
  }
  if (with_model && get_string(P, "nonhomogeneous", "no") != "no")
    throw Error("nonhomogeneous models are outside the B200 hot path (SURVEY.md s2.1); use nonhomogeneous=no");
  if (with_model) {
  in.model = make_model(get_string(P, "model", "JC69"), in.alpha, data_dir_of(argv0));
  display_result("Substitution model", in.model.name);
  if (!in.model.warning.empty()) display_message(in.model.warning);
  in.rdist = make_rate_distribution(get_string(P, "rate_distribution", "Constant()"));
  display_result("Rate distribution", in.rdist.name);
  display_result("Number of classes", in.rdist.rates.size());
  std::string opt = get_string(P, "optimization", "None");
  if (lower(parse_procedure(opt).name) != "none" && !opt.empty())
    display_message("WARNING!!! optimization=" + opt + " is outside the B200 hot path: parameters are used as given.");
  // nijt (PhylogeneticsApplicationTools::getSubstitutionCount, CoMap.cpp:152)
  std::string nijt = get_string(P, "nijt", "Uniformization");
  if (nijt.empty()) nijt = "Uniformization";
  Procedure nj = parse_procedure(nijt);
  if (nj.name == "Uniformization") in.count_method = CMB_COUNT_UNIFORMIZATION;
  else if (nj.name == "Decomposition") in.count_method = CMB_COUNT_DECOMPOSITION;
  else if (nj.name == "Naive") in.count_method = CMB_COUNT_NAIVE;
  else if (nj.name == "Laplace") { // Laplace(trunc=10): LaplaceSubstitutionCount, unweighted
    int trunc = atoi(get_string(nj.args, "trunc", "10").c_str());
    if (trunc < 2 || trunc > 20) throw Error("nijt=Laplace: trunc must be in 2..20");
    if (get_string(nj.args, "weight", "None") != "None") throw Error("nijt=Laplace does not take weights");
    in.count_method = CMB_COUNT_LAPLACE_TRUNC(trunc);
  }
  else if (nj.name == "Label") { // LabelSubstitutionCount: one label per substitution type (for statistic=MI)
    if (get_string(nj.args, "weight", "None") != "None") throw Error("nijt=Label does not take weights");
    in.count_method = CMB_COUNT_LABEL;
  }
  else if (nj.name == "ProbOneJump") { // OneJumpSubstitutionCount: P(at least one substitution on the branch | its ends)
    if (get_string(nj.args, "weight", "None") != "None") throw Error("nijt=ProbOneJump does not take weights");
    in.count_method = CMB_COUNT_ONE_JUMP;
  }
  else throw Error("nijt=" + nj.name + " is not available in this build (Uniformization, Decomposition, Naive, Laplace, Label, ProbOneJump)");
  in.weights = make_count_weights(get_string(nj.args, "weight", "None"), in.alpha, &in.weights_symmetric, data_dir_of(argv0));
  if (!in.weights.empty()) display_result("Substitution count weights", get_string(nj.args, "weight", "None"));
  in.average = get_bool(P, "nijt.average", true); // "really for benchmarking only" upstream; k1_variants.cu here
  in.joint = get_bool(P, "nijt.joint", true);
  if (!in.average || !in.joint) display_result("Mapping variant", std::string(in.average ? "average" : "no averaging") + (in.joint ? ", joint pair" : ", marginal"));
  display_result("Substitution count", nj.name);
  }
  // leaf rows: sequence of every leaf, in leaf id order
  std::map<std::string, int> row;
  for (size_t i = 0; i < in.aln.names.size(); i++) row[in.aln.names[i]] = (int)i;
  const size_t T = in.tree.leaves.size(), S = in.cols.size();
  if (S == 0) throw Error("no site left to analyse after filtering");
  std::map<char, int> code_of;
  in.code_mask.clear();
  for (size_t k = 0; k < in.alpha.states.size(); k++) in.code_mask.push_back(1u << k);
  in.codes.assign(T * S, 0);
  for (size_t k = 0; k < T; k++) {
    const std::string& nm = in.tree.name[in.tree.leaves[k]];
    auto it = row.find(nm);
    if (it == row.end()) throw Error("leaf '" + nm + "' of the tree has no sequence in the alignment");
    const std::string& s = in.aln.seqs[it->second];
    for (size_t j = 0; j < S; j++) {
      char c = s[in.cols[j]];
      uint32_t m = in.alpha.mask_of(c);
      int code;
      if (m && !(m & (m - 1)) && c != '-') code = __builtin_ctz(m);
      else {
        auto f = code_of.find((char)toupper((unsigned char)c));
        if (f == code_of.end()) {
          if (in.code_mask.size() >= 256) throw Error("too many distinct ambiguity characters");
          code = (int)in.code_mask.size();
          code_of[(char)toupper((unsigned char)c)] = code;
          in.code_mask.push_back(m);
        } else code = f->second;
      }
      in.codes[k * S + j] = (uint8_t)code;
    }
  }
  display_result("Number of sites in file", in.aln.length());
  display_result("Number of sites to analyse", S);
}

void dry_run_dump(const Inputs& in) {
  std::cout.precision(17);
  std::cout << "DRYRUN n_nodes " << in.tree.parent.size() << "\n";
  std::cout << "DRYRUN parent";
  for (int p : in.tree.parent) std::cout << ' ' << p;
  std::cout << "\nDRYRUN brlen";
  for (double b : in.tree.brlen) std::cout << ' ' << b;
  std::cout << "\nDRYRUN leaves";
  for (int l : in.tree.leaves) std::cout << ' ' << in.tree.name[l];
  std::cout << "\nDRYRUN sequences";          // the alignment's own order (mica without a model keeps it)
  for (auto& n : in.aln.names) std::cout << ' ' << n;
  std::cout << "\nDRYRUN A " << in.model.A << "\nDRYRUN Q";
  for (double q : in.model.Q) std::cout << ' ' << q;
  std::cout << "\nDRYRUN pi";
  for (double q : in.model.pi) std::cout << ' ' << q;
  std::cout << "\nDRYRUN rates";
  for (double q : in.rdist.rates) std::cout << ' ' << q;
  std::cout << "\nDRYRUN probs";
  for (double q : in.rdist.probs) std::cout << ' ' << q;
  std::cout << "\nDRYRUN coords";
  for (int c : in.cols) std::cout << ' ' << c + 1;
  std::cout << "\nDRYRUN code_mask";
  for (uint32_t m : in.code_mask) std::cout << ' ' << m;
  std::cout << "\nDRYRUN codes";
  for (uint8_t c : in.codes) std::cout << ' ' << (int)c;
  std::cout << "\nDRYRUN count_method " << in.count_method;
  std::cout << "\nDRYRUN map_mode " << in.average << " " << in.joint;
  std::cout << "\nDRYRUN weights";
  for (double x : in.weights) std::cout << ' ' << x;
  std::cout << std::endl;
}

int stat_id_of(const Params& P, const Inputs& in) {
  Procedure st = parse_procedure(get_string(P, "statistic", "Correlation"));
  if (st.name == "Cosinus") return CMB_STAT_COSINUS;
  if (st.name == "Correlation") return CMB_STAT_CORRELATION;
  if (st.name == "Covariance") return CMB_STAT_COVARIANCE;
  if (st.name == "Cosubstitution") return CMB_STAT_COSUBSTITUTION;
  if (st.name == "Compensation") { // CoETools.cpp:564-574
    if (in.weights.empty())
      throw Error("Compensation distance must be used with a mapping procedure with weights, e.g. "
                  "'nijt=Uniformization(weight=Diff(index1=Volume, symmetrical=no))'.");
    if (in.weights_symmetric)
      throw Error("Compensation distance must be used with a mapping procedure allowing non-symmetric weights, e.g. "
                  "'nijt=Uniformization(weight=Diff(index1=Volume, symmetrical=no))'.");
    return CMB_STAT_COMPENSATION;
  }
  if (st.name == "CorrectedCorrelation") return CMB_STAT_CORRECTED_CORRELATION; // mean vector: CoMap.cpp:350-359
  if (st.name == "MI") { // CoETools.cpp:576-596
    std::string nj = get_string(P, "nijt", "Label"); // upstream compares the raw option string, default "Label"
    if (nj == "Label") {
      if (in.average) throw Error("MI distance with 'nijt=Label' can't be used with 'nijt.average=yes'.");
      return CMB_STAT_MI_LABEL; // bounds -0.5, 0.5, ...: one category per substitution label
    }
    return CMB_STAT_MI;
  }
  throw Error("Unknown statistic used: " + get_string(P, "statistic", ""));
}

std::string group_string(const int32_t* m, int64_t n, const std::vector<int>* coords) {
  std::string s = "[";
  for (int64_t i = 0; i < n; i++) {
    if (i) s += ';';
    s += std::to_string(coords ? (*coords)[m[i]] + 1 : m[i]);
  }
  return s + "]";
}

// Newick of the clustering dendrogram with leaf names translated to coordinates
// (ClusterTools::translate + Newick::writeTree, CoMap.cpp:553-561)
std::string dendrogram_newick(const std::vector<int32_t>& left, const std::vector<int32_t>& right,
                              const std::vector<double>& height, int64_t S, const std::vector<int>& cols) {
  std::vector<std::string> txt(2 * S - 1);
  auto h = [&](int v) { return v < S ? 0. : height[v - S]; };
  for (int64_t v = 0; v < S; v++) txt[v] = std::to_string(cols[v] + 1);
  for (int64_t k = 0; k + 1 < S; k++) {
    int l = left[k], r = right[k];
    std::ostringstream ss;
    ss << "(" << txt[l] << ":" << (height[k] - h(l)) << "," << txt[r] << ":" << (height[k] - h(r)) << ")";
    txt[S + k] = ss.str();
    txt[l].clear();
    txt[r].clear();
  }
  return txt[2 * S - 2] + ";";
}

// comap_b200.gpus = N: N contexts on devices 0..N-1 joined by one NCCL communicator (cmb_comm_init_all), driven by
// one host thread each.  Context 0 is the data set's own; the others hold the same tree / model / alignment and
// map it themselves (a 5000-site mapping is cheaper than shipping its 40 MB).
template <class F> void on_all(int n, F f) {
  std::vector<std::thread> th;
  std::vector<std::string> err(n);
  for (int r = 0; r < n; r++)
    th.emplace_back([&, r] {
      try { f(r); } catch (const std::exception& e) { err[r] = e.what(); if (err[r].empty()) err[r] = "error"; }
    });
  for (auto& t : th) t.join();
  for (auto& e : err)
    if (!e.empty()) throw Error(e);
}

struct Mapped {           // a data set on the device and its per-site results
  cmb_ctx* ctx = nullptr;
  std::vector<double> norm, pr, ll;
  std::vector<int32_t> rc;
};

// cmb_set_* + CoETools::getVectors (CoETools.cpp:364-413) + norms (CoMap.cpp:158-163) + writeInfos
// (CoETools.cpp:496-531) for one data set; P holds that data set's view of the options
Mapped map_data_set(Inputs& in, const Params& P, const std::string& suffix) {
  Mapped m;
  int64_t S = (int64_t)in.cols.size();
  const int B = (int)in.tree.parent.size() - 1;
  chk(cmb_ctx_create(-1, nullptr, &m.ctx));
  chk(cmb_set_tree(m.ctx, (int32_t)in.tree.parent.size(), in.tree.parent.data(), in.tree.brlen.data()));
  chk(cmb_set_model(m.ctx, in.model.A, in.model.Q.data(), in.model.pi.data(), (int32_t)in.rdist.rates.size(),
                    in.rdist.rates.data(), in.rdist.probs.data(), in.count_method,
                    in.weights.empty() ? nullptr : in.weights.data()));
  chk(cmb_set_map_mode(m.ctx, in.average, in.joint));
  chk(cmb_set_alignment(m.ctx, S, in.codes.data(), (int32_t)in.code_mask.size(), in.code_mask.data()));
  {
    Procedure st = parse_procedure(get_string(P, "statistic", "Correlation"));
    if (st.name == "MI") chk(cmb_set_mi_threshold(m.ctx, get_double(st.args, "threshold", 0.99)));
  }
  const std::string in_vec = get_path(P, "input.vectors.file", "none");
  std::string vec_path = get_path(P, "output.vectors.file", "none");
  if (in_vec != "none") vec_path = "none"; // CoETools.cpp:374-390: vectors are read OR computed (+ written)
  else display_result("Output mapping to file" + suffix, vec_path);
  std::vector<double> n_out;
  m.norm.resize(S); m.pr.resize(S); m.ll.resize(S); m.rc.resize(S);
  if (vec_path != "none") n_out.resize((size_t)S * B);
  if (cmb_map(m.ctx, n_out.empty() ? nullptr : n_out.data(), m.norm.data(), m.pr.data(), m.rc.data(), m.ll.data())) {
    // a site likelihood of 0 (CoETools.cpp:233-262): stop with the per-site log-likelihoods written out, or with
    // input.sequence.remove_saturated_sites = yes drop those sites and map again
    int64_t n_sat = 0;
    for (int64_t i = 0; i < S; i++) n_sat += !std::isfinite(m.ll[i]);
    if (!n_sat) throw Error(cmb_last_error());
    if (!get_bool(P, "input.sequence.remove_saturated_sites", false)) {
      std::ofstream debug("DEBUG_likelihoods.txt");
      for (int64_t i = 0; i < S; i++) debug << "Position " << in.cols[i] + 1 << " = " << m.ll[i] << std::endl;
      debug.close();
      std::cerr << "ERROR!!! !!! Site-specific likelihood have been written in file DEBUG_likelihoods.txt ." << std::endl;
      std::cerr << "ERROR!!! !!! 0 values (inf in log) may be due to computer overflow, particularily if datasets are big (>~500 sequences)." << std::endl;
      std::cerr << "ERROR!!! !!! You may want to try input.sequence.remove_saturated_sites = yes to ignore positions with likelihood 0." << std::endl;
      exit(1);
    }
    const int64_t T = (int64_t)in.codes.size() / S;
    std::vector<int64_t> keep;
    for (int64_t i = S; i > 0; --i)
      if (!std::isfinite(m.ll[i - 1])) display_result("Ignore saturated site", std::to_string(in.cols[i - 1] + 1));
    for (int64_t i = 0; i < S; i++)
      if (std::isfinite(m.ll[i])) keep.push_back(i);
    const int64_t S2 = (int64_t)keep.size();
    display_result("Number of sites retained", std::to_string(S2));
    if (S2 == 0) throw Error("Likelihood is still 0 after saturated sites are removed! Looks like a bug...");
    std::vector<uint8_t> codes2((size_t)T * S2);
    std::vector<int> cols2(S2);
    for (int64_t t = 0; t < T; t++)
      for (int64_t k = 0; k < S2; k++) codes2[(size_t)t * S2 + k] = in.codes[(size_t)t * S + keep[k]];
    for (int64_t k = 0; k < S2; k++) cols2[k] = in.cols[keep[k]];
    in.codes.swap(codes2);
    in.cols.swap(cols2);
    S = S2;
    chk(cmb_set_alignment(m.ctx, S, in.codes.data(), (int32_t)in.code_mask.size(), in.code_mask.data()));
    m.norm.resize(S); m.pr.resize(S); m.ll.resize(S); m.rc.resize(S);
    if (vec_path != "none") n_out.resize((size_t)S * B);
    chk(cmb_map(m.ctx, n_out.empty() ? nullptr : n_out.data(), m.norm.data(), m.pr.data(), m.rc.data(), m.ll.data()));
  }
  if (in_vec != "none") {
    // restart from a mapping file (LegacySubstitutionMappingTools::readFromStream, CoETools.cpp:376-384):
    // header "Branches\tMean\tSite<coord>...", one row per branch: id, length, the branch's entry per site
    display_result("Substitution mapping in file" + suffix, in_vec);
    std::ifstream vf(in_vec);
    if (!vf) throw Error("input.vectors.file: cannot open '" + in_vec + "'");
    std::string line;
    std::getline(vf, line);
    std::istringstream hs(line);
    std::string tok;
    int64_t n_cols = 0;
    while (std::getline(hs, tok, '\t')) n_cols++;
    if (n_cols != S + 2)
      throw Error("input.vectors.file: " + std::to_string(n_cols - 2) + " sites in the mapping file, " + std::to_string(S) +
                  " sites to analyse");
    std::vector<double> n_in((size_t)S * B);
    for (int b = 0; b < B; b++) {
      if (!std::getline(vf, line)) throw Error("input.vectors.file: " + std::to_string(b) + " branches in the file, tree has " + std::to_string(B));
      std::istringstream ls(line);
      std::getline(ls, tok, '\t'); // branch id
      std::getline(ls, tok, '\t'); // branch length
      for (int64_t s2 = 0; s2 < S; s2++) {
        if (!std::getline(ls, tok, '\t')) throw Error("input.vectors.file: short row for branch " + std::to_string(b));
        n_in[(size_t)s2 * B + b] = std::stod(tok);
      }
    }
    chk(cmb_load_vectors(m.ctx, n_in.data(), m.norm.data()));
  }
  if (vec_path != "none") {
    // LegacySubstitutionMappingTools::writeToStream (CoETools.cpp:408-412)
    std::ofstream out(vec_path);
    out << "Branches\tMean";
    for (int c : in.cols) out << "\tSite" << c + 1;
    out << "\n";
    for (int b = 0; b < B; b++) {
      out << b << "\t" << in.tree.brlen[b];
      for (int64_t s = 0; s < S; s++) out << "\t" << n_out[(size_t)s * B + b];
      out << "\n";
    }
  }
  std::string infos = get_path(P, "output.infos", "none");
  if (infos != "none") {
    display_result("Alignment information logfile", infos);
    std::ofstream out(infos);
    out << "Group\tIsComplete\tIsConstant\tRC\tPR\tN\tlogLn" << std::endl;
    for (int64_t i = 0; i < S; i++)
      out << "[" << in.cols[i] + 1 << "]\t" << (site_is_complete(in.aln, in.alpha, in.cols[i]) ? 1 : 0) << "\t"
          << (site_is_constant(in.aln, in.alpha, in.cols[i]) ? 1 : 0) << "\t" << m.rc[i] << "\t" << m.pr[i] << "\t"
          << m.norm[i] << "\t" << m.ll[i] << std::endl;
  }
  return m;
}

// ---------------------------------------------------------------------------------------------------------------
// mica param=FILE key=value ...   (CoMap/Mica.cpp:132-704): mutual information between alignment columns, optionally
// conditioned on the norms of a substitution mapping (use_model = yes), with a null distribution by parametric or
// nonparametric bootstrap, by the z-score method, or none.  Same option keys, messages where cheap, same table.
// null.method = permutations (miTest, Mica.cpp:92-118) runs on the device too (cmb_mica_permutations); upstream's shuffles
// come from an unseeded generator, here they are a function of --seed.
int mica_main(Inputs& in, const char* argv0) {
  const Params& P = in.app.params;
  const bool with_model = get_bool(P, "use_model", false);
  prepare(in, argv0, nullptr, nullptr, with_model);
  display_result("Number of sequences", in.aln.names.size());
  display_result("Number of sites", in.cols.size());
  display_message(std::string("Model of sequence evolution............: ") + (with_model ? "yes" : "no"));
  const int64_t S = (int64_t)in.cols.size();
  if (S < 2) throw Error("at least two sites are needed");
  uint64_t seed = in.app.seed;
  if (!in.app.seed_given) seed = ((uint64_t)std::random_device{}() << 32) ^ std::random_device{}();
  // a context on `device` (-1: the current one) holding the tree, the model and the alignment
  auto load = [&](int device) {
    cmb_ctx* c = nullptr;
    chk(cmb_ctx_create(device, nullptr, &c));
    chk(cmb_set_tree(c, (int32_t)in.tree.parent.size(), in.tree.parent.data(), in.tree.brlen.data()));
    if (with_model) { // Mica.cpp:303-339: likelihood, then the mapping (Uniformization, total counts) for the norms
      chk(cmb_set_model(c, in.model.A, in.model.Q.data(), in.model.pi.data(), (int32_t)in.rdist.rates.size(),
                        in.rdist.rates.data(), in.rdist.probs.data(), CMB_COUNT_UNIFORMIZATION, nullptr));
    } else { // the library wants a model before it takes an alignment; a uniform one, never used
      const int A = (int)in.alpha.states.size();
      std::vector<double> Q((size_t)A * A, 1. / (A - 1)), pi(A, 1. / A);
      for (int x = 0; x < A; x++) Q[(size_t)x * A + x] = -1.;
      const double one = 1.;
      chk(cmb_set_model(c, A, Q.data(), pi.data(), 1, &one, &one, CMB_COUNT_NAIVE, nullptr));
    }
    chk(cmb_set_alignment(c, S, in.codes.data(), (int32_t)in.code_mask.size(), in.code_mask.data()));
    return c;
  };
  cmb_ctx* ctx = load(-1);
  std::vector<double> norms;
  if (with_model) {
    norms.resize(S);
    chk(cmb_map(ctx, nullptr, norms.data(), nullptr, nullptr, nullptr));
  }
  // comap_b200.gpus = N: the permutation test's pairs and the parametric bootstrap's replicates are spread over
  // contexts on devices 0..N-1 holding the same tree, model and alignment; the other null methods build their samples
  // on the host and, like the table, stay on context 0
  const int n_gpus = (int)get_int(P, "comap_b200.gpus", 1);
  if (n_gpus < 1) throw Error("comap_b200.gpus must be at least 1");
  const std::string method = get_string(P, "null.method", "none");
  const bool parametric = method == "parametric-bootstrap";
  std::vector<cmb_ctx*> ctxs{ctx};
  if (n_gpus > 1 && (method == "permutations" || (parametric && with_model))) {
    display_result("GPUs", n_gpus);
    ctxs.resize(n_gpus, nullptr);
    on_all(n_gpus, [&](int r) {
      if (r == 0) return;
      ctxs[r] = load(r);
      if (parametric) chk(cmb_map(ctxs[r], nullptr, nullptr, nullptr, nullptr, nullptr));
    });
    if (parametric) chk(cmb_comm_init_all(ctxs.data(), n_gpus));
  }
  const int n_dev = (int)ctxs.size();
  const std::string path = get_path(P, "output.file", "none");
  if (path == "none") throw Error("output.file is not set");
  display_result("Output file", path);
  display_message("Computing average MIs..................: ");
  std::vector<double> entropy(S), average(S);
  chk(cmb_mica_sites(ctx, entropy.data(), average.data()));
  double full_average = 0.;
  for (double a : average) full_average += a;
  full_average /= (double)S; // VectorTools::mean
  const int64_t n_pairs = S * (S - 1) / 2;
  std::vector<int32_t> I(n_pairs), J(n_pairs), nsim(n_pairs, 0);
  std::vector<double> mi(n_pairs), hj(n_pairs), hm(n_pairs), nm(n_pairs), pv(n_pairs);
  int64_t rows = 0;
  const int key = with_model ? CMB_MICA_KEY_NMIN : CMB_MICA_KEY_HMIN;

  // null distribution (Mica.cpp:369-628)
  display_result("Null distribution", method);
  bool compute_p = false;
  int64_t max_perm = 0;
  if (method != "none") {
    if (method == "z-score") compute_p = true;
    else if (method == "permutations") compute_p = false;
    else compute_p = get_bool(P, "null.compute_pvalues", true);
    int K = 0;
    double kmax = 0.;
    if (compute_p) {
      K = (int)get_int(P, "null.nb_rate_classes", 10);
      display_result("Number of sub-distributions", K);
      if (K < 1) throw Error("Domain: number of classes must be > 0"); // Domain.cpp:49
      const std::vector<double>& v = with_model ? norms : entropy;
      for (double x : v) kmax = x > kmax ? x : kmax;
    }
    const std::string simpath = get_path(P, "null.output.file", "none");
    const bool to_file = simpath != "none" && !simpath.empty();
    const int rep_cpu = (int)get_int(P, "null.nb_rep_CPU", 10), rep_ram = (int)get_int(P, "null.nb_rep_RAM", 100);
    if (method == "nonparametric-bootstrap") { // :401-468: pairs of sites resampled with replacement
      display_message("Computing null distribution............: ");
      const int64_t n = (int64_t)rep_cpu * rep_ram;
      std::mt19937_64 gen(seed);
      std::vector<int32_t> a(n), b(n);
      for (int r = 0; r < rep_cpu; r++) { // sampleSites twice per outer replicate
        for (int j = 0; j < rep_ram; j++) a[(size_t)r * rep_ram + j] = (int32_t)(gen() % (uint64_t)S);
        for (int j = 0; j < rep_ram; j++) b[(size_t)r * rep_ram + j] = (int32_t)(gen() % (uint64_t)S);
      }
      std::vector<double> smi(n), shj(n), skey(n);
      chk(cmb_mica_pair_list(ctx, n, a.data(), b.data(), smi.data(), shj.data()));
      std::vector<double> shm(n), snm(n);
      for (int64_t r = 0; r < n; r++) {
        shm[r] = std::min(entropy[a[r]], entropy[b[r]]);
        if (with_model) snm[r] = std::min(norms[a[r]], norms[b[r]]);
        skey[r] = with_model ? snm[r] : shm[r];
      }
      if (to_file) {
        display_result("Null output file", simpath);
        std::ofstream so(simpath);
        so << "MI\tHjoint\tHmin" << (with_model ? "\tNmin" : "") << std::endl;
        for (int64_t r = 0; r < n; r++) {
          so << smi[r] << "\t" << shj[r] << "\t" << shm[r];
          if (with_model) so << "\t" << snm[r];
          so << std::endl;
        }
      }
      if (compute_p) chk(cmb_null_load(ctx, smi.data(), skey.data(), n, K, kmax));
    } else if (method == "parametric-bootstrap") { // :470-545
      if (!with_model) throw Error("You need to specify a model of sequence evolution in order to use a parametric bootstrap approach!");
      const bool continuous_sim = get_bool(P, "simulations.continuous", false);
      display_result("Rate distribution for simulations", continuous_sim ? "continuous" : "discrete");
      if (continuous_sim) {
        if (in.rdist.cont_kind == 0) throw Error("simulations.continuous=yes is available for Constant, Gamma and Invariant(dist=Gamma) rate distributions");
        for (cmb_ctx* c : ctxs) chk(cmb_set_continuous_rates(c, in.rdist.cont_kind, in.rdist.alpha, in.rdist.p_inv));
      }
      display_message("Computing null distribution............: ");
      const int64_t n = (int64_t)rep_cpu * rep_ram;
      std::vector<double> raw(to_file ? (size_t)n * 3 : 0);
      const int weighted = get_bool(P, "simulations.weighted_classes", false) ? 1 : 0;
      if (n_dev == 1)
        chk(cmb_mica_null_parametric(ctx, seed, rep_cpu, rep_ram, weighted, compute_p ? K : 0, kmax, to_file ? raw.data() : nullptr));
      else // outer replicates sharded over the GPUs; rank r's rows start at its first replicate
        on_all(n_dev, [&](int r) {
          const int q = rep_cpu / n_dev, m = rep_cpu % n_dev, r0 = r * q + std::min(r, m);
          chk(cmb_mica_null_parametric_sharded(ctxs[r], seed, rep_cpu, rep_ram, weighted, compute_p ? K : 0, kmax,
                                               to_file ? raw.data() + (size_t)r0 * rep_ram * 3 : nullptr));
        });
      if (to_file) {
        display_result("Null output file", simpath);
        std::ofstream so(simpath);
        so << "MI\tHjoint\tHmin\tNmin" << std::endl;
        for (int64_t r = 0; r < n; r++) { // upstream indexes the OBSERVED entropies by (replicate, site in replicate), Mica.cpp:526
          const int64_t i = r / rep_ram, j = r % rep_ram;
          const double h = (i < S && j < S) ? std::min(entropy[i], entropy[j]) : std::nan("");
          so << raw[r * 3] << "\t" << raw[r * 3 + 1] << "\t" << h << "\t" << raw[r * 3 + 2] << std::endl;
        }
      }
    } else if (method == "z-score") { // :546-606: the distribution of all the observed pairs, corrected or not
      const std::string zs = get_string(P, "null.method_zscore.stat", "MIp");
      display_result("Compute p-value for", zs);
      if (zs != "MIp" && zs != "MIc" && zs != "MI") throw Error("Unkown statistic, should be 'MI', 'MIp' or 'MIc'.");
      display_message("Computing total distribution...........: ");
      chk(cmb_mica_pairs(ctx, key, 0, n_pairs, I.data(), J.data(), mi.data(), hj.data(), hm.data(), nm.data(), nullptr, nullptr, &rows));
      std::vector<double> st(n_pairs), kk(n_pairs);
      for (int64_t r = 0; r < n_pairs; r++) {
        const double apc = average[I[r]] * average[J[r]] / full_average, rcw = average[I[r]] * average[J[r]] / 2.;
        st[r] = zs == "MIp" ? mi[r] - apc : zs == "MIc" ? mi[r] / rcw : mi[r];
        kk[r] = with_model ? nm[r] : hm[r];
      }
      chk(cmb_null_load(ctx, st.data(), kk.data(), n_pairs, K, kmax));
    } else if (method == "permutations") { // :608-619, miTest :92-118
      max_perm = get_int(P, "null.max_number_of_permutations", 1000);
      if (max_perm <= 0) throw Error("Permutation number should be greater than 0!");
      display_result("Maximum number of permutations", max_perm);
    } else throw Error("Unvalid null distribution method specified: " + method);
  }

  // the table (Mica.cpp:630-689)
  display_message("Computing all MI scores................: ");
  chk(cmb_mica_pairs(ctx, key, compute_p ? 1 : 0, n_pairs, I.data(), J.data(), mi.data(), hj.data(), hm.data(), nm.data(),
                     compute_p ? pv.data() : nullptr, compute_p ? nsim.data() : nullptr, &rows));
  std::vector<double> perm_p;
  std::vector<int32_t> perm_nb;
  if (max_perm > 0) {
    perm_p.resize(n_pairs); perm_nb.resize(n_pairs);
    const int32_t mp = (int32_t)std::min<int64_t>(max_perm, INT32_MAX);
    if (n_dev == 1) chk(cmb_mica_permutations(ctx, seed, mp, n_pairs, perm_p.data(), perm_nb.data(), nullptr));
    else { // GPU r tests the pairs r, r + N, r + 2N, ...; its rows are scattered back into the table's order
      on_all(n_dev, [&](int r) {
        const int64_t cap = r < n_pairs ? (n_pairs - 1 - r) / n_dev + 1 : 0;
        std::vector<double> p(cap);
        std::vector<int32_t> nb(cap);
        int64_t got = 0;
        chk(cmb_mica_permutations_shard(ctxs[r], seed, mp, r, n_dev, cap, p.data(), nb.data(), &got));
        for (int64_t k = 0; k < got; k++) { perm_p[r + k * n_dev] = p[k]; perm_nb[r + k * n_dev] = nb[k]; }
      });
    }
  }
  {
    std::ofstream out(path);
    std::string header = "Group\tMI\tAPC\tRCW\tHjoint\tHmin";
    if (with_model) header += "\tNmin";
    if (max_perm > 0) header += "\tPerm.p.value\tPerm.nb";
    if (compute_p) header += "\tBs.p.value\tBs.nb";
    header += "\n";
    out.write(header.data(), (std::streamsize)header.size());
    write_rows_parallel(out, rows, 256, [&](int64_t r, char* p) {
      const double apc = average[I[r]] * average[J[r]] / full_average, rcw = average[I[r]] * average[J[r]] / 2.;
      char* q = p;
      q += snprintf(q, 40, "[%d;%d]\t", in.cols[I[r]] + 1, in.cols[J[r]] + 1);
      q += fmt_g(q, mi[r]); *q++ = '\t';
      q += fmt_g(q, apc); *q++ = '\t';
      q += fmt_g(q, rcw); *q++ = '\t';
      q += fmt_g(q, hj[r]); *q++ = '\t';
      q += fmt_g(q, hm[r]);
      if (with_model) { *q++ = '\t'; q += fmt_g(q, nm[r]); }
      if (max_perm > 0) { *q++ = '\t'; q += fmt_g(q, perm_p[r]); q += snprintf(q, 16, "\t%d", perm_nb[r]); }
      if (compute_p) {
        if (std::isnan(pv[r])) q += snprintf(q, 8, "\tNA\t0");
        else { *q++ = '\t'; q += fmt_g(q, pv[r]); q += snprintf(q, 16, "\t%d", nsim[r]); }
      }
      *q++ = '\n';
      return (int)(q - p);
    });
  }
  for (cmb_ctx* c : ctxs) chk(cmb_ctx_destroy(c));
  display_message("\nBye bye ;-)");
  return 0;
}

} // namespace

int main(int argc, char** argv) {
  std::cout << "\n\n***********************************************************\n"
            << "* This is comap_b200: CoMap's hot path on NVIDIA B200      *\n"
            << "*     Coevolution Detection Using Substitution Mapping    *\n"
            << "***********************************************************\n"
            << std::endl;
  if (argc == 1) {
    std::cout << "comap_b200 param=option_file [key=value ...] [--seed=N] [--dry-run]\n"
              << "Option keys are CoMap's (see the CoMap manual / SURVEY.md s5.1)." << std::endl;
    return 0;
  }
  try {
    auto t_start = std::chrono::steady_clock::now();
    Inputs in;
    in.app = parse_command_line(argc, argv);
    bool dry = false;
    for (int i = 1; i < argc; i++) dry |= std::string(argv[i]) == "--dry-run";
    const Params& P = in.app.params;
    { // the same executable serves `mica` (CoMap/Mica.cpp) when it is invoked under that name or with comap_b200.program=mica
      std::string prog = argv[0];
      prog = prog.substr(prog.find_last_of('/') == std::string::npos ? 0 : prog.find_last_of('/') + 1);
      if (!dry && (prog.rfind("mica", 0) == 0 || get_string(P, "comap_b200.program", "comap") == "mica")) return mica_main(in, argv[0]);
    }
    prepare(in, argv[0]);
    if (dry) {
      dry_run_dump(in);
      if (get_path(P, "input.sequence.file2", "none") != "none") { // second data set, same dump after a marker
        const Params P2 = second_data_set_params(P);
        Inputs in2;
        in2.app = in.app;
        prepare(in2, argv[0], &P2, &in.tree);
        std::cout << "DRYRUN second_data_set 1" << std::endl;
        dry_run_dump(in2);
      }
      return 0;
    }
    int64_t S = (int64_t)in.cols.size();
    const int T = (int)in.tree.leaves.size();
    const int B = (int)in.tree.parent.size() - 1;
    uint64_t seed = in.app.seed;
    if (!in.app.seed_given) seed = ((uint64_t)std::random_device{}() << 32) ^ std::random_device{}();

    (void)T;
    (void)B;
    const bool weighted_classes = get_bool(P, "simulations.weighted_classes", false);
    display_result("Rate distribution for simulations", get_bool(P, "simulations.continuous", false) ? "continuous" : "discrete");
    const bool continuous_sim = get_bool(P, "simulations.continuous", false);
    if (continuous_sim && in.rdist.cont_kind == 0)
      throw Error("simulations.continuous=yes is available for Constant, Gamma and Invariant(dist=Gamma) rate distributions");

    display_message("\n\n-*- Get substitution vectors -*-\n");
    Mapped m1 = map_data_set(in, P, "");
    S = (int64_t)in.cols.size(); // saturated sites may have been removed
    cmb_ctx* ctx = m1.ctx;
    if (continuous_sim) chk(cmb_set_continuous_rates(ctx, in.rdist.cont_kind, in.rdist.alpha, in.rdist.p_inv));
    const int n_gpus = (int)get_int(P, "comap_b200.gpus", 1);
    if (n_gpus < 1) throw Error("comap_b200.gpus must be at least 1");
    std::vector<cmb_ctx*> ctxs{ctx};
    if (n_gpus > 1) {
      display_result("GPUs", n_gpus);
      ctxs.resize(n_gpus, nullptr);
      on_all(n_gpus, [&](int r) {
        if (r == 0) return;
        chk(cmb_ctx_create(r, nullptr, &ctxs[r]));
        chk(cmb_set_tree(ctxs[r], (int32_t)in.tree.parent.size(), in.tree.parent.data(), in.tree.brlen.data()));
        chk(cmb_set_model(ctxs[r], in.model.A, in.model.Q.data(), in.model.pi.data(), (int32_t)in.rdist.rates.size(),
                          in.rdist.rates.data(), in.rdist.probs.data(), in.count_method, in.weights.empty() ? nullptr : in.weights.data()));
        chk(cmb_set_map_mode(ctxs[r], in.average, in.joint));
        chk(cmb_set_alignment(ctxs[r], S, in.codes.data(), (int32_t)in.code_mask.size(), in.code_mask.data()));
        Procedure st = parse_procedure(get_string(P, "statistic", "Correlation"));
        if (st.name == "MI") chk(cmb_set_mi_threshold(ctxs[r], get_double(st.args, "threshold", 0.99)));
        if (continuous_sim) chk(cmb_set_continuous_rates(ctxs[r], in.rdist.cont_kind, in.rdist.alpha, in.rdist.p_inv));
        chk(cmb_map(ctxs[r], nullptr, nullptr, nullptr, nullptr, nullptr));
      });
      if (get_path(P, "input.vectors.file", "none") != "none")
        throw Error("comap_b200.gpus > 1 cannot be combined with input.vectors.file");
      chk(cmb_comm_init_all(ctxs.data(), n_gpus));
    }
    std::string analysis = get_string(P, "analysis", "pairwise");
    display_result("Analysis type", analysis);
    // Ancestral sequences, a side output "not used in the analysis" (CoMap.cpp:168-198): marginal reconstruction of
    // every inner node for the selected sites, the existing sequences appended, written as output.sequence.file
    {
      const std::string rec = get_string(P, "asr.method", "none");
      display_result("Ancestral state reconstruction method", rec);
      if (rec == "marginal") {
        const int n_nodes = (int)in.tree.parent.size();
        std::vector<uint8_t> anc((size_t)n_nodes * S);
        chk(cmb_ancestral_states(ctx, anc.data()));
        const std::string seq_out = get_path(P, "output.sequence.file", "none");
        if (seq_out != "none") {
          const std::string fmt = get_string(P, "output.sequence.format", "Fasta");
          if (lower(parse_procedure(fmt).name) != "fasta") throw Error("output.sequence.format '" + fmt + "' is not supported (Fasta)");
          std::ofstream out(seq_out);
          auto put = [&](const std::string& name, const std::string& seq) {
            out << ">" << name << "\n";
            for (size_t k = 0; k < seq.size(); k += 100) out << seq.substr(k, 100) << "\n";
          };
          std::vector<bool> is_leaf(n_nodes, false);
          for (int v : in.tree.leaves) is_leaf[v] = true;
          for (int v = 0; v < n_nodes; v++) {
            if (is_leaf[v]) continue;
            std::string seq((size_t)S, '?');
            for (int64_t j = 0; j < S; j++) seq[j] = in.alpha.states[anc[(size_t)v * S + j]];
            put(std::to_string(v), seq); // unnamed inner nodes are called by their id
          }
          for (size_t r = 0; r < in.aln.names.size(); r++) {
            std::string seq((size_t)S, '?');
            for (int64_t j = 0; j < S; j++) seq[j] = in.aln.seqs[r][in.cols[j]];
            put(in.aln.names[r], seq);
          }
          display_result("Output sequence file", seq_out);
        }
      } else if (rec != "none") throw Error("Unknown ancestral state reconstruction method: " + rec);
    }
    // output.tags.file (CoETools.cpp:314-345): the tree with every node named by its id, and the leaf names' translation
    {
      const std::string tags = get_path(P, "output.tags.file", "none");
      display_result("Tagged tree file", tags);
      if (tags != "none") {
        const int n_nodes = (int)in.tree.parent.size();
        std::string tln = get_path(P, "output.tags.translation", "tags_translation.txt");
        display_result("Tagged tree names translation", tln);
        if (tln != "none") {
          std::ofstream t(tln);
          t << "Name\tId" << std::endl;
          for (int v : in.tree.leaves) t << in.tree.name[v] << "\t" << v << std::endl;
        }
        std::vector<std::vector<int>> kids(n_nodes);
        for (int v = 0; v < n_nodes - 1; v++) kids[in.tree.parent[v]].push_back(v);
        std::function<void(int, std::ostream&)> wr = [&](int v, std::ostream& o) {
          if (!kids[v].empty()) {
            o << "(";
            for (size_t k = 0; k < kids[v].size(); k++) { if (k) o << ","; wr(kids[v][k], o); }
            o << ")";
          }
          o << v;
          if (v != n_nodes - 1) o << ":" << in.tree.brlen[v];
        };
        std::ofstream o(tags);
        wr(n_nodes - 1, o);
        o << ";" << std::endl;
      }
    }

    if (analysis == "none") {
      // mapping only
    } else if (analysis == "pairwise") {
      const int stat_id = stat_id_of(P, in);
      const bool null = get_bool(P, "statistic.null", true);
      if (get_path(P, "input.sequence.file2", "none") != "none") {
        // ---- two data sets (CoMap.cpp:236-347): data set 2 on the same topology, rectangle of
        //      statistics, null distribution of the two simulators
        const Params P2 = second_data_set_params(P);
        Inputs in2;
        in2.app = in.app;
        prepare(in2, argv[0], &P2, &in.tree);
        display_message("\n... and get its substitution vectors.\n");
        Mapped m2 = map_data_set(in2, P2, "2");
        if (continuous_sim) {
          if (in2.rdist.cont_kind == 0) throw Error("simulations.continuous=yes: unsupported rate distribution for data set 2");
          chk(cmb_set_continuous_rates(m2.ctx, in2.rdist.cont_kind, in2.rdist.alpha, in2.rdist.p_inv));
        }
        const int64_t S2 = (int64_t)in2.cols.size();
        // comap_b200.gpus = N: data set 2 on every GPU too, mapped there (the corrected correlation of the null needs
        // both observed mean vectors on each GPU); the rectangle of statistics stays on GPU 0
        std::vector<cmb_ctx*> ctxs2{m2.ctx};
        if (n_gpus > 1) {
          if (get_path(P2, "input.vectors.file", "none") != "none")
            throw Error("comap_b200.gpus > 1 cannot be combined with input.vectors.file2");
          ctxs2.resize(n_gpus, nullptr);
          on_all(n_gpus, [&](int r) {
            if (r == 0) return;
            chk(cmb_ctx_create(r, nullptr, &ctxs2[r]));
            chk(cmb_set_tree(ctxs2[r], (int32_t)in2.tree.parent.size(), in2.tree.parent.data(), in2.tree.brlen.data()));
            chk(cmb_set_model(ctxs2[r], in2.model.A, in2.model.Q.data(), in2.model.pi.data(), (int32_t)in2.rdist.rates.size(),
                              in2.rdist.rates.data(), in2.rdist.probs.data(), in2.count_method,
                              in2.weights.empty() ? nullptr : in2.weights.data()));
            chk(cmb_set_map_mode(ctxs2[r], in2.average, in2.joint));
            chk(cmb_set_alignment(ctxs2[r], S2, in2.codes.data(), (int32_t)in2.code_mask.size(), in2.code_mask.data()));
            Procedure st = parse_procedure(get_string(P2, "statistic", "Correlation"));
            if (st.name == "MI") chk(cmb_set_mi_threshold(ctxs2[r], get_double(st.args, "threshold", 0.99)));
            if (continuous_sim) chk(cmb_set_continuous_rates(ctxs2[r], in2.rdist.cont_kind, in2.rdist.alpha, in2.rdist.p_inv));
            chk(cmb_map(ctxs2[r], nullptr, nullptr, nullptr, nullptr, nullptr));
          });
        }
        display_message("\n\n-*- Compute statistics -*-\n");
        display_message("Compares data set 1 with data set 2.");
        const bool indep = get_bool(P, "independant_comparisons", false);
        cmb_filters f;
        f.min_rate_class = (int32_t)get_int(P, "statistic.min_rate_class", 0);
        f.min_rate = get_double(P, "statistic.min_rate", 0.);
        f.max_rate_class_diff = (int32_t)get_int(P, "statistic.max_rate_class_diff", -1);
        f.max_rate_diff = get_double(P, "statistic.max_rate_diff", -1.);
        f.min_stat = get_double(P, "statistic.min", 0.);
        const int32_t min_rc2 = (int32_t)get_int(P2, "statistic.min_rate_class", 0);
        const double min_r2 = get_double(P2, "statistic.min_rate", 0.);
        std::string stat_path = get_path(P, "statistic.output.file", "statistics.txt");
        if (stat_path == "none") stat_path = "statistics.txt";
        display_message(std::to_string(S) + " sites * " + std::to_string(S2) + " = " +
                        std::to_string(indep ? S : S * S2) + " pairs to compute!");
        const int64_t cap = indep ? S : S * S2;
        std::vector<int32_t> I(cap), J(cap), RC(cap);
        std::vector<double> ST(cap), PR(cap), NM(cap);
        int64_t rows = 0;
        // nmin_by_row = 1: upstream pairs norms1[i] with norms2[i] (CoETools.cpp:803); comap_b200.nmin_by_site=yes fixes it
        chk(cmb_pairs_inter(m1.ctx, m2.ctx, stat_id, &f, min_rc2, min_r2, indep ? 1 : 0,
                            get_bool(P, "comap_b200.nmin_by_site", false) ? 0 : 1, cap, I.data(), J.data(), ST.data(),
                            RC.data(), PR.data(), NM.data(), &rows));
        {
          std::ofstream out(stat_path);
          out << "Group\tStat\tRCmin\tPRmin\tNmin\n";
          write_rows_parallel(out, rows, 160, [&](int64_t r, char* p) {
            char* q = p;
            q += snprintf(q, 40, "[%d;%d]\t", in.cols[I[r]] + 1, in2.cols[J[r]] + 1);
            q += fmt_g(q, ST[r]); *q++ = '\t';
            q += snprintf(q, 16, "%d", RC[r]); *q++ = '\t';
            q += fmt_g(q, PR[r]); *q++ = '\t';
            q += fmt_g(q, NM[r]); *q++ = '\n';
            return (int)(q - p);
          });
        }
        display_result("Wrote statistics to", stat_path);
        display_result("Number of pairs written", rows);
        if (null) {
          // CoETools::computeInterNullDistribution (CoETools.cpp:874-897): defaults 10 x 1000
          std::string null_path = get_path(P, "statistic.null.output.file", "statistics.null.txt");
          if (null_path == "none") null_path = "statistics.null.txt";
          const int rep_cpu = (int)get_int(P, "statistic.null.nb_rep_CPU", 10);
          const int rep_ram = (int)get_int(P, "statistic.null.nb_rep_RAM", 1000);
          display_message("Compute statistic under null hypothesis...");
          std::vector<double> raw((size_t)rep_cpu * rep_ram * 4);
          if (n_gpus == 1)
            chk(cmb_null_inter(m1.ctx, m2.ctx, stat_id, seed, rep_cpu, rep_ram, weighted_classes ? 1 : 0, raw.data()));
          else // outer replicates in contiguous ranges over the GPUs, each range's rows at its first replicate
            on_all(n_gpus, [&](int r) {
              const int q = rep_cpu / n_gpus, m = rep_cpu % n_gpus, r0 = r * q + std::min(r, m), r1 = r0 + q + (r < m ? 1 : 0);
              chk(cmb_null_inter_range(ctxs[r], ctxs2[r], stat_id, seed, rep_cpu, rep_ram, r0, r1, weighted_classes ? 1 : 0,
                                       raw.data() + (size_t)r0 * rep_ram * 4));
            });
          std::ofstream out(null_path);
          out << "Stat\tRCmin\tPRmin\tNmin\n";
          write_rows_parallel(out, (int64_t)rep_cpu * rep_ram, 80, [&](int64_t r, char* p) {
            char* q = p;
            q += fmt_g(q, raw[r * 4]); *q++ = '\t';
            q += snprintf(q, 16, "%d", (int)raw[r * 4 + 1]); *q++ = '\t';
            q += fmt_g(q, raw[r * 4 + 2]); *q++ = '\t';
            q += fmt_g(q, raw[r * 4 + 3]); *q++ = '\n';
            return (int)(q - p);
          });
          display_result("Wrote null distribution to", null_path);
        }
        for (cmb_ctx* c : ctxs2) chk(cmb_ctx_destroy(c));
        for (cmb_ctx* c : ctxs) chk(cmb_ctx_destroy(c));
        double secs = std::chrono::duration<double>(std::chrono::steady_clock::now() - t_start).count();
        std::cout << "Total execution time: " << secs << "s" << std::endl;
        std::cout << "Bye bye ;-)" << std::endl;
        return 0;
      }
      display_message("\n\n-*- Perform pairwise analysis -*-\n");
      std::string stat_path = get_path(P, "statistic.output.file", "statistics.txt");
      if (stat_path == "none") stat_path = "statistics.txt";
      cmb_filters f;
      f.min_rate_class = (int32_t)get_int(P, "statistic.min_rate_class", 0);
      f.min_rate = get_double(P, "statistic.min_rate", 0.);
      f.max_rate_class_diff = (int32_t)get_int(P, "statistic.max_rate_class_diff", -1);
      f.max_rate_diff = get_double(P, "statistic.max_rate_diff", -1.);
      f.min_stat = get_double(P, "statistic.min", 0.);
      if (null) {
        // CoETools.cpp:638-652, 836-872
        const int K = (int)get_int(P, "statistic.null.nb_rate_classes", 10);
        display_result("Number of sub-distributions", K);
        const int rep_cpu = (int)get_int(P, "statistic.null.nb_rep_CPU", 100);
        const int rep_ram = (int)get_int(P, "statistic.null.nb_rep_RAM", 1000);
        std::string null_path = get_path(P, "statistic.null.output.file", "none");
        if (null_path != "none") display_result("Write simulation results to", null_path);
        display_result("Nb of simulations to perform", (long)rep_cpu * rep_ram);
        if (!get_bool(P, "statistic.null.compute_pvalue", true) && null_path == "none")
          display_message("WARNING!!! statistic.null.compute_pvalue=no without an output file: nothing to do.");
        std::vector<double> raw;
        if (null_path != "none") raw.resize((size_t)rep_cpu * rep_ram * 4);
        if (n_gpus == 1)
          chk(cmb_null_intra(ctx, stat_id, seed, rep_cpu, rep_ram, 0, rep_cpu, weighted_classes ? 1 : 0, K, -1.,
                             raw.empty() ? nullptr : raw.data()));
        else // outer replicates sharded over the GPUs; rank r's rows start at its first replicate
          on_all(n_gpus, [&](int r) {
            const int q = rep_cpu / n_gpus, m = rep_cpu % n_gpus, r0 = r * q + std::min(r, m);
            chk(cmb_null_intra_sharded(ctxs[r], stat_id, seed, rep_cpu, rep_ram, weighted_classes ? 1 : 0, K, -1.,
                                       raw.empty() ? nullptr : raw.data() + (size_t)r0 * rep_ram * 4));
          });
        if (null_path != "none") {
          std::ofstream out(null_path);
          out << "Stat\tRCmin\tPRmin\tNmin\n"; // AnalysisTools.cpp:580,642
          write_rows_parallel(out, (int64_t)rep_cpu * rep_ram, 80, [&](int64_t r, char* p) {
            char* q = p;
            q += fmt_g(q, raw[r * 4]); *q++ = '\t';
            q += snprintf(q, 16, "%d", (int)raw[r * 4 + 1]); *q++ = '\t';
            q += fmt_g(q, raw[r * 4 + 2]); *q++ = '\t';
            q += fmt_g(q, raw[r * 4 + 3]); *q++ = '\n';
            return (int)(q - p);
          });
        }
      }
      const bool pvalues = null && get_bool(P, "statistic.null.compute_pvalue", true);
      display_message("\n\n-*- Compute statistics -*- \n");
      display_message(std::to_string(S) + " sites => " + std::to_string(S * (S + 1) / 2) + " pairs to compute!");
      const int64_t cap = S * (S - 1) / 2;
      std::vector<int32_t> I(cap), J(cap), RC(cap);
      std::vector<double> ST(cap), PR(cap), NM(cap), PV(pvalues ? cap : 0);
      std::vector<int32_t> NS(pvalues ? cap : 0);
      int64_t rows = 0;
      if (n_gpus == 1)
        chk(cmb_pairs(ctx, stat_id, &f, pvalues ? 1 : 0, 0, 1, cap, I.data(), J.data(), ST.data(), RC.data(), PR.data(),
                      NM.data(), pvalues ? PV.data() : nullptr, pvalues ? NS.data() : nullptr, &rows));
      else {
        // rows i with i mod 2N in {r, 2N - 1 - r} are scored by GPU r; the shards are merged back into the
        // reference's order (i ascending, then j)
        struct Shard { std::vector<int32_t> I, J, RC, NS; std::vector<double> ST, PR, NM, PV; int64_t rows = 0; };
        std::vector<Shard> sh(n_gpus);
        on_all(n_gpus, [&](int r) {
          int64_t c = 0;
          for (int64_t i = 0; i < S; i++) {
            const int64_t md = i % (2 * n_gpus);
            if (md == r || md == 2 * n_gpus - 1 - r) c += S - 1 - i;
          }
          Shard& h = sh[r];
          h.I.resize(c); h.J.resize(c); h.RC.resize(c); h.ST.resize(c); h.PR.resize(c); h.NM.resize(c);
          if (pvalues) { h.PV.resize(c); h.NS.resize(c); }
          chk(cmb_pairs(ctxs[r], stat_id, &f, pvalues ? 1 : 0, r, n_gpus, c, h.I.data(), h.J.data(), h.ST.data(), h.RC.data(),
                        h.PR.data(), h.NM.data(), pvalues ? h.PV.data() : nullptr, pvalues ? h.NS.data() : nullptr, &h.rows));
        });
        std::vector<int64_t> cur(n_gpus, 0);
        for (int64_t i = 0; i + 1 < S; i++) {
          const int64_t md = i % (2 * n_gpus);
          const int r = (int)(md < n_gpus ? md : 2 * n_gpus - 1 - md);
          Shard& h = sh[r];
          int64_t a = cur[r], b = a;
          while (b < h.rows && h.I[b] == i) b++;
          const int64_t n = b - a;
          std::copy(h.I.begin() + a, h.I.begin() + b, I.begin() + rows);
          std::copy(h.J.begin() + a, h.J.begin() + b, J.begin() + rows);
          std::copy(h.ST.begin() + a, h.ST.begin() + b, ST.begin() + rows);
          std::copy(h.RC.begin() + a, h.RC.begin() + b, RC.begin() + rows);
          std::copy(h.PR.begin() + a, h.PR.begin() + b, PR.begin() + rows);
          std::copy(h.NM.begin() + a, h.NM.begin() + b, NM.begin() + rows);
          if (pvalues) {
            std::copy(h.PV.begin() + a, h.PV.begin() + b, PV.begin() + rows);
            std::copy(h.NS.begin() + a, h.NS.begin() + b, NS.begin() + rows);
          }
          cur[r] = b;
          rows += n;
        }
      }
      std::ofstream out(stat_path);
      out << "Group\tStat\tRCmin\tPRmin\tNmin";
      if (null) out << "\tPValue\tNsim";
      out << "\n";
      write_rows_parallel(out, rows, 160, [&](int64_t r, char* p) {
        char* q = p;
        q += snprintf(q, 40, "[%d;%d]\t", in.cols[I[r]] + 1, in.cols[J[r]] + 1);
        q += fmt_g(q, ST[r]); *q++ = '\t';
        q += snprintf(q, 16, "%d", RC[r]); *q++ = '\t';
        q += fmt_g(q, PR[r]); *q++ = '\t';
        q += fmt_g(q, NM[r]);
        if (null) {
          if (pvalues && !std::isnan(PV[r])) {
            *q++ = '\t';
            q += fmt_g(q, PV[r]);
            q += snprintf(q, 24, "\t%lld", (long long)NS[r]);
          } else q += snprintf(q, 8, "\tNA\t0");
        }
        *q++ = '\n';
        return (int)(q - p);
      });
      display_result("Wrote statistics to", stat_path);
      display_result("Number of pairs written", rows);
    } else if (analysis == "clustering") {
      display_message("\n\n-*- Perform clustering analysis -*-\n");
      std::string method = get_string(P, "clustering.method", "complete");
      if (method != "none") {
        std::string dm = get_string(P, "clustering.distance", "cor");
        int dist_id;
        if (dm == "Euclidian" || dm == "euclidian") dist_id = CMB_DIST_EUCLIDIAN;
        else if (dm == "Correlation" || dm == "cor") dist_id = CMB_DIST_CORRELATION;
        else if (dm == "Compensation" || dm == "comp") { // CoMap.cpp:412-422
          if (in.weights.empty())
            throw Error("Compensation distance must be used with a mapping procedure with weights, e.g. "
                        "'nijt=Uniformization(weight=Diff(index1=Volume, symmetrical=no))'.");
          if (in.weights_symmetric)
            throw Error("Compensation distance must be used with a mapping procedure allowing non-symmetric weights, e.g. "
                        "'nijt=Uniformization(weight=Diff(index1=Volume, symmetrical=no))'.");
          dist_id = CMB_DIST_COMPENSATION;
        } else throw Error("Unknown distance method.");
        display_result("Distance to use", dm);
        int link;
        if (method == "complete") link = CMB_LINK_COMPLETE;
        else if (method == "single") link = CMB_LINK_SINGLE;
        else if (method == "average") link = CMB_LINK_AVERAGE;
        else throw Error("Unknown clustering method.");
        std::string mat_path = get_path(P, "clustering.output.matrix.file", "none");
        std::vector<double> mat;
        if (mat_path != "none") mat.resize((size_t)S * S);
        chk(cmb_distance_matrix(ctx, dist_id, mat.empty() ? nullptr : mat.data()));
        if (mat_path != "none") {
          // PhylipDistanceMatrixFormat(extended = true): count, then "name  d d d ..."
          std::ofstream out(mat_path);
          out << "   " << S << "\n";
          for (int64_t i = 0; i < S; i++) {
            out << in.cols[i] + 1 << " ";
            for (int64_t j = 0; j < S; j++) out << " " << mat[(size_t)i * S + j];
            out << "\n";
          }
          display_result("Wrote matrix to file", mat_path);
        }
        display_result("Clustering method", method);
        std::vector<int32_t> left(S - 1), right(S - 1);
        std::vector<double> height(S - 1);
        chk(cmb_cluster(ctx, link, left.data(), right.data(), height.data()));
        const int max_size = (int)get_int(P, "clustering.maximum_group_size", 10);
        std::vector<int32_t> members((size_t)std::max<int64_t>(1, (S - 1) * max_size));
        std::vector<int64_t> offs(S + 1);
        std::vector<double> gh(S), gs(S), gn(S);
        int64_t ng = 0;
        chk(cmb_groups(ctx, dist_id, max_size, members.data(), offs.data(), gh.data(), gs.data(), gn.data(), &ng));
        std::string groups_path = get_path(P, "clustering.output.groups.file", "groups_output_stats.txt");
        if (groups_path == "none") groups_path = "groups_output_stats.txt";
        display_result("Site clusters output file", groups_path);
        {
          std::ofstream out(groups_path);
          out << "Group\tSize\tIsConstant\tDmax\tStat\tNmin\n"; // CoMap.cpp:494-550
          for (int64_t g = 0; g < ng; g++) {
            const int64_t n = offs[g + 1] - offs[g];
            bool cst = false;
            for (int64_t k = 0; k < n && !cst; k++) cst = site_is_constant(in.aln, in.alpha, in.cols[members[offs[g] + k]]);
            out << group_string(&members[offs[g]], n, &in.cols) << "\t" << n << "\t" << (cst ? "yes" : "no") << "\t"
                << gh[g] * 2. << "\t" << gs[g] << "\t" << gn[g] << "\n";
          }
        }
        std::string tree_path = get_path(P, "clustering.output.tree.file", "none");
        if (tree_path != "none") {
          std::ofstream out(tree_path);
          out << dendrogram_newick(left, right, height, S, in.cols) << std::endl;
          display_result("Wrote tree to file", tree_path);
        }
        display_message("\n\n-*- Compute null distribution of clusters -*-\n");
        display_result("Maximum group size to test", max_size);
        if (get_bool(P, "clustering.null", false)) {
          std::string sim_path = get_path(P, "clustering.null.output.file", "groups_output_null.txt");
          const int nrep = (int)get_int(P, "clustering.null.number", 1);
          display_result("Number of simulations", nrep);
          display_result("Simulations output file", sim_path);
          std::ofstream out;
          if (sim_path != "none") {
            out.open(sim_path);
            out << "Rep\tGroup\tSize\tDmax\tStat\tNmin\n"; // ClusterTools.cpp:219
          }
          // replicates in batches so the host buffers stay small; with several GPUs a batch is dealt to them in
          // contiguous replicate ranges (replicas only: no exchange) and written in replicate order
          const int batch = std::max(1, (int)std::min<int64_t>(nrep, (int64_t)n_gpus * (1 << 22) / std::max<int64_t>(1, S)));
          struct NullRows {
            std::vector<int32_t> rep, size, mem; std::vector<double> dmax, st, nm; std::vector<int64_t> off; int64_t nr = 0;
          };
          for (int r0 = 0; r0 < nrep; r0 += batch) {
            const int r1 = std::min(nrep, r0 + batch);
            std::vector<NullRows> part(n_gpus);
            on_all(n_gpus, [&](int g) {
              const int nb = r1 - r0, q = nb / n_gpus, m = nb % n_gpus;
              const int a = r0 + g * q + std::min(g, m), b = a + q + (g < m ? 1 : 0);
              if (a == b) return;
              NullRows& x = part[g];
              const int64_t cap_rows = (int64_t)(b - a) * (S - 1), cap_mem = cap_rows * max_size;
              x.rep.resize(cap_rows); x.size.resize(cap_rows); x.mem.resize((size_t)std::max<int64_t>(1, cap_mem));
              x.dmax.resize(cap_rows); x.st.resize(cap_rows); x.nm.resize(cap_rows); x.off.resize(cap_rows + 1);
              chk(cmb_cluster_null(ctxs[g], dist_id, link, seed, a, b, weighted_classes ? 1 : 0, max_size, cap_rows, cap_mem,
                                   x.rep.data(), x.size.data(), x.dmax.data(), x.st.data(), x.nm.data(), x.mem.data(),
                                   x.off.data(), &x.nr));
            });
            if (out.is_open())
              for (const NullRows& x : part)
                for (int64_t k = 0; k < x.nr; k++) // Group holds matrix indices here (ClusterTools.cpp:284)
                  out << x.rep[k] << "\t" << group_string(&x.mem[x.off[k]], x.off[k + 1] - x.off[k], nullptr) << "\t" << x.size[k]
                      << "\t" << x.dmax[k] << "\t" << x.st[k] << "\t" << x.nm[k] << "\n";
          }
        }
      }
    } else if (analysis == "candidates") {
      // ---- candidate groups (CoMap.cpp:592-711)
      const int stat_id = stat_id_of(P, in);
      std::string groups_path = get_path(P, "candidates.input.file", "none");
      if (groups_path != "none") {
        display_result("Candidate groups are in file", groups_path);
        const int64_t min_sim = get_int(P, "candidates.null.min", 1000);
        display_result("Minimum number of simulations", min_sim);
        display_result("Verbose level", get_int(P, "candidates.null.verbose", 1));
        std::map<int, int> pos_index; // coordinate -> site index
        for (size_t i = 0; i < in.cols.size(); i++) pos_index[in.cols[i] + 1] = (int)i;
        // DataTable::read(file, sep, header = true)
        std::string sep = get_string(P, "candidates.input.column_sep", "\t");
        if (sep == "\\t" || sep == "tab") sep = "\t";
        std::ifstream gf(groups_path);
        if (!gf) throw Error("candidates.input.file: cannot open '" + groups_path + "'");
        auto split = [&](const std::string& line) {
          std::vector<std::string> out;
          size_t a = 0;
          for (;;) {
            size_t b = line.find(sep, a);
            out.push_back(line.substr(a, b == std::string::npos ? std::string::npos : b - a));
            if (b == std::string::npos) break;
            a = b + sep.size();
          }
          return out;
        };
        std::string line;
        std::getline(gf, line);
        if (!line.empty() && line.back() == '\r') line.pop_back();
        std::vector<std::string> header = split(line);
        std::vector<std::vector<std::string>> table;
        while (std::getline(gf, line)) {
          if (!line.empty() && line.back() == '\r') line.pop_back();
          if (line.empty()) continue;
          table.push_back(split(line));
          if (table.back().size() != header.size())
            throw Error("candidates.input.file: row " + std::to_string(table.size()) + " has " +
                        std::to_string(table.back().size()) + " columns, header has " + std::to_string(header.size()));
        }
        const std::string col_name = get_string(P, "candidates.input.column_name", "Group");
        const auto hc = std::find(header.begin(), header.end(), col_name);
        if (hc == header.end()) throw Error("candidates.input.file: no column '" + col_name + "'");
        const size_t gc = (size_t)(hc - header.begin());
        double omega = get_double(P, "candidates.omega", 0.25);
        display_result("Norm interval", omega);
        if (omega < 0) {
          display_message("WARNING!!! Norm range parameter 'omega' must be positive... |omega| was used instead.");
          omega = -omega;
        }
        // groups: digits and ; , only (CoMap.cpp:632-664)
        std::vector<int64_t> off{0};
        std::vector<int32_t> gsites;
        std::vector<uint8_t> analysable;
        for (size_t i = 0; i < table.size(); i++) {
          std::string clean;
          for (char ch : table[i][gc])
            if (std::strchr("0123456789;,", ch)) clean += ch;
          std::vector<int> positions;
          std::string tok;
          for (char ch : clean + ";") {
            if (ch == ';' || ch == ',') {
              if (!tok.empty()) positions.push_back(std::stoi(tok));
              tok.clear();
            } else tok += ch;
          }
          if (positions.size() <= 1)
            throw Error("Error, group " + std::to_string(i) + " has " + std::to_string(positions.size()) + "sites.");
          bool ok = true;
          for (int pos : positions) {
            auto it = pos_index.find(pos);
            if (it == pos_index.end()) {
              ok = false;
              display_message("WARNING!!! Position " + std::to_string(pos) + " is not included in the selected sites. The group "
                              "will be ignored (line " + std::to_string(i + 1) + " in input file).");
              break;
            }
            gsites.push_back(it->second);
          }
          off.push_back((int64_t)gsites.size());
          analysable.push_back(ok ? 1 : 0);
        }
        display_result("Number of groups to test", table.size());
        if (table.empty()) throw Error("ERROR!!! No group can be tested!");
        const int max_trials = (int)get_int(P, "candidates.nb_max_trials", 10);
        const int rep_ram = (int)get_int(P, "candidates.null.nb_rep_RAM", 1000);
        std::vector<double> gstat(table.size()), gp(table.size());
        int64_t n_sim = 0;
        chk(cmb_candidates(ctx, stat_id, (int32_t)table.size(), off.data(), gsites.data(), analysable.data(), omega, min_sim,
                           max_trials, rep_ram, seed, weighted_classes ? 1 : 0, gstat.data(), gp.data(), nullptr, nullptr,
                           &n_sim));
        display_result("Number of sites simulated", n_sim);
        // table + Stat + p-value (TextTools::toString(x, 6)), DataTable::write
        std::string out_path = get_path(P, "candidates.output.file", "none");
        if (out_path == "none") throw Error("candidates.output.file is not set");
        std::string osep = get_string(P, "candidates.output.column_sep", sep);
        if (osep == "\\t" || osep == "tab") osep = "\t";
        std::ofstream out(out_path);
        for (size_t k = 0; k < header.size(); k++) out << header[k] << osep;
        out << "Stat" << osep << "p-value\n";
        char buf[64];
        for (size_t i = 0; i < table.size(); i++) {
          for (const auto& cell : table[i]) out << cell << osep;
          if (analysable[i]) { fmt_g(buf, gstat[i]); out << buf << osep; fmt_g(buf, gp[i]); out << buf << "\n"; }
          else out << "NA" << osep << "NA\n";
        }
        display_result("Wrote results in file", out_path);
      }
    } else throw Error("Unknown analysis type: " + analysis);

    for (size_t r = 1; r < ctxs.size(); r++) chk(cmb_ctx_destroy(ctxs[r]));
    chk(cmb_ctx_destroy(ctx));
    double secs = std::chrono::duration<double>(std::chrono::steady_clock::now() - t_start).count();
    std::cout << "Total execution time: " << secs << "s" << std::endl;
    std::cout << "Bye bye ;-)" << std::endl;
    return 0;
  } catch (const std::exception& e) {
    // CoMap.cpp:730-734: message, exit(-1)
    std::cout << std::endl << e.what() << std::endl;
    return 255;
  }
}
