// Shared declarations of libcomap_b200.so (host side).  Product code: nothing here may
// reference oracle/.
#pragma once
#include <cuda_runtime.h>
#include <cstdint>
#include <cstdio>
#include <map>
#include <stdexcept>
#include <string>
#include <vector>

namespace cmb {

struct Error : std::runtime_error {
  explicit Error(const std::string& m) : std::runtime_error(m) {}
};

[[noreturn]] void fail(const char* fmt, ...);

#define CMB_CUDA(expr)                                                                   \
  do {                                                                                   \
    cudaError_t _e = (expr);                                                             \
    if (_e != cudaSuccess)                                                               \
      ::cmb::fail("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__); \
  } while (0)

inline size_t align256(size_t x) { return (x + 255) & ~size_t(255); }

// Device buffer that only grows (arena-style reuse across batches); frees its memory when destroyed.
struct DevBuf {
  void* p = nullptr;
  size_t cap = 0;
  DevBuf() = default;
  DevBuf(const DevBuf&) = delete;
  DevBuf& operator=(const DevBuf&) = delete;
  DevBuf(DevBuf&& o) noexcept : p(o.p), cap(o.cap) { o.p = nullptr; o.cap = 0; }
  DevBuf& operator=(DevBuf&& o) noexcept {
    if (this != &o) { release(); p = o.p; cap = o.cap; o.p = nullptr; o.cap = 0; }
    return *this;
  }
  ~DevBuf() { release(); }
  void reserve(size_t bytes);
  void release();
  template <class T> T* as() const { return static_cast<T*>(p); }
};

// ---------------------------------------------------------------- K0: model tables
// P_c(b) = exp(Q d_b r_c) and W_c(b) = p_c * P_c(b) o n_c(b) for every branch x class
// (host fp64; SURVEY.md s2.2 K0).  Layout [branch][c][x][y].
struct ModelTables {
  int A = 0, C = 0, B = 0;
  std::vector<double> pi, rates, probs;
  std::vector<double> P;    // [B][C][A][A]
  std::vector<double> W;    // [B][C][A][A], includes p_c
  std::vector<double> N;    // [B][C][A][A] the counts themselves (mapping variants, k1_variants.cu)
  std::vector<double> cumP; // [B][C][A][A] running row sums of P (simulator)
};
void build_model_tables(ModelTables& mt, int A, const double* Q, const double* pi, int C,
                        const double* rates, const double* probs, int count_method,
                        const double* weights, int B, const double* brlen);

// eigen-decomposition of a reversible generator, Q = R diag(ev) L (tables.cpp); R, L row-major A x A
void build_spectrum(int A, const double* Q, const double* pi, std::vector<double>& ev, std::vector<double>& R, std::vector<double>& L);

// ---------------------------------------------------------------- tree + op streams
constexpr int kMaxStack = 20; // per-thread stack depth; log2(#leaves)+2 suffices
constexpr int kChunkSites = 128; // sites per CTA / per partial chunk of the tensor-core K1 kernels (A = 4)

struct BinNode {
  int left = -1, right = -1, parent = -1;
  int branch = -1;   // original branch id (table + output row) or -1 for a virtual edge
  int tip_row = -1;  // alignment row for leaves
  int slot = -1;     // storage slot of the down partial (inner, non-root)
  int leaves = 0;    // leaves below
  bool cherry = false; // inner non-root node whose two children are leaves: no slot
  int orig = -1;     // original node id (-1 for virtual nodes)
};

struct Tree {
  int n_nodes = 0, n_leaves = 0, B = 0;
  std::vector<int32_t> parent;
  std::vector<double> brlen;      // with the 1e-6 floor applied
  std::vector<int> leaf_row;      // node -> alignment row or -1
  std::vector<BinNode> bin;       // binarised tree, root = bin_root
  int bin_root = -1;
  int n_slots = 0;
  std::vector<int> down_order;    // inner bin nodes, post-order (larger child first)
  std::vector<int> up_order;      // inner bin nodes, pre-order (smaller child first)
  int down_depth = 0, up_depth = 0;
};
void build_tree(Tree& t, int n_nodes, const int32_t* parent, const double* brlen);
void assign_slots(Tree& t, bool skip_cherries);

// Packed op stream for one class block [c0, c0+cb).
struct OpStream {
  std::vector<unsigned char> bytes;
  std::vector<uint32_t> chunk_off, chunk_bytes, chunk_nrec;
  std::vector<int32_t> aux;   // 8 ints per record: flags, ref_a, ref_b, 0, ref_a2, ref_b2, 0, 0 (producer-side view)
  uint32_t n_records = 0;
  uint32_t chunk_cap = 0; // largest chunk in bytes
  int stack_depth = 0;    // message stack depth the walk needs (tensor-core down stream)
  uint32_t stage_bytes = 0; // tensor-core up stream: largest packed stage (record | tip rows | partial chunks)
  uint32_t blk_off_max[3] = {0, 0, 0}; // ... largest chunk offset among the nodes with 0 / 1 / 2 stored children
};
constexpr uint32_t kDownTipA = 1, kDownTipB = 2, kDownPush = 4, kDownRoot = 8;
constexpr uint32_t kUpTipA = 1, kUpTipB = 2, kUpPop = 4, kUpPush = 8, kUpTakeA = 16, kUpTakeB = 32,
                   kUpCherryA = 64, kUpCherryB = 128;
struct DownHdr { uint32_t flags; int32_t row_a, row_b, slot; };
struct UpHdr { uint32_t flags; int32_t ref_a, ref_b, out_a, out_b, ref_a2, ref_b2, pad2; };
// tensor-core up stream (k1_mma.cu): out_x1 / out_x2 = output rows of the two leaf branches of a cherry child
// kase = (kind a * 3 + kind b) | push level << 8 | pop level << 16 (0xff: no pop); kinds 0 inner, 1 tip, 2 cherry
struct UpMmaHdr { uint32_t kase; int32_t tips_off, blk_off; uint32_t flags; int32_t out_a, out_b, out_a1, out_a2, out_b1, out_b2, ref_a, ref_b; };
void build_down_stream(OpStream& s, const Tree& t, const ModelTables& mt, int c0, int cb);
void build_up_stream(OpStream& s, const Tree& t, const ModelTables& mt, int c0, int cb);
// Same walk with the tables packed as DMMA m8n8k4 B-operand fragments (A = 4, all classes).
void build_up_mma_stream(OpStream& s, const Tree& t, const ModelTables& mt);
void build_down_mma_stream(OpStream& s, const Tree& t, const ModelTables& mt);
// proteins (A = 20) on the FP64 tensor cores (k1_mma20.cu): one record per (node, class)
constexpr int kChunkSites20 = 64; // sites per CTA / per partial chunk of the protein tensor-core kernels
void build_up_mma20_stream(OpStream& s, const Tree& t, const ModelTables& mt, int sites_per_cta);
void build_down_mma20_stream(OpStream& s, const Tree& t, const ModelTables& mt);
// Simulation walk: per inner bin node (pre-order, smaller first), cumulative tables of
// all classes.  Same header as UpHdr with ref = tip row / unused, out = original node id.
void build_sim_stream(OpStream& s, const Tree& t, const ModelTables& mt);

} // namespace cmb
