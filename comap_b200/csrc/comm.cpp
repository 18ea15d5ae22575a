// Multi-GPU plumbing of libcomap_b200.so (SURVEY.md s8e): one cmb_ctx per GPU; the only exchange step of
// the pairwise path is the all-gather of the null samples, issued with NCCL on the context's stream so no
// host synchronisation sits between the last null kernel and the binning of the gathered samples.
//
// NCCL is bound at run time (dlopen of libnccl.so.2): a single-GPU user needs no NCCL, and inside a process
// that already loaded one (torch bundles its own) the same instance is used.
#include "../../include/comap_b200.h"
#include "context.h"
#include <dlfcn.h>
#include <cstring>
#include <mutex>

namespace cmb {

namespace {
// the slice of nccl.h this file needs (NCCL's C ABI is stable across 2.x)
struct ncclComm;
typedef struct ncclComm* ncclComm_t;
struct ncclUniqueId { char internal[128]; };
enum { ncclFloat64 = 8 };
struct NcclApi {
  int (*GetUniqueId)(ncclUniqueId*) = nullptr;
  int (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int) = nullptr;
  int (*CommInitAll)(ncclComm_t*, int, const int*) = nullptr;
  int (*CommDestroy)(ncclComm_t) = nullptr;
  int (*AllGather)(const void*, void*, size_t, int, ncclComm_t, cudaStream_t) = nullptr;
  int (*GroupStart)() = nullptr;
  int (*GroupEnd)() = nullptr;
  const char* (*GetErrorString)(int) = nullptr;
  bool ok = false;
};
NcclApi& nccl() {
  static NcclApi api;
  static std::once_flag once;
  std::call_once(once, [] {
    void* h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
    if (!h) h = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
    if (!h) return;
    auto sym = [&](const char* n) { return dlsym(h, n); };
    api.GetUniqueId = (decltype(api.GetUniqueId))sym("ncclGetUniqueId");
    api.CommInitRank = (decltype(api.CommInitRank))sym("ncclCommInitRank");
    api.CommInitAll = (decltype(api.CommInitAll))sym("ncclCommInitAll");
    api.CommDestroy = (decltype(api.CommDestroy))sym("ncclCommDestroy");
    api.AllGather = (decltype(api.AllGather))sym("ncclAllGather");
    api.GroupStart = (decltype(api.GroupStart))sym("ncclGroupStart");
    api.GroupEnd = (decltype(api.GroupEnd))sym("ncclGroupEnd");
    api.GetErrorString = (decltype(api.GetErrorString))sym("ncclGetErrorString");
    api.ok = api.GetUniqueId && api.CommInitRank && api.CommInitAll && api.CommDestroy && api.AllGather &&
             api.GroupStart && api.GroupEnd && api.GetErrorString;
  });
  if (!api.ok) fail("multi-GPU run: libnccl.so.2 could not be loaded (%s)", dlerror() ? dlerror() : "missing symbols");
  return api;
}
void nccl_check(int rc, const char* what) {
  if (rc != 0) fail("%s failed: %s", what, nccl().GetErrorString(rc));
}
} // namespace

// all-gather of `count` doubles per rank on the context's stream
void comm_all_gather(Context& c, const double* send, double* recv, size_t count) {
  if (!c.comm) fail("internal: no communicator");
  nccl_check(nccl().AllGather(send, recv, count, ncclFloat64, (ncclComm_t)c.comm, c.stream), "ncclAllGather");
}

} // namespace cmb

using namespace cmb;

extern "C" {

int cmb_comm_unique_id(void* id128) {
  CMB_TRY
  ncclUniqueId id;
  nccl_check(nccl().GetUniqueId(&id), "ncclGetUniqueId");
  std::memcpy(id128, &id, sizeof id);
  CMB_CATCH
}

int cmb_comm_init(cmb_ctx* ctx, int32_t n_ranks, int32_t rank, const void* id128) {
  CMB_TRY
  Context& c = ctx->c;
  if (n_ranks < 1 || rank < 0 || rank >= n_ranks) fail("cmb_comm_init: bad rank %d of %d", rank, n_ranks);
  if (c.comm) fail("cmb_comm_init: the context already has a communicator");
  CMB_CUDA(cudaSetDevice(c.device));
  ncclUniqueId id;
  std::memcpy(&id, id128, sizeof id);
  ncclComm_t comm = nullptr;
  nccl_check(nccl().CommInitRank(&comm, n_ranks, id, rank), "ncclCommInitRank");
  c.comm = comm; c.comm_rank = rank; c.comm_size = n_ranks; c.own_comm = true;
  CMB_CATCH
}

int cmb_comm_init_all(cmb_ctx** ctxs, int32_t n) {
  CMB_TRY
  if (n < 1) fail("cmb_comm_init_all: no contexts");
  std::vector<int> devs(n);
  std::vector<ncclComm_t> comms(n, nullptr);
  for (int i = 0; i < n; i++) {
    if (ctxs[i]->c.comm) fail("cmb_comm_init_all: context %d already has a communicator", i);
    devs[i] = ctxs[i]->c.device;
    for (int j = 0; j < i; j++)
      if (devs[j] == devs[i]) fail("cmb_comm_init_all: contexts %d and %d share device %d", j, i, devs[i]);
  }
  nccl_check(nccl().CommInitAll(comms.data(), n, devs.data()), "ncclCommInitAll");
  for (int i = 0; i < n; i++) {
    Context& c = ctxs[i]->c;
    c.comm = comms[i]; c.comm_rank = i; c.comm_size = n; c.own_comm = true;
  }
  CMB_CATCH
}

int cmb_comm_set(cmb_ctx* ctx, void* nccl_comm, int32_t n_ranks, int32_t rank) {
  CMB_TRY
  Context& c = ctx->c;
  if (n_ranks < 1 || rank < 0 || rank >= n_ranks) fail("cmb_comm_set: bad rank %d of %d", rank, n_ranks);
  nccl(); // the library must be loadable
  c.comm = nccl_comm; c.comm_rank = rank; c.comm_size = n_ranks; c.own_comm = false;
  CMB_CATCH
}

int cmb_comm_destroy(cmb_ctx* ctx) {
  CMB_TRY
  Context& c = ctx->c;
  if (c.comm && c.own_comm) {
    CMB_CUDA(cudaSetDevice(c.device));
    CMB_CUDA(cudaStreamSynchronize(c.stream));
    nccl_check(nccl().CommDestroy((ncclComm_t)c.comm), "ncclCommDestroy");
  }
  c.comm = nullptr; c.comm_rank = 0; c.comm_size = 1; c.own_comm = false;
  CMB_CATCH
}

int cmb_comm_rank(cmb_ctx* ctx, int32_t* rank, int32_t* n_ranks) {
  if (rank) *rank = ctx->c.comm_rank;
  if (n_ranks) *n_ranks = ctx->c.comm_size;
  return 0;
}

int cmb_comm_group_start(void) {
  CMB_TRY
  nccl_check(nccl().GroupStart(), "ncclGroupStart");
  CMB_CATCH
}
int cmb_comm_group_end(void) {
  CMB_TRY
  nccl_check(nccl().GroupEnd(), "ncclGroupEnd");
  CMB_CATCH
}

} // extern "C"
