// Data-parallel collectives.  The reference is single-process (SURVEY 2.1: no DP, no comm
// backend), so this file is new surface: one NCCL communicator per process (= per GPU), used for
//   * the per-step SUM all-reduce of the flat gradient arena (the layout optimizer.py:14-15
//     already imposes by concatenating every gradient), over NVLink 5 / NVSwitch
//   * the 2-float all-gather of the (max, sum-exp) pair that makes the batch-global softmax of
//     losses.py:26-27 exact under batch sharding
// NCCL is bound at run time with dlopen so that libtnn_b200.so loads (and every single-GPU entry
// point works) on hosts without libnccl.
#include <dlfcn.h>

#include <cstring>

#include "common.cuh"

namespace tnn {
namespace nccl {

typedef struct ncclComm* ncclComm_t;
typedef struct {
  char internal[128];
} ncclUniqueId;
typedef int ncclResult_t;
enum { ncclFloat32 = 7, ncclFloat64 = 8 };
enum { ncclSum = 0 };

struct Api {
  void* handle = nullptr;
  ncclResult_t (*GetVersion)(int*) = nullptr;
  ncclResult_t (*GetUniqueId)(ncclUniqueId*) = nullptr;
  ncclResult_t (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int) = nullptr;
  ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
  ncclResult_t (*AllReduce)(const void*, void*, size_t, int, int, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*AllGather)(const void*, void*, size_t, int, ncclComm_t, cudaStream_t) = nullptr;
  const char* (*GetErrorString)(ncclResult_t) = nullptr;
};

// NCCL's element type for a dtype code, -1 for any other code
static int nccl_type(int dtype) {
  if (dtype == TNN_F32) return ncclFloat32;
  if (dtype == TNN_F64) return ncclFloat64;
  return -1;
}

static Api g_api;
static ncclComm_t g_comm = nullptr;
static int g_world = 1, g_rank = 0;

static int load_api() {
  if (g_api.handle) return 0;
  const char* env = getenv("TNN_NCCL_LIB");
  const char* names[] = {env, "libnccl.so.2", "libnccl.so"};
  void* h = nullptr;
  for (const char* n : names) {
    if (!n) continue;
    h = dlopen(n, RTLD_NOW | RTLD_GLOBAL);
    if (h) break;
  }
  if (!h) TNN_FAIL(std::string("cannot load NCCL (set TNN_NCCL_LIB): ") + dlerror());
#define LOAD(field, sym)                                         \
  g_api.field = (decltype(g_api.field))dlsym(h, sym);            \
  if (!g_api.field) TNN_FAIL(std::string("NCCL symbol missing: ") + sym);
  LOAD(GetVersion, "ncclGetVersion");
  LOAD(GetUniqueId, "ncclGetUniqueId");
  LOAD(CommInitRank, "ncclCommInitRank");
  LOAD(CommDestroy, "ncclCommDestroy");
  LOAD(AllReduce, "ncclAllReduce");
  LOAD(AllGather, "ncclAllGather");
  LOAD(GetErrorString, "ncclGetErrorString");
#undef LOAD
  g_api.handle = h;
  return 0;
}

}  // namespace nccl
}  // namespace tnn

using namespace tnn;
using namespace tnn::nccl;

#define TNN_NCCL(call)                                                                   \
  do {                                                                                   \
    ncclResult_t _r = (call);                                                            \
    if (_r != 0) TNN_FAIL(std::string(#call) + ": " + g_api.GetErrorString(_r));         \
  } while (0)

extern "C" {

int tnn_nccl_version(int* v) {
  if (load_api()) return 1;
  TNN_NCCL(g_api.GetVersion(v));
  return 0;
}

int tnn_nccl_unique_id(void* id128) {
  if (load_api()) return 1;
  ncclUniqueId id;
  TNN_NCCL(g_api.GetUniqueId(&id));
  memcpy(id128, &id, sizeof(id));
  return 0;
}

int tnn_nccl_init(int rank, int world, const void* id128) {
  TNN_REQUIRE_INIT();
  if (load_api()) return 1;
  if (g_comm) TNN_FAIL("tnn_nccl_init: communicator already initialised");
  ncclUniqueId id;
  memcpy(&id, id128, sizeof(id));
  TNN_NCCL(g_api.CommInitRank(&g_comm, world, id, rank));
  g_world = world;
  g_rank = rank;
  return 0;
}

int tnn_nccl_destroy(void) {
  if (g_comm) {
    cudaStreamSynchronize(ctx().stream);
    cudaStreamSynchronize(ctx().comm_stream);
    g_api.CommDestroy(g_comm);
    g_comm = nullptr;
  }
  g_world = 1;
  g_rank = 0;
  return 0;
}

int tnn_allreduce_sum(int dtype, void* buf, int64_t n) {
  TNN_REQUIRE_INIT();
  if (!g_comm) TNN_FAIL("tnn_allreduce_sum: call tnn_nccl_init first");
  const int type = nccl_type(dtype);
  if (type < 0) TNN_FAIL("tnn_allreduce_sum: bad dtype");
  TNN_NCCL(g_api.AllReduce(buf, buf, (size_t)n, type, ncclSum, g_comm, ctx().stream));
  ctx().launches++;
  return 0;
}

// ---- all-reduce beside the optimiser -------------------------------------------------------------
// The gradient arena is reduced in chunks on a second stream; the fused optimiser kernel for chunk
// i runs on the compute stream as soon as chunk i is reduced, while chunk i+1 is still on the wire:
//     tnn_comm_wait_compute();                       backward has produced every gradient
//     for each chunk: tnn_allreduce_sum_comm(chunk); tnn_compute_wait_comm(); optimiser(chunk)
// (Overlap with the backward GEMMs themselves is not possible today: the persistent GEMM owns every
// SM's register file, see DESIGN.md section 6.)
int tnn_comm_wait_compute(void) {
  TNN_REQUIRE_INIT();
  Context& c = ctx();
  TNN_CUDA(cudaEventRecord(c.ev_compute, c.stream));
  TNN_CUDA(cudaStreamWaitEvent(c.comm_stream, c.ev_compute, 0));
  return 0;
}

int tnn_compute_wait_comm(void) {
  TNN_REQUIRE_INIT();
  Context& c = ctx();
  TNN_CUDA(cudaEventRecord(c.ev_comm, c.comm_stream));
  TNN_CUDA(cudaStreamWaitEvent(c.stream, c.ev_comm, 0));
  return 0;
}

int tnn_allreduce_sum_comm(int dtype, void* buf, int64_t n) {
  TNN_REQUIRE_INIT();
  if (!g_comm) TNN_FAIL("tnn_allreduce_sum_comm: call tnn_nccl_init first");
  const int type = nccl_type(dtype);
  if (type < 0) TNN_FAIL("tnn_allreduce_sum_comm: bad dtype");
  TNN_NCCL(g_api.AllReduce(buf, buf, (size_t)n, type, ncclSum, g_comm, ctx().comm_stream));
  ctx().launches++;
  return 0;
}

int tnn_allgather(int dtype, void* recv, const void* send, int64_t n_per_rank) {
  TNN_REQUIRE_INIT();
  if (!g_comm) TNN_FAIL("tnn_allgather: call tnn_nccl_init first");
  const int type = nccl_type(dtype);
  if (type < 0) TNN_FAIL("tnn_allgather: bad dtype");
  TNN_NCCL(g_api.AllGather(send, recv, (size_t)n_per_rank, type, g_comm, ctx().stream));
  ctx().launches++;
  return 0;
}

}  // extern "C"
