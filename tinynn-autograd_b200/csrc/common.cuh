// Shared internals of libtnn_b200: error plumbing, the per-process context and launch helpers.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string>
#include <type_traits>

#include "../../include/tnn_b200.h"

namespace tnn {

struct Context {
  bool inited = false;
  int device = 0;
  int sm_count = 148;
  size_t l2_bytes = 0;
  cudaStream_t stream = nullptr;       // compute stream: every kernel goes here
  cudaStream_t copy_stream = nullptr;  // H2D prefetch
  cudaStream_t comm_stream = nullptr;  // gradient all-reduce chunks running beside the optimiser (comm.cu)
  cudaStream_t d2h_stream = nullptr;   // asynchronous read-backs (tnn_d2h_async): a host read of step i's
                                       // loss must not wait for step i+1, which is already queued
  cudaEvent_t ev_comm = nullptr;       // last comm-stream fence
  cudaEvent_t ev_copy = nullptr;       // last copy-stream fence
  cudaEvent_t ev_compute = nullptr;    // last compute-stream fence
  uint64_t launches = 0;               // kernels launched by this library
  int prof_family = 0;                 // tnn_prof_enable
  void* scratch = nullptr;             // reduction partials (grown on demand)
  size_t scratch_bytes = 0;
  void* l2_flush_buf = nullptr;
  size_t l2_flush_bytes = 0;
};

Context& ctx();
void set_error(const std::string& msg);
int fail(const char* file, int line, const std::string& msg);
// reduction scratch on the compute stream (valid until the next call that asks for scratch)
int get_scratch(size_t nbytes, void** out);
// arrival counters of the split column reductions (reduce.cu, batchnorm.cu): MAX_COL_COUNTERS of them,
// allocated on first use, each zero between launches
constexpr int64_t MAX_COL_COUNTERS = 1 << 16;
int col_fold_counters(unsigned int** out);

// bracket a launch with events when profiling of `family` is on
void prof_begin(int family);
void prof_end(int family);

}  // namespace tnn

#define TNN_FAIL(msg) return ::tnn::fail(__FILE__, __LINE__, (msg))

#define TNN_CUDA(call)                                                              \
  do {                                                                              \
    cudaError_t _e = (call);                                                        \
    if (_e != cudaSuccess)                                                          \
      return ::tnn::fail(__FILE__, __LINE__,                                        \
                         std::string(#call) + ": " + cudaGetErrorString(_e));       \
  } while (0)

#define TNN_REQUIRE_INIT()                                                          \
  do {                                                                              \
    if (!::tnn::ctx().inited) TNN_FAIL("tnn_init() has not been called");           \
  } while (0)

// after a <<<>>> launch: count it and surface launch-configuration errors immediately
#define TNN_POST_LAUNCH()                                                           \
  do {                                                                              \
    ::tnn::ctx().launches++;                                                        \
    cudaError_t _e = cudaGetLastError();                                            \
    if (_e != cudaSuccess)                                                          \
      return ::tnn::fail(__FILE__, __LINE__,                                        \
                         std::string("kernel launch: ") + cudaGetErrorString(_e));  \
  } while (0)

namespace tnn {

// ---- programmatic dependent launch for chains of small kernels (experiment, off by default) ---------
// The MNIST-sized step is 13 kernels of 3-7 us each; replayed from a CUDA graph it still pays the
// launch latency and the CTA ramp of every kernel behind the previous one's drain.  A kernel launched
// with launch_small(..., pdl = true) under TNN_PDL=1 may be SCHEDULED as soon as every CTA of its
// predecessor has passed pdl_sync() (or exited); its own pdl_sync() then holds it until the predecessor
// has completed and its writes are visible.  The bodies still run strictly one after the other -- same
// arithmetic, same order (the whole GPU suite passes with it on) -- only launch and scheduling overlap.
// Measured on the recorded MNIST step: 0.0889 ms with the attribute against 0.0844 ms without (same
// box, alternating runs, profiles/r02h_pdl_experiment.md): with the trigger at the top of every kernel
// the whole chain becomes resident at once and the parked CTAs cost more than the hidden launch
// latency gains, so the attribute is NOT set unless TNN_PDL=1.  pdl_sync() is a no-op in a kernel
// launched the ordinary way.
__device__ __forceinline__ void pdl_sync() {
#if defined(__CUDA_ARCH__) && __CUDA_ARCH__ >= 900
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  asm volatile("griddepcontrol.wait;" ::: "memory");
#endif
}

inline bool pdl_on() {
  static int on = -1;
  if (on < 0) {
    const char* e = getenv("TNN_PDL");
    on = (e && e[0] == '1') ? 1 : 0;
  }
  return on == 1;
}

// cudaLaunchKernelEx with optional cluster dimension (cluster_z > 1) and the programmatic-dependency
// attribute; the kernel must call pdl_sync() before it touches global memory
template <typename... KArgs, typename... Args>
inline cudaError_t launch_small(void (*kernel)(KArgs...), dim3 grid, dim3 block, cudaStream_t st, bool pdl,
                                unsigned cluster_z, Args&&... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = 0;
  cfg.stream = st;
  cudaLaunchAttribute attr[2];
  unsigned n = 0;
  if (cluster_z > 1) {
    attr[n].id = cudaLaunchAttributeClusterDimension;
    attr[n].val.clusterDim.x = 1;
    attr[n].val.clusterDim.y = 1;
    attr[n].val.clusterDim.z = cluster_z;
    ++n;
  }
  if (pdl && pdl_on()) {
    attr[n].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[n].val.programmaticStreamSerializationAllowed = 1;
    ++n;
  }
  cfg.attrs = attr;
  cfg.numAttrs = n;
  return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}

// EL consecutive elements moved as one access (16 bytes for EL = 16 / sizeof(T))
template <typename T, int EL>
struct alignas(sizeof(T) * EL) Pack {
  T v[EL];
};

inline bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

// The C++ type of a float dtype code: f(float{}) for TNN_F32, f(double{}) for TNN_F64.  Any other
// code fails with a message naming the entry point `name`.  f returns int like the entry points.
template <typename F>
inline int with_float_type(int dtype, const char* name, F&& f) {
  if (dtype == TNN_F32) return f(float{});
  if (dtype == TNN_F64) return f(double{});
  TNN_FAIL(std::string(name) + ": bad dtype");
}

// A runtime choice (a vector path, a phase) as a template argument: f(std::true_type{}) or
// f(std::false_type{}), whose parameter converts to a bool template argument
template <typename F>
inline decltype(auto) with_bool(bool flag, F&& f) {
  return flag ? f(std::true_type{}) : f(std::false_type{});
}

__host__ __device__ inline int64_t ceil_div(int64_t a, int64_t b) { return (a + b - 1) / b; }

// A column reduction whose rows are split across nsplit CTAs: each CTA has written its partial, and
// the LAST one to arrive for the column block (its counter `cnt`) folds them -- in split order, so
// the result does not depend on which CTA that is.  Called by every thread of the CTA; true in the
// last one, whose later reads see every partial.  That CTA rearms the counter for the next launch.
__device__ __forceinline__ bool col_fold_last_arrival(unsigned int* cnt, unsigned int nsplit) {
  __shared__ bool is_last;
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0 && threadIdx.y == 0) {
    const unsigned int prev = atomicAdd(cnt, 1u);
    is_last = prev == nsplit - 1;
    if (is_last) *cnt = 0u;
  }
  __syncthreads();
  if (!is_last) return false;
  __threadfence();
  return true;
}

// grid for a grid-stride elementwise kernel: enough CTAs to fill the chip a few times over,
// in multiples of the SM count
inline int ew_grid(int64_t work_items, int threads, int per_sm = 8) {
  int64_t blocks = ceil_div(work_items, threads);
  int64_t cap = (int64_t)ctx().sm_count * per_sm;
  if (blocks > cap) blocks = cap;
  if (blocks < 1) blocks = 1;
  return (int)blocks;
}

}  // namespace tnn
