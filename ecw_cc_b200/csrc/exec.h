// exec.h — the context behind the C API (capi.cu) and the stream executor of its plans (exec.cu).
#pragma once
#include <cuda_runtime.h>

#include <initializer_list>
#include <map>
#include <memory>
#include <stdexcept>
#include <string>
#include <vector>

#include "../../include/ecw_b200.h"
#include "ccsd_plan.h"

namespace ecw {

// NCCL, resolved at run time from the library the process already has (torch's bundled libnccl.so.2): the product
// library itself has no link-time dependency on it.  Only the handful of entry points the executor needs.
struct NcclId { char internal[128]; };
struct NcclApi {
  void* handle = nullptr;
  int (*GetUniqueId)(void*) = nullptr;
  int (*CommInitRank)(void**, int, /* ncclUniqueId by value: */ NcclId, int) = nullptr;
  int (*CommDestroy)(void*) = nullptr;
  int (*AllGather)(const void*, void*, size_t, int, void*, cudaStream_t) = nullptr;
  int (*Send)(const void*, size_t, int, int, void*, cudaStream_t) = nullptr;
  int (*Recv)(void*, size_t, int, int, void*, cudaStream_t) = nullptr;
  int (*GroupStart)() = nullptr;
  int (*GroupEnd)() = nullptr;
  const char* (*GetErrorString)(int) = nullptr;
};

struct Fail : std::runtime_error { using std::runtime_error::runtime_error; };

inline void ck(cudaError_t e, const char* what) {
  if (e != cudaSuccess) throw Fail(std::string(what) + ": " + cudaGetErrorString(e));
}

}  // namespace ecw

struct ecw_ctx {
  ecw::Sizes z;
  ecw::NcclApi nccl;
  void* nccl_comm = nullptr;       // ncclComm_t of this context (SURVEY 8(b)); null: collectives yield to the host
  std::string err;
  double* ptr[ecw::S_COUNT];
  int64_t ws_bytes = 0;
  std::map<std::string, std::unique_ptr<ecw::Plan>> plans;
  bool profile = false;
  bool profile_run = false;   // `profile` latched at the start of the call in flight (ecw_resume keeps it)
  bool force_dmma = false;    // ecw_ctx_set_engine_override: build the plans without the INT8 route
  // resumable execution (plans with collectives yield to the host)
  const ecw::Plan* run_plan_ptr = nullptr;
  size_t pc = 0;
  double run_alpha = 0.0;
  int64_t pending[6] = {0, 0, 0, 0, 0, 0};
  double* copy_scal_to = nullptr;
  ecw::Plan op_plan;       // plan of the last primitive op
  int64_t need_ws = 0;
  std::vector<cudaEvent_t> ev;
  const ecw::Plan* last_plan = nullptr;
  bool call_has_oz = false;      // the plan of the last call contains INT8 products (ecw_int8_error_bound)
  // CUDA-graph replay of the cached plans (tupdate / lupdate / gamma / energy on one GPU): a call whose plan and
  // pointer bindings were seen before is ONE cudaGraphLaunch instead of several hundred kernel launches — the small
  // molecular shapes (configs 1-3) are launch bound.  Captured on a private stream, launched on the caller's.
  struct GraphEntry { cudaGraphExec_t exec = nullptr; uint64_t stamp = 0; };
  std::map<std::string, GraphEntry> graphs;
  cudaStream_t cap_stream = nullptr;
  bool use_graphs = true;
  uint64_t graph_clock = 0;
  int64_t graph_hits = 0, graph_captures = 0;
  int sm_count = 0;        // 0: launchers query / assume 148
  int64_t nccl_ops = 0;    // collectives the executor enqueued itself
  ecw_ctx() { for (auto& p : ptr) p = nullptr; }
};

namespace ecw {

// throws "slot '<name>' is not bound" for the first of `slots` without a pointer
void require_slots(const ecw_ctx* c, std::initializer_list<int> slots);
// the cached plan of a function of the C API (built on first use; the configuration setters drop the cache)
Plan& get_plan(ecw_ctx* c, const std::string& func, int flags);
// plans are rebuilt after every change of the configuration: nothing may keep pointing into the old ones
void drop_graphs(ecw_ctx* c);
void drop_plans(ecw_ctx* c);
// Runs P on the stream.  cached_plan: P is one of get_plan's, so a call on one GPU may replay a CUDA graph.
// Returns 0 when done, 1 when the plan stopped at a collective the host performs (then ecw_resume).
int run_plan(ecw_ctx* c, const Plan& P, double alpha_rt, cudaStream_t st, bool cached_plan = false);
// continues the call in flight from c->pc
int run_plan_resume(ecw_ctx* c, cudaStream_t st);

}  // namespace ecw
