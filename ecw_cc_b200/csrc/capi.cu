// capi.cu — context, plan cache, stream executor and the extern "C" surface
// declared in include/ecw_b200.h.
#include "../../include/ecw_b200.h"

#include <dlfcn.h>

#include <algorithm>
#include <cmath>
#include <cstring>
#include <map>
#include <memory>
#include <sstream>
#include <string>
#include <vector>

#include "ccsd_plan.h"
#include "kernels.h"

using namespace ecw;

// NCCL, resolved at run time from the library the process already has (torch's bundled libnccl.so.2): the product
// library itself has no link-time dependency on it.  Only the handful of entry points the executor needs.
struct NcclApi {
  void* handle = nullptr;
  int (*GetUniqueId)(void*) = nullptr;
  int (*CommInitRank)(void**, int, /* ncclUniqueId by value: */ struct NcclId, int) = nullptr;
  int (*CommDestroy)(void*) = nullptr;
  int (*AllGather)(const void*, void*, size_t, int, void*, cudaStream_t) = nullptr;
  int (*Send)(const void*, size_t, int, int, void*, cudaStream_t) = nullptr;
  int (*Recv)(void*, size_t, int, int, void*, cudaStream_t) = nullptr;
  int (*GroupStart)() = nullptr;
  int (*GroupEnd)() = nullptr;
  const char* (*GetErrorString)(int) = nullptr;
};
struct NcclId { char internal[128]; };
constexpr int kNcclDouble = 8;     // ncclFloat64

struct ecw_ctx {
  Sizes z;
  NcclApi nccl;
  void* nccl_comm = nullptr;       // ncclComm_t of this context (SURVEY 8(b)); null: collectives yield to the host
  std::string err;
  double* ptr[S_COUNT];
  int64_t ws_bytes = 0;
  std::map<std::string, std::unique_ptr<Plan>> plans;
  bool profile = false;
  bool profile_run = false;   // `profile` latched at the start of the call in flight (ecw_resume keeps it)
  bool force_dmma = false;    // ecw_ctx_set_engine_override: build the plans without the INT8 route
  // resumable execution (plans with collectives yield to the host)
  const Plan* run_plan_ptr = nullptr;
  size_t pc = 0;
  double run_alpha = 0.0;
  int64_t pending[6] = {0, 0, 0, 0, 0, 0};
  double* copy_scal_to = nullptr;
  Plan op_plan;            // plan of the last primitive op
  int64_t need_ws = 0;
  std::vector<cudaEvent_t> ev;
  const Plan* last_plan = nullptr;
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

namespace {

int slot_by_name(const char* name) {
  for (int s = 0; s < S_COUNT; ++s)
    if (strcmp(name, slot_name(s)) == 0) return s;
  return -1;
}

int64_t slot_elems(const Sizes& z, int s) {
  const int64_t o = z.nocc, v = z.nvir, n = o + v, po = npair(o), pv = npair(v);
  switch (s) {
    case S_T1: case S_L1: case S_OUT1: return o * v;
    case S_T2: case S_L2: case S_OUT2: case S_OOVV: case S_OOVV_PH: case S_OVOV_PH: return o * o * v * v;
    case S_FSP: case S_FOCK: case S_RDM1: return n * n;
    case S_SCAL: return 16;
    case S_OOOO: return o * o * o * o;
    case S_OOOV: return o * o * o * v;
    case S_OVVV: return o * v * v * v;
    case S_OOOO_P: return po * po;
    case S_OOVV_P: return po * pv;
    case S_OVVV_P: return o * v * pv;
    case S_VVVV_P: case S_VVVV_OZ: case S_VVVV_OZS: {
      const int64_t nshmax = (pv + z.world - 1) / z.world;
      const int64_t n0 = std::min<int64_t>(pv, (int64_t)z.rank * nshmax);
      const int64_t nsh = std::min<int64_t>(pv, n0 + nshmax) - n0;
      if (s == S_VVVV_P) return nsh * pv;
      if (s == S_VVVV_OZS) return ozaki_stat_elems(nsh, 1);         // [row scales | row sums]
      return (ozaki_plane_bytes(nsh, pv, z.oz_ns > 0 ? z.oz_ns : 7) + 7) / 8;   // in 8-byte units
    }
    case S_OVVV_OZ1: return (ozaki_plane_bytes2(o * v, 1, pv, z.oz_ns > 0 ? z.oz_ns : 7) + 7) / 8;
    case S_OVVV_OZ1S: return ozaki_stat_elems(o * v, 1);
    case S_OVVV_OZ2: return (ozaki_plane_bytes2(pv, o, v, z.oz_ns > 0 ? z.oz_ns : 7) + 7) / 8;
    case S_OVVV_OZ2S: return ozaki_stat_elems(pv, o);
    default: return -1;
  }
}

struct Fail : std::runtime_error { using std::runtime_error::runtime_error; };

void ck(cudaError_t e, const char* what) {
  if (e != cudaSuccess) throw Fail(std::string(what) + ": " + cudaGetErrorString(e));
}

// plans are rebuilt after every change of the configuration: nothing may keep pointing into the old ones
void drop_graphs(ecw_ctx* c) {
  for (auto& kv : c->graphs)
    if (kv.second.exec) cudaGraphExecDestroy(kv.second.exec);
  c->graphs.clear();
}

void drop_plans(ecw_ctx* c) {
  drop_graphs(c);
  c->plans.clear();
  c->run_plan_ptr = nullptr;
  c->last_plan = nullptr;
  for (auto e : c->ev) cudaEventDestroy(e);
  c->ev.clear();
}

Plan& get_plan(ecw_ctx* c, const std::string& func, int flags) {
  std::string key = func + "/" + std::to_string(flags) + (c->force_dmma ? "/dmma" : "");
  auto it = c->plans.find(key);
  if (it != c->plans.end()) return *it->second;
  std::unique_ptr<Plan> P(new Plan());
  Sizes zz = c->z;
  if (c->force_dmma) zz.oz_ns = 0;
  const int ha = (flags & ECW_HAS_ALPHA) ? 1 : 0, eq = (flags & ECW_EQUATION) ? 1 : 0;
  const bool as = (flags & ECW_ANTISYM) != 0;
  if (func == "tupdate") (as ? build_ccsd_tupdate : build_ccsd_tupdate_general)(*P, zz, ha, eq);
  else if (func == "lupdate") (as ? build_ccsd_lupdate : build_ccsd_lupdate_general)(*P, zz, ha, eq);
  else if (func == "gamma") build_ccsd_gamma(*P, zz);
  else if (func == "energy") build_ccsd_energy(*P, zz);
  else if (func == "ccs_t1inter") build_ccs_t1inter(*P, zz);
  else if (func == "ccs_l1inter") build_ccs_l1inter(*P, zz, flags & 1);
  else if (func == "ccs_r1inter") build_ccs_r1inter(*P, zz, flags & 1);
  else if (func == "ccs_esl1inter") build_ccs_esl1inter(*P, zz, flags & 1);
  else throw Fail("unknown function '" + func + "'");
  Plan& ref = *P;
  c->plans[key] = std::move(P);
  return ref;
}

double* resolve(ecw_ctx* c, const Tensor& t, bool required = true) {
  if (!t.valid()) {
    if (required) throw Fail("plan references an unset operand");
    return nullptr;
  }
  double* base = c->ptr[t.slot];
  if (!base) throw Fail(std::string("slot '") + slot_name(t.slot) + "' is not bound");
  return base + t.off;
}

void exec_ewise(ecw_ctx* c, const Op& op, cudaStream_t st);   // ccs helpers (ccs_exec.cu)

// Runs ops from c->pc until the end (returns 0) or until a collective op (returns 1: the host
// performs it — torch.distributed over NCCL — and calls ecw_resume).
int run_plan_resume(ecw_ctx* c, cudaStream_t st) {
  const Plan& P = *c->run_plan_ptr;
  const double alpha_rt = c->run_alpha;
  while (c->pc < P.ops.size()) {
    const Op& op = P.ops[c->pc];
    switch (op.kind) {
      case OP_GEMM: {
        GemmArgs g{};
        g.A = resolve(c, op.a); g.B = resolve(c, op.b); g.C = resolve(c, op.c);
        g.M = op.M; g.N = op.N; g.K = op.K; g.lda = op.lda; g.ldb = op.ldb; g.ldc = op.ldc;
        g.sA = op.sA; g.sB = op.sB; g.sC = op.sC; g.batch = op.batch; g.splitk = op.splitk; g.kchunk = op.kchunk;
        g.ta = op.ta; g.tb = op.tb; g.alpha = op.alpha; g.beta = op.beta;
        ck(launch_gemm(g, st), "gemm");
        break;
      }
      case OP_REDUCE:
        ck(launch_reduce(resolve(c, op.a), op.i0, op.M, op.N, resolve(c, op.c), op.i1, op.i2, op.alpha, op.beta, st),
           "reduce");
        break;
      case OP_PERMUTE: {
        PermArgs a{};
        a.in = resolve(c, op.a); a.out = resolve(c, op.c); a.nd = op.c.nd;
        for (int d = 0; d < op.c.nd; ++d) { a.dim[d] = op.c.dim[d]; a.sin[d] = op.a.str[d]; a.sout[d] = op.c.str[d]; }
        a.alpha = op.alpha; a.beta = op.beta;
        ck(launch_permute(a, st), "permute");
        break;
      }
      case OP_FILL:
        ck(launch_fill(resolve(c, op.c), op.c.size(), op.alpha, st), "fill");
        break;
      case OP_TAU:
        ck(launch_tau(resolve(c, op.a), resolve(c, op.b), resolve(c, op.c), (int)op.b.dim[0], (int)op.b.dim[1],
                      op.alpha, op.beta, st, op.i2 ? (int)op.i0 : 0, op.i2 ? (int)op.i1 : -1), "tau");
        break;
      case OP_ASYM4:
        ck(launch_asym4(op.b.valid() ? resolve(c, op.b) : nullptr, op.alpha, resolve(c, op.a), resolve(c, op.c), op.beta,
                        (int)op.c.dim[0], (int)op.c.dim[2], st), "asym4");
        break;
      case OP_PACK: {
        PackArgs a{};
        a.src = resolve(c, op.a); a.dst = resolve(c, op.c);
        a.d0 = op.a.dim[0]; a.d1 = op.a.dim[1]; a.d2 = op.a.dim[2]; a.d3 = op.a.dim[3];
        a.s0 = op.a.str[0]; a.s1 = op.a.str[1]; a.s2 = op.a.str[2]; a.s3 = op.a.str[3];
        a.ld = op.c.str[0]; a.flags = (int)op.i0; a.alpha = op.alpha; a.beta = op.beta;
        ck(launch_pack(a, st), "pack");
        break;
      }
      case OP_UNPACK: {
        PackArgs a{};
        a.src = resolve(c, op.a); a.dst = resolve(c, op.c);
        a.d0 = op.c.dim[0]; a.d1 = op.c.dim[1]; a.d2 = op.c.dim[2]; a.d3 = op.c.dim[3];
        a.s0 = op.c.str[0]; a.s1 = op.c.str[1]; a.s2 = op.c.str[2]; a.s3 = op.c.str[3];
        a.ld = op.a.str[0]; a.flags = (int)op.i0; a.alpha = op.alpha; a.beta = op.beta;
        ck(launch_unpack(a, st), "unpack");
        break;
      }
      case OP_FINISH: {
        int o = (int)op.i0;
        int v = (int)(op.d.dim[0] - o);
        ck(launch_finish(resolve(c, op.a), resolve(c, op.b), resolve(c, op.d), op.d.str[0], resolve(c, op.c), o, v,
                         (int)op.i1, (int)op.i2, (int)op.i3, alpha_rt, op.d0, (int)op.d1, st), "finish");
        break;
      }
      case OP_DOT:
        if (!c->ptr[S_SCAL]) throw Fail("slot 'scal' is not bound");
        ck(launch_dot(resolve(c, op.a), resolve(c, op.b), op.a.size(), resolve(c, op.c), (int)op.i1,
                      c->ptr[S_SCAL] + op.i0, op.alpha, op.beta, st), "dot");
        break;
      case OP_SCALE_DEV:
        if (!c->ptr[S_SCAL]) throw Fail("slot 'scal' is not bound");
        ck(launch_scale_dev(resolve(c, op.c), op.c.size(), c->ptr[S_SCAL] + op.i0, op.d0, op.d1, st), "scale_dev");
        break;
      case OP_DIAG_ADD:
        ck(launch_diag_add(resolve(c, op.c), op.c.str[0], op.c.dim[0], resolve(c, op.d), op.d.str[0], op.i0, op.alpha,
                           st), "diag_add");
        break;
      case OP_RDM1:
        ck(launch_rdm1(resolve(c, op.a), resolve(c, op.b), resolve(c, op.d), resolve(c, op.e), resolve(c, op.c),
                       (int)op.a.dim[0], (int)op.e.dim[0], st), "rdm1");
        break;
      case OP_EWISE:
        exec_ewise(c, op, st);
        break;
      case OP_ALLGATHER:
      case OP_ALLTOALL: {
        if (op.a.slot != S_WS || op.c.slot != S_WS) throw Fail("collective operands must live in the workspace");
        if (c->nccl_comm) {
          // stream-ordered on the caller's stream: no return to the host
          const double* snd = resolve(c, op.a);
          double* rcv = resolve(c, op.c);
          const size_t count = (size_t)op.i0;
          int rc = 0;
          if (op.kind == OP_ALLGATHER) {
            rc = c->nccl.AllGather(snd, rcv, count, kNcclDouble, c->nccl_comm, st);
          } else {
            c->nccl.GroupStart();
            for (int q = 0; q < (int)op.i1 && rc == 0; ++q) {
              rc = c->nccl.Send(snd + (size_t)q * count, count, kNcclDouble, q, c->nccl_comm, st);
              if (rc == 0) rc = c->nccl.Recv(rcv + (size_t)q * count, count, kNcclDouble, q, c->nccl_comm, st);
            }
            const int rc2 = c->nccl.GroupEnd();
            if (rc == 0) rc = rc2;
          }
          if (rc != 0) throw Fail(std::string("NCCL: ") + (c->nccl.GetErrorString ? c->nccl.GetErrorString(rc) : "error"));
          ++c->nccl_ops;
          break;
        }
        c->pending[0] = op.kind == OP_ALLTOALL ? 2 : 1;     // kind: 1 all-gather, 2 all-to-all
        c->pending[1] = op.a.off;          // element offset of this rank's contribution in the workspace
        c->pending[2] = op.i0;             // elements per rank
        c->pending[3] = op.c.off;          // element offset of the gathered buffer (world * count elements)
        c->pending[4] = op.i1;             // world
        c->pending[5] = op.i2;             // rank
        ++c->pc;
        if (c->profile_run) ck(cudaEventRecord(c->ev[c->pc], st), "cudaEventRecord");
        return 1;
      }
      case OP_OZ_SPLIT:
        ck(launch_ozaki_split2(resolve(c, op.a), op.M, op.i1, op.K, op.lda, op.ldc, op.ldb, (int)op.i0,
                               reinterpret_cast<int8_t*>(resolve(c, op.c)), resolve(c, op.d), st), "ozaki_split");
        break;
      case OP_OZ_GEMM: {
        OzBatch bt{};
        bt.batch = op.batch;
        bt.a_row0 = op.oz[0]; bt.a_rowb = op.oz[1]; bt.b_row0 = op.oz[2]; bt.b_rowb = op.oz[3];
        bt.a_kb0 = op.oz[4]; bt.a_kbb = op.oz[5]; bt.b_kb0 = op.oz[6]; bt.b_kbb = op.oz[7];
        bt.a_t0 = op.oz[8]; bt.a_tb = op.oz[9]; bt.b_t0 = op.oz[10]; bt.b_tb = op.oz[11];
        bt.nkb = op.oz[12];
        bt.c_b = op.sC;
        ck(launch_ozaki_gemm_batched(reinterpret_cast<const int8_t*>(resolve(c, op.a)), resolve(c, op.d), op.lda,
                                     reinterpret_cast<const int8_t*>(resolve(c, op.b)), resolve(c, op.e), op.ldb, op.M,
                                     op.N, op.K, resolve(c, op.c), op.i1, op.i2, op.alpha, op.beta, (int)op.i0, bt, st,
                                     c->sm_count),
           "ozaki_gemm");
        if (c->ptr[S_SCAL])
          ck(launch_ozaki_bound(resolve(c, op.d), resolve(c, op.e), op.M, op.N, op.K, op.alpha, (int)op.i0, bt,
                                c->ptr[S_SCAL] + 15, st), "ozaki_bound");
        break;
      }
      default:
        throw Fail("unknown op kind");
    }
    ++c->pc;
    if (c->profile_run) ck(cudaEventRecord(c->ev[c->pc], st), "cudaEventRecord");
  }
  if (c->copy_scal_to) {
    ck(cudaMemcpyAsync(c->copy_scal_to, c->ptr[S_SCAL], sizeof(double), cudaMemcpyDeviceToDevice, st), "copy scalar");
    c->copy_scal_to = nullptr;
  }
  c->run_plan_ptr = nullptr;
  return 0;
}

int run_plan(ecw_ctx* c, const Plan& P, double alpha_rt, cudaStream_t st, bool cached_plan = false) {
  if (P.workspace_elems() * 8 > c->ws_bytes)
    throw Fail("workspace too small: need " + std::to_string(P.workspace_elems() * 8) + " bytes, have " +
               std::to_string(c->ws_bytes));
  c->profile_run = c->profile;
  c->call_has_oz = false;
  bool collectives = false;
  for (const Op& op : P.ops) {
    if (op.kind == OP_OZ_GEMM) c->call_has_oz = true;
    if (op.kind == OP_ALLGATHER || op.kind == OP_ALLTOALL) collectives = true;
  }
  if (cached_plan && c->use_graphs && !c->profile_run && !collectives && c->z.world == 1 && P.ops.size() >= 8) {
    // key: the plan, the run-time scalar and every pointer a launch can resolve
    std::string key(reinterpret_cast<const char*>(c->ptr), sizeof(c->ptr));
    const void* pp = &P;
    key.append(reinterpret_cast<const char*>(&pp), sizeof(pp));
    key.append(reinterpret_cast<const char*>(&alpha_rt), sizeof(alpha_rt));
    key.append(reinterpret_cast<const char*>(&c->copy_scal_to), sizeof(c->copy_scal_to));
    auto it = c->graphs.find(key);
    if (it == c->graphs.end()) {
      if (!c->cap_stream) ck(cudaStreamCreateWithFlags(&c->cap_stream, cudaStreamNonBlocking), "cudaStreamCreate");
      ck(cudaStreamBeginCapture(c->cap_stream, cudaStreamCaptureModeRelaxed), "cudaStreamBeginCapture");
      cudaGraph_t graph = nullptr;
      try {
        if (c->ptr[S_SCAL]) ck(cudaMemsetAsync(c->ptr[S_SCAL] + 15, 0, sizeof(double), c->cap_stream), "reset int8 bound");
        c->run_plan_ptr = &P;
        c->pc = 0;
        c->run_alpha = alpha_rt;
        run_plan_resume(c, c->cap_stream);
      } catch (...) {
        cudaStreamEndCapture(c->cap_stream, &graph);
        if (graph) cudaGraphDestroy(graph);
        cudaGetLastError();
        c->run_plan_ptr = nullptr;
        throw;
      }
      ck(cudaStreamEndCapture(c->cap_stream, &graph), "cudaStreamEndCapture");
      ecw_ctx::GraphEntry ge;
      cudaError_t e = cudaGraphInstantiate(&ge.exec, graph, 0);
      cudaGraphDestroy(graph);
      ck(e, "cudaGraphInstantiate");
      if (c->graphs.size() >= 24) {                 // least recently used entry goes
        auto old = c->graphs.begin();
        for (auto jt = c->graphs.begin(); jt != c->graphs.end(); ++jt)
          if (jt->second.stamp < old->second.stamp) old = jt;
        cudaGraphExecDestroy(old->second.exec);
        c->graphs.erase(old);
      }
      it = c->graphs.emplace(key, ge).first;
      ++c->graph_captures;
    } else {
      ++c->graph_hits;
      c->copy_scal_to = nullptr;
    }
    it->second.stamp = ++c->graph_clock;
    ck(cudaGraphLaunch(it->second.exec, st), "cudaGraphLaunch");
    return 0;
  }
  // run-time error bound of the INT8-route products of this call (scal[15], ecw_int8_error_bound)
  if (c->ptr[S_SCAL]) ck(cudaMemsetAsync(c->ptr[S_SCAL] + 15, 0, sizeof(double), st), "reset int8 bound");
  if (c->profile_run) {
    for (auto e : c->ev) cudaEventDestroy(e);
    c->ev.assign(P.ops.size() + 1, nullptr);
    for (auto& e : c->ev) ck(cudaEventCreate(&e), "cudaEventCreate");
    ck(cudaEventRecord(c->ev[0], st), "cudaEventRecord");
    c->last_plan = &P;
  }
  c->run_plan_ptr = &P;
  c->pc = 0;
  c->run_alpha = alpha_rt;
  return run_plan_resume(c, st);
}

template <typename F>
int guarded(ecw_ctx* c, F&& f) {
  try {
    f();
    return 0;
  } catch (const std::exception& e) {
    if (c) c->err = e.what();
    return -1;
  }
}

template <typename F>
int guarded_rc(ecw_ctx* c, F&& f) {
  try {
    return f();
  } catch (const std::exception& e) {
    if (c) { c->err = e.what(); c->run_plan_ptr = nullptr; }
    return -1;
  }
}

void require_device() {
  int n = 0;
  cudaError_t e = cudaGetDeviceCount(&n);
  if (e != cudaSuccess || n == 0)
    throw Fail("no CUDA device: the ECW-CC residual path has no CPU implementation");
}

}  // namespace

// small CCS element-wise helpers live in ccs_plan.cpp / ccs_exec (none needed yet)
namespace {
void exec_ewise(ecw_ctx* c, const Op& op, cudaStream_t st) {
  // i0 = 0: out = alpha * a * b + beta * out (strided; a and/or b may be absent)
  Ew2Args e{};
  e.a = op.a.valid() ? resolve(c, op.a) : nullptr;
  e.b = op.b.valid() ? resolve(c, op.b) : nullptr;
  e.out = resolve(c, op.c);
  e.nd = op.c.nd;
  for (int d = 0; d < op.c.nd; ++d) {
    e.dim[d] = op.c.dim[d];
    e.so[d] = op.c.str[d];
    e.sa[d] = op.a.valid() ? op.a.str[d] : 0;
    e.sb[d] = op.b.valid() ? op.b.str[d] : 0;
  }
  e.alpha = op.alpha;
  e.beta = op.beta;
  ck(launch_ew2(e, st), "ew2");
}
}  // namespace

extern "C" {

const char* ecw_version(void) { return "ecw_b200 0.1 (sm_100a)"; }

int ecw_ctx_create(ecw_ctx** out, int nocc, int nvir) {
  if (!out || nocc < 1 || nvir < 1) return -1;
  ecw_ctx* c = new ecw_ctx();
  c->z.nocc = nocc;
  c->z.nvir = nvir;
  *out = c;
  return 0;
}

void ecw_ctx_destroy(ecw_ctx* c) {
  if (!c) return;
  for (auto e : c->ev) cudaEventDestroy(e);
  drop_graphs(c);
  if (c->cap_stream) cudaStreamDestroy(c->cap_stream);
  if (c->nccl_comm && c->nccl.CommDestroy) c->nccl.CommDestroy(c->nccl_comm);
  delete c;
}

namespace {
bool load_nccl(NcclApi& api, const char* libpath, std::string& err) {
  if (api.handle) return true;
  const char* names[] = {libpath, "libnccl.so.2", "libnccl.so"};
  void* h = nullptr;
  for (const char* n : names) {
    if (!n || !*n) continue;
    h = dlopen(n, RTLD_NOW | RTLD_GLOBAL);
    if (h) break;
  }
  if (!h) { err = std::string("cannot load NCCL: ") + (dlerror() ? dlerror() : "not found"); return false; }
  auto sym = [&](const char* name) { return dlsym(h, name); };
  api.GetUniqueId = reinterpret_cast<int (*)(void*)>(sym("ncclGetUniqueId"));
  api.CommInitRank = reinterpret_cast<int (*)(void**, int, NcclId, int)>(sym("ncclCommInitRank"));
  api.CommDestroy = reinterpret_cast<int (*)(void*)>(sym("ncclCommDestroy"));
  api.AllGather = reinterpret_cast<int (*)(const void*, void*, size_t, int, void*, cudaStream_t)>(sym("ncclAllGather"));
  api.Send = reinterpret_cast<int (*)(const void*, size_t, int, int, void*, cudaStream_t)>(sym("ncclSend"));
  api.Recv = reinterpret_cast<int (*)(void*, size_t, int, int, void*, cudaStream_t)>(sym("ncclRecv"));
  api.GroupStart = reinterpret_cast<int (*)()>(sym("ncclGroupStart"));
  api.GroupEnd = reinterpret_cast<int (*)()>(sym("ncclGroupEnd"));
  api.GetErrorString = reinterpret_cast<const char* (*)(int)>(sym("ncclGetErrorString"));
  if (!api.GetUniqueId || !api.CommInitRank || !api.AllGather || !api.Send || !api.Recv || !api.GroupStart || !api.GroupEnd) {
    err = "NCCL library lacks a required entry point";
    return false;
  }
  api.handle = h;
  return true;
}
}  // namespace

int ecw_nccl_unique_id(const char* libpath, void* id128) {
  NcclApi api;
  std::string err;
  if (!id128 || !load_nccl(api, libpath, err)) return -1;
  return api.GetUniqueId(id128) == 0 ? 0 : -1;
}

int ecw_ctx_init_nccl(ecw_ctx* c, const char* libpath, const void* id128, int rank, int world) {
  return guarded(c, [&] {
    require_device();
    if (!id128 || world < 2 || rank < 0 || rank >= world) throw Fail("ecw_ctx_init_nccl: bad arguments");
    if (c->z.world != world || c->z.rank != rank) throw Fail("ecw_ctx_init_nccl: rank / world differ from ecw_ctx_set_shard");
    std::string err;
    if (!load_nccl(c->nccl, libpath, err)) throw Fail(err);
    NcclId id;
    memcpy(id.internal, id128, sizeof(id.internal));
    void* comm = nullptr;
    const int rc = c->nccl.CommInitRank(&comm, world, id, rank);
    if (rc != 0) throw Fail(std::string("ncclCommInitRank: ") + (c->nccl.GetErrorString ? c->nccl.GetErrorString(rc) : "error"));
    c->nccl_comm = comm;
  });
}

int64_t ecw_ctx_nccl_ops(ecw_ctx* c) { return c ? c->nccl_ops : -1; }

const char* ecw_last_error(ecw_ctx* c) { return c ? c->err.c_str() : "null context"; }

int ecw_ctx_set_shard(ecw_ctx* c, int rank, int world) {
  if (!c || world < 1 || rank < 0 || rank >= world) return -1;
  c->z.rank = rank;
  c->z.world = world;
  drop_plans(c);
  return 0;
}

int ecw_ctx_set_gemm(ecw_ctx* c, int int8_digits, double min_flops) {
  if (!c || (int8_digits != 0 && (int8_digits < 3 || int8_digits > 8))) return -1;
  if (c->z.vvvv_planes && int8_digits != c->z.oz_ns) {
    c->err = "ecw_ctx_set_gemm: the vvvv digit planes are already bound for another digit count";
    return -1;
  }
  c->z.oz_ns = int8_digits;
  c->z.oz_min_flops = min_flops;
  drop_plans(c);
  return 0;
}

int ecw_ctx_get_gemm(ecw_ctx* c) { return c ? c->z.oz_ns : -1; }

int ecw_ctx_set_engine_override(ecw_ctx* c, int force_dmma) {
  if (!c) return -1;
  c->force_dmma = force_dmma != 0;
  c->run_plan_ptr = nullptr;
  return 0;
}

int ecw_int8_error_bound(ecw_ctx* c, double* bound_out, void* stream) {
  return guarded(c, [&] {
    require_device();
    if (!bound_out) throw Fail("ecw_int8_error_bound: null pointer");
    if (!c->ptr[S_SCAL]) throw Fail("slot 'scal' is not bound");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (!c->call_has_oz) {          // the last call launched no INT8 product: nothing to read, no synchronisation
      *bound_out = 0.0;
      return;
    }
    ck(cudaMemcpyAsync(bound_out, c->ptr[S_SCAL] + 15, sizeof(double), cudaMemcpyDeviceToHost, st), "read int8 bound");
    ck(cudaStreamSynchronize(st), "cudaStreamSynchronize");
  });
}

int ecw_ctx_set_graphs(ecw_ctx* c, int on) {
  if (!c) return -1;
  c->use_graphs = on != 0;
  if (!on) drop_graphs(c);
  return 0;
}

int ecw_ctx_graph_stats(ecw_ctx* c, int64_t* hits, int64_t* captures) {
  if (!c) return -1;
  if (hits) *hits = c->graph_hits;
  if (captures) *captures = c->graph_captures;
  return 0;
}

int ecw_ctx_set_int8_splitk(ecw_ctx* c, int64_t min_k) {
  if (!c) return -1;
  c->z.oz_splitk_min_k = min_k;
  drop_plans(c);
  return 0;
}

int ecw_ctx_test_assume_vvvv_planes(ecw_ctx* c) {
  if (!c || c->z.oz_ns <= 0) return -1;
  c->z.vvvv_planes = true;
  drop_plans(c);
  return 0;
}

int ecw_ctx_test_assume_ovvv_planes(ecw_ctx* c) {
  if (!c || c->z.oz_ns <= 0 || (c->z.nocc % 8) || (c->z.nvir % 8)) return -1;
  c->z.ovvv_planes = true;
  drop_plans(c);
  return 0;
}

int ecw_ctx_test_cut_cache_min(ecw_ctx* c, int64_t min_elems) {
  if (!c || min_elems < 1) return -1;
  c->z.cut_cache_min_elems = min_elems;
  drop_plans(c);
  return 0;
}

int ecw_eris_vvvv_planes(ecw_ctx* c, const double* rows, int64_t row0, int64_t nrows, void* stream) {
  return guarded(c, [&] {
    require_device();
    if (c->z.oz_ns <= 0) throw Fail("ecw_eris_vvvv_planes: the INT8 GEMM engine is off (ecw_ctx_set_gemm)");
    if (!c->ptr[S_VVVV_OZ] || !c->ptr[S_VVVV_OZS]) throw Fail("slots 'vvvv_oz' / 'vvvv_ozs' are not bound");
    const int64_t pv = npair(c->z.nvir);
    const int64_t nsh = slot_elems(c->z, S_VVVV_P) / std::max<int64_t>(pv, 1);
    if (row0 < 0 || nrows < 0 || row0 + nrows > nsh) throw Fail("ecw_eris_vvvv_planes: row range outside this rank's shard");
    if (nrows > 0)
      ck(launch_ozaki_split(rows, nrows, pv, pv, 1, c->z.oz_ns, reinterpret_cast<int8_t*>(c->ptr[S_VVVV_OZ]),
                            c->ptr[S_VVVV_OZS], static_cast<cudaStream_t>(stream), row0, nsh), "ozaki_split(vvvv)");
    if (row0 + nrows == nsh) {          // last chunk: from now on plans read the planes, not "vvvv_p"
      c->z.vvvv_planes = true;
      drop_plans(c);
    }
  });
}

int ecw_eris_ovvv_planes(ecw_ctx* c, void* stream) {
  return guarded(c, [&] {
    require_device();
    if (c->z.oz_ns <= 0) throw Fail("ecw_eris_ovvv_planes: the INT8 GEMM engine is off (ecw_ctx_set_gemm)");
    const int64_t o = c->z.nocc, v = c->z.nvir, pv = npair(v);
    if ((o % 8) || (v % 8)) throw Fail("ecw_eris_ovvv_planes: needs nocc % 8 == 0 and nvir % 8 == 0");
    for (int s : {S_OVVV_P, S_OVVV_OZ1, S_OVVV_OZ1S, S_OVVV_OZ2, S_OVVV_OZ2S})
      if (!c->ptr[s]) throw Fail(std::string("slot '") + slot_name(s) + "' is not bound");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    // OZ1: rows (m,a), k = ef_p (contiguous);  OZ2: rows ef_p (contiguous), k = (m, a) with a padded to 32 per m
    ck(launch_ozaki_split2(c->ptr[S_OVVV_P], o * v, 1, pv, pv, 0, 1, c->z.oz_ns,
                           reinterpret_cast<int8_t*>(c->ptr[S_OVVV_OZ1]), c->ptr[S_OVVV_OZ1S], st), "ozaki_split(ovvv 1)");
    ck(launch_ozaki_split2(c->ptr[S_OVVV_P], pv, o, v, 1, v * pv, pv, c->z.oz_ns,
                           reinterpret_cast<int8_t*>(c->ptr[S_OVVV_OZ2]), c->ptr[S_OVVV_OZ2S], st), "ozaki_split(ovvv 2)");
    c->z.ovvv_planes = true;          // from now on plans read the planes, not "ovvv_p"
    drop_plans(c);
  });
}

int ecw_resume(ecw_ctx* c, void* stream) {
  return guarded_rc(c, [&] {
    if (!c->run_plan_ptr) throw Fail("ecw_resume: no call in flight");
    return run_plan_resume(c, static_cast<cudaStream_t>(stream));
  });
}

int ecw_pending_collective(ecw_ctx* c, int64_t* desc6) {
  if (!c || !c->run_plan_ptr) return -1;
  for (int i = 0; i < 6; ++i) desc6[i] = c->pending[i];
  return 0;
}

int64_t ecw_slot_elems(ecw_ctx* c, const char* slot) {
  if (!c) return -1;
  int s = slot_by_name(slot);
  if (s < 0) { c->err = std::string("unknown slot '") + slot + "'"; return -1; }
  return slot_elems(c->z, s);
}

int ecw_bind(ecw_ctx* c, const char* slot, void* p) {
  return guarded(c, [&] {
    int s = slot_by_name(slot);
    if (s < 0) throw Fail(std::string("unknown slot '") + slot + "'");
    c->ptr[s] = static_cast<double*>(p);
  });
}

int64_t ecw_workspace_bytes(ecw_ctx* c, const char* func, int flags) {
  int64_t r = -1;
  guarded(c, [&] { r = get_plan(c, func, flags).workspace_elems() * 8; });
  return r;
}

int ecw_set_workspace(ecw_ctx* c, void* p, int64_t bytes) {
  return guarded(c, [&] {
    c->ptr[S_WS] = static_cast<double*>(p);
    c->ws_bytes = bytes;
  });
}

int ecw_eris_pack_from_dense(ecw_ctx* c, const double* ovov, const double* vvvv, void* stream) {
  return guarded(c, [&] {
    require_device();
    if (c->z.world != 1) throw Fail("ecw_eris_pack_from_dense: pack before ecw_ctx_set_shard (vvvv_p must be bound whole)");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const int64_t o = c->z.nocc, v = c->z.nvir;
    for (int s : {S_OOOO, S_OOOV, S_OOVV, S_OVVV, S_OOVV_PH, S_OVOV_PH, S_OOOO_P, S_OOVV_P, S_OVVV_P, S_VVVV_P})
      if (!c->ptr[s]) throw Fail(std::string("slot '") + slot_name(s) + "' is not bound");
    ck(launch_eris_layouts_from_dense(c->ptr[S_OOVV], ovov, c->ptr[S_OOVV_PH], c->ptr[S_OVOV_PH], (int)o, (int)v, st),
       "ph layouts");
    auto pk = [&](const double* src, int64_t d0, int64_t d1, int64_t d2, int64_t d3, int flags, double* dst) {
      PackArgs a{};
      a.src = src; a.dst = dst; a.d0 = d0; a.d1 = d1; a.d2 = d2; a.d3 = d3;
      a.s3 = 1; a.s2 = d3; a.s1 = d2 * d3; a.s0 = d1 * d2 * d3;
      a.ld = (flags & 2) ? npair(d2) : d2 * d3;
      a.flags = flags; a.alpha = 1.0; a.beta = 0.0;
      ck(launch_pack(a, st), "pack");
    };
    pk(c->ptr[S_OOOO], o, o, o, o, 3, c->ptr[S_OOOO_P]);
    pk(c->ptr[S_OOVV], o, o, v, v, 3, c->ptr[S_OOVV_P]);
    pk(c->ptr[S_OVVV], o, v, v, v, 2, c->ptr[S_OVVV_P]);
    pk(vvvv, v, v, v, v, 3, c->ptr[S_VVVV_P]);
  });
}

int ecw_eris_synthetic(ecw_ctx* c, double scale, void* stream) {
  return guarded(c, [&] {
    require_device();
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const int o = (int)c->z.nocc, v = (int)c->z.nvir;
    const int64_t po = npair(o), pv = npair(v);
    struct { int slot, kind; int64_t rows; } tab[] = {
        {S_OOOO, SY_OOOO, o}, {S_OOOV, SY_OOOV, o}, {S_OOVV, SY_OOVV, o}, {S_OOVV_PH, SY_OOVV_PH, o},
        {S_OVOV_PH, SY_OVOV_PH, o}, {S_OVVV, SY_OVVV, o}, {S_OOOO_P, SY_OOOO_P, po}, {S_OOVV_P, SY_OOVV_P, po},
        {S_OVVV_P, SY_OVVV_P, o}, {S_VVVV_P, SY_VVVV_P, pv}};
    for (auto& t : tab) {
      // INT8 engine: the packed vvvv exists only as digit planes, cut chunk by chunk by the caller
      // (ecw_synth_tensor rows -> ecw_eris_vvvv_planes)
      if (t.slot == S_VVVV_P && !c->ptr[t.slot] && c->z.oz_ns > 0) continue;
      if (!c->ptr[t.slot]) throw Fail(std::string("slot '") + slot_name(t.slot) + "' is not bound");
      int64_t r0 = 0, nr = t.rows;
      if (t.slot == S_VVVV_P) {   // this rank's rows of the packed virtual pair index
        const int64_t nshmax = (pv + c->z.world - 1) / c->z.world;
        r0 = std::min<int64_t>(pv, (int64_t)c->z.rank * nshmax);
        nr = std::min<int64_t>(pv, r0 + nshmax) - r0;
      }
      ck(launch_synth(t.kind, c->ptr[t.slot], o, v, r0, nr, scale, st), "synth");
    }
  });
}

int ecw_synth_tensor(int kind, double* out, int nocc, int nvir, int64_t row0, int64_t nrows, double scale,
                     void* stream) {
  return guarded(nullptr, [&] {
    require_device();
    ck(launch_synth(kind, out, nocc, nvir, row0, nrows, scale, static_cast<cudaStream_t>(stream)), "synth");
  });
}

int ecw_ccsd_tupdate(ecw_ctx* c, const double* t1, const double* t2, const double* fsp, const double* fock,
                     int flags, double alpha, double* t1new, double* t2new, void* stream) {
  return guarded_rc(c, [&] {
    require_device();
    c->ptr[S_T1] = const_cast<double*>(t1); c->ptr[S_T2] = const_cast<double*>(t2);
    c->ptr[S_FSP] = const_cast<double*>(fsp); c->ptr[S_FOCK] = const_cast<double*>(fock);
    c->ptr[S_OUT1] = t1new; c->ptr[S_OUT2] = t2new;
    return run_plan(c, get_plan(c, "tupdate", flags), alpha, static_cast<cudaStream_t>(stream), true);
  });
}

int ecw_ccsd_lupdate(ecw_ctx* c, const double* t1, const double* t2, const double* l1, const double* l2,
                     const double* fsp, const double* fock, int flags, double alpha, double* l1new, double* l2new,
                     void* stream) {
  return guarded_rc(c, [&] {
    require_device();
    c->ptr[S_T1] = const_cast<double*>(t1); c->ptr[S_T2] = const_cast<double*>(t2);
    c->ptr[S_L1] = const_cast<double*>(l1); c->ptr[S_L2] = const_cast<double*>(l2);
    c->ptr[S_FSP] = const_cast<double*>(fsp); c->ptr[S_FOCK] = const_cast<double*>(fock);
    c->ptr[S_OUT1] = l1new; c->ptr[S_OUT2] = l2new;
    return run_plan(c, get_plan(c, "lupdate", flags), alpha, static_cast<cudaStream_t>(stream), true);
  });
}

int ecw_ccsd_gamma(ecw_ctx* c, const double* t1, const double* t2, const double* l1, const double* l2, double* rdm1,
                   void* stream) {
  return guarded_rc(c, [&] {
    require_device();
    c->ptr[S_T1] = const_cast<double*>(t1); c->ptr[S_T2] = const_cast<double*>(t2);
    c->ptr[S_L1] = const_cast<double*>(l1); c->ptr[S_L2] = const_cast<double*>(l2);
    c->ptr[S_RDM1] = rdm1;
    return run_plan(c, get_plan(c, "gamma", 0), 0.0, static_cast<cudaStream_t>(stream), true);
  });
}

int ecw_ccsd_energy(ecw_ctx* c, const double* t1, const double* t2, const double* fsp, double* e_out, void* stream) {
  return guarded_rc(c, [&] {
    require_device();
    c->ptr[S_T1] = const_cast<double*>(t1); c->ptr[S_T2] = const_cast<double*>(t2);
    c->ptr[S_FSP] = const_cast<double*>(fsp);
    if (!c->ptr[S_SCAL]) throw Fail("slot 'scal' is not bound");
    c->copy_scal_to = e_out;
    return run_plan(c, get_plan(c, "energy", 0), 0.0, static_cast<cudaStream_t>(stream), true);
  });
}

// ---- ECW-CCS intermediates (csrc/ccs_plan.cpp): one cached plan each
int ecw_ccs_t1inter(ecw_ctx* c, const double* ts, const double* fsp, double* F, void* stream) {
  return guarded_rc(c, [&] {
    require_device();
    c->ptr[S_T1] = const_cast<double*>(ts); c->ptr[S_FSP] = const_cast<double*>(fsp);
    c->ptr[S_RDM1] = F;
    return run_plan(c, get_plan(c, "ccs_t1inter", 0), 0.0, static_cast<cudaStream_t>(stream), true);
  });
}

int ecw_ccs_l1inter(ecw_ctx* c, const double* ts, const double* fsp, int e_term, double* F, double* W, double* e_out,
                    void* stream) {
  return guarded_rc(c, [&] {
    require_device();
    c->ptr[S_T1] = const_cast<double*>(ts); c->ptr[S_FSP] = const_cast<double*>(fsp);
    c->ptr[S_RDM1] = F; c->ptr[S_OUT2] = W;
    if (e_term) {
      if (!c->ptr[S_SCAL]) throw Fail("slot 'scal' is not bound");
      c->copy_scal_to = e_out;
    }
    return run_plan(c, get_plan(c, "ccs_l1inter", e_term ? 1 : 0), 0.0, static_cast<cudaStream_t>(stream), true);
  });
}

static int ccs_es_inter(ecw_ctx* c, const char* func, const double* ts, const double* fsp, const double* vm, double* F,
                        double* W, double* X, double* e_out, void* stream) {
  return guarded_rc(c, [&] {
    require_device();
    if (!c->ptr[S_SCAL]) throw Fail("slot 'scal' is not bound");
    c->ptr[S_T1] = const_cast<double*>(ts); c->ptr[S_FSP] = const_cast<double*>(fsp);
    c->ptr[S_FOCK] = const_cast<double*>(vm);
    c->ptr[S_RDM1] = F; c->ptr[S_OUT2] = W; c->ptr[S_OUT1] = X;
    c->copy_scal_to = e_out;
    return run_plan(c, get_plan(c, func, vm ? 1 : 0), 0.0, static_cast<cudaStream_t>(stream), true);
  });
}

int ecw_ccs_r1inter(ecw_ctx* c, const double* ts, const double* fsp, const double* vm, double* F, double* W, double* X,
                    double* e_out, void* stream) {
  return ccs_es_inter(c, "ccs_r1inter", ts, fsp, vm, F, W, X, e_out, stream);
}

int ecw_ccs_esl1inter(ecw_ctx* c, const double* ts, const double* fsp, const double* vm, double* F, double* W, double* X,
                      double* e_out, void* stream) {
  return ccs_es_inter(c, "ccs_esl1inter", ts, fsp, vm, F, W, X, e_out, stream);
}

int ecw_antisym_defect(const double* x, int nocc, int nvir, double* out, void* stream) {
  return guarded(nullptr, [&] {
    require_device();
    ck(launch_antisym_defect(x, nocc, nvir, out, static_cast<cudaStream_t>(stream)), "antisym_defect");
  });
}

int ecw_subdiff(const double* eq, const double* var, double alpha, double* out, int64_t n, void* stream) {
  return guarded(nullptr, [&] {
    require_device();
    ck(launch_subdiff(eq, var, alpha, out, n, static_cast<cudaStream_t>(stream)), "subdiff");
  });
}

int64_t ecw_plan_dump(ecw_ctx* c, const char* func, int flags, char* buf, int64_t buflen) {
  int64_t r = -1;
  guarded(c, [&] {
    std::string s = get_plan(c, func, flags).dump_json();
    if ((int64_t)s.size() + 1 > buflen) { r = -(int64_t)(s.size() + 1); return; }
    memcpy(buf, s.c_str(), s.size() + 1);
    r = (int64_t)s.size();
  });
  return r;
}

int64_t ecw_plan_dump_contract(ecw_ctx* c, double alpha, const ecw_tensor* A, const char* sa, const ecw_tensor* B,
                               const char* sb, double beta, const ecw_tensor* C, const char* sc, char* buf,
                               int64_t buflen) {
  int64_t r = -1;
  guarded(c, [&] {
    // host only: the lowering ecw_op_contract would launch (operands named a0, a1, b0; ptr fields are ignored)
    auto desc = [](const ecw_tensor* t, int slot) {
      Tensor x;
      if (t->nd < 0 || t->nd > MAXD) throw Fail("ecw_tensor: rank out of range");
      x.slot = slot;
      x.nd = t->nd;
      for (int i = 0; i < t->nd; ++i) { x.dim[i] = t->dim[i]; x.str[i] = t->str[i]; }
      if (x.nd == 0) { x.nd = 1; x.dim[0] = 1; x.str[0] = 1; }
      return x;
    };
    Plan P;
    P.oz_ns = c->z.oz_ns; P.oz_min_flops = c->z.oz_min_flops; P.nocc = c->z.nocc; P.nvir = c->z.nvir;
    P.oz_splitk_min_k = c->z.oz_splitk_min_k;
    P.contract(alpha, desc(A, S_A0), sa, desc(B, S_A1), sb, beta, desc(C, S_B0), sc, "op");
    std::string s = P.dump_json();
    if ((int64_t)s.size() + 1 > buflen) { r = -(int64_t)(s.size() + 1); return; }
    memcpy(buf, s.c_str(), s.size() + 1);
    r = (int64_t)s.size();
  });
  return r;
}

double ecw_plan_flops(ecw_ctx* c, const char* func, int flags) {
  double r = -1.0;
  guarded(c, [&] { r = get_plan(c, func, flags).gemm_flops; });
  return r;
}

int64_t ecw_plan_launches(ecw_ctx* c, const char* func, int flags) {
  int64_t r = -1;
  guarded(c, [&] {
    const Plan& P = get_plan(c, func, flags);
    int64_t n = 0;
    for (auto& op : P.ops)
      n += (op.kind == OP_DOT || op.kind == OP_OZ_SPLIT) ? 2 : ((op.kind == OP_ALLGATHER || op.kind == OP_ALLTOALL) ? 0 : 1);
    r = n;
  });
  return r;
}

int ecw_dgemm(int ta, int tb, int64_t M, int64_t N, int64_t K, double alpha, const double* A, int64_t lda,
              const double* B, int64_t ldb, double beta, double* C, int64_t ldc, int cfg, void* stream) {
  return guarded(nullptr, [&] {
    require_device();
    GemmArgs g{};
    g.A = A; g.B = B; g.C = C; g.M = M; g.N = N; g.K = K; g.lda = lda; g.ldb = ldb; g.ldc = ldc;
    g.batch = 1; g.splitk = 1; g.kchunk = K; g.ta = ta; g.tb = tb; g.alpha = alpha; g.beta = beta;
    ck(launch_gemm(g, static_cast<cudaStream_t>(stream), cfg), "dgemm");
  });
}

// ---- FP64 GEMM on the INT8 tcgen05 pipe (ozaki.cu): raw entry points for tools/ and tests/
int64_t ecw_ozaki_plane_bytes(int64_t R, int64_t K, int ns) { return ozaki_plane_bytes(R, K, ns); }
int64_t ecw_ozaki_padded_rows(int64_t R) { return ozaki_padded_rows(R); }
int64_t ecw_ozaki_stat_elems(int64_t R) { return ozaki_stat_elems(R, 1); }
int64_t ecw_ozaki_stat_elems2(int64_t R, int64_t K1) { return ozaki_stat_elems(R, K1); }
int64_t ecw_ozaki_plane_bytes2(int64_t R, int64_t K1, int64_t K2, int ns) { return ozaki_plane_bytes2(R, K1, K2, ns); }
int ecw_ozaki_tile_n(int ns) { return ozaki_tile_n(ns); }

int ecw_ozaki_split(const double* X, int64_t R, int64_t K, int64_t rs, int64_t ks, int ns, void* planes, double* scale,
                    void* stream) {
  return guarded(nullptr, [&] {
    require_device();
    ck(launch_ozaki_split(X, R, K, rs, ks, ns, static_cast<int8_t*>(planes), scale, static_cast<cudaStream_t>(stream)),
       "ozaki_split");
  });
}

int ecw_ozaki_split2(const double* X, int64_t R, int64_t K1, int64_t K2, int64_t rs, int64_t ks1, int64_t ks2, int ns,
                     void* planes, double* stats, void* stream) {
  return guarded(nullptr, [&] {
    require_device();
    ck(launch_ozaki_split2(X, R, K1, K2, rs, ks1, ks2, ns, static_cast<int8_t*>(planes), stats,
                           static_cast<cudaStream_t>(stream)), "ozaki_split2");
  });
}

int ecw_ozaki_gemm_batched(const void* pa, const double* sa, int64_t a_rows, const void* pb, const double* sb,
                           int64_t b_rows, int64_t M, int64_t N, int64_t K, double* C, int64_t crs, int64_t ccs,
                           double alpha, double beta, int ns, const int64_t* bt14, void* stream) {
  return guarded(nullptr, [&] {
    require_device();
    OzBatch bt{};
    bt.batch = bt14[0];
    bt.a_row0 = bt14[1]; bt.a_rowb = bt14[2]; bt.b_row0 = bt14[3]; bt.b_rowb = bt14[4];
    bt.a_kb0 = bt14[5]; bt.a_kbb = bt14[6]; bt.b_kb0 = bt14[7]; bt.b_kbb = bt14[8];
    bt.a_t0 = bt14[9]; bt.a_tb = bt14[10]; bt.b_t0 = bt14[11]; bt.b_tb = bt14[12];
    bt.c_b = bt14[13];
    bt.nkb = bt14[14];
    ck(launch_ozaki_gemm_batched(static_cast<const int8_t*>(pa), sa, a_rows, static_cast<const int8_t*>(pb), sb, b_rows, M,
                                 N, K, C, crs, ccs, alpha, beta, ns, bt, static_cast<cudaStream_t>(stream), 0),
       "ozaki_gemm_batched");
  });
}

int ecw_ozaki_split_rows(const double* X, int64_t R, int64_t K, int64_t rs, int64_t ks, int ns, void* planes,
                         double* scale, int64_t row0, int64_t total_rows, void* stream) {
  return guarded(nullptr, [&] {
    require_device();
    ck(launch_ozaki_split(X, R, K, rs, ks, ns, static_cast<int8_t*>(planes), scale, static_cast<cudaStream_t>(stream),
                          row0, total_rows),
       "ozaki_split_rows");
  });
}

int ecw_ozaki_gemm(const void* pa, const double* sa, const void* pb, const double* sb, int64_t M, int64_t N, int64_t K,
                   double* C, int64_t crs, int64_t ccs, double alpha, double beta, int ns, void* stream) {
  return guarded(nullptr, [&] {
    require_device();
    ck(launch_ozaki_gemm(static_cast<const int8_t*>(pa), sa, static_cast<const int8_t*>(pb), sb, M, N, K, C, crs, ccs,
                         alpha, beta, ns, static_cast<cudaStream_t>(stream), 0),
       "ozaki_gemm");
  });
}

// ---- primitive device ops (the CCS host class and the GCC intermediate getters are sequences of these)
namespace {

Tensor from_desc(const ecw_tensor* t, int slot) {
  Tensor r;
  if (!t || !t->ptr) return r;
  if (t->nd < 0 || t->nd > MAXD) throw Fail("ecw_tensor: rank out of range");
  r.slot = slot;
  r.off = 0;
  r.nd = t->nd;
  for (int i = 0; i < t->nd; ++i) { r.dim[i] = t->dim[i]; r.str[i] = t->str[i]; }
  if (r.nd == 0) { r.nd = 1; r.dim[0] = 1; r.str[0] = 1; }
  return r;
}

int run_op_plan(ecw_ctx* c, Plan& P, double alpha_rt, void* stream) {
  if (P.workspace_elems() * 8 > c->ws_bytes) {
    c->need_ws = P.workspace_elems() * 8;
    c->err = "workspace too small for this op (ecw_op_workspace_needed)";
    return -2;
  }
  return run_plan(c, P, alpha_rt, static_cast<cudaStream_t>(stream));
}

}  // namespace

int64_t ecw_op_workspace_needed(ecw_ctx* c) { return c ? c->need_ws : -1; }

int ecw_op_contract(ecw_ctx* c, double alpha, const ecw_tensor* A, const char* sa, const ecw_tensor* B, const char* sb,
                    double beta, const ecw_tensor* C, const char* sc, void* stream) {
  return guarded_rc(c, [&] {
    require_device();
    Plan P;
    P.oz_ns = c->force_dmma ? 0 : c->z.oz_ns; P.oz_min_flops = c->z.oz_min_flops; P.nocc = c->z.nocc; P.nvir = c->z.nvir;
    P.oz_splitk_min_k = c->z.oz_splitk_min_k;
    c->ptr[S_A0] = (double*)A->ptr; c->ptr[S_A1] = (double*)B->ptr; c->ptr[S_B0] = (double*)C->ptr;
    P.contract(alpha, from_desc(A, S_A0), sa, from_desc(B, S_A1), sb, beta, from_desc(C, S_B0), sc, "op");
    c->op_plan = std::move(P);
    return run_op_plan(c, c->op_plan, 0.0, stream);
  });
}

int ecw_op_axpby(ecw_ctx* c, double alpha, const ecw_tensor* A, const char* sa, double beta, const ecw_tensor* C,
                 const char* sc, void* stream) {
  return guarded_rc(c, [&] {
    require_device();
    Plan P;
    c->ptr[S_A0] = (double*)A->ptr; c->ptr[S_B0] = (double*)C->ptr;
    P.permute(alpha, from_desc(A, S_A0), sa, beta, from_desc(C, S_B0), sc, "op");
    c->op_plan = std::move(P);
    return run_op_plan(c, c->op_plan, 0.0, stream);
  });
}

int ecw_op_mul(ecw_ctx* c, double alpha, const ecw_tensor* A, const ecw_tensor* B, double beta, const ecw_tensor* C,
               void* stream) {
  return guarded_rc(c, [&] {
    require_device();
    Plan P;
    Tensor a = from_desc(A, S_A0), b = from_desc(B, S_A1), cc = from_desc(C, S_B0);
    if (A && A->ptr) c->ptr[S_A0] = (double*)A->ptr;
    if (B && B->ptr) c->ptr[S_A1] = (double*)B->ptr;
    c->ptr[S_B0] = (double*)C->ptr;
    for (const Tensor* t : {&a, &b})
      if (t->valid()) {
        if (t->nd != cc.nd) throw Fail("ecw_op_mul: rank mismatch");
        for (int i = 0; i < cc.nd; ++i) if (t->dim[i] != cc.dim[i]) throw Fail("ecw_op_mul: shape mismatch");
      }
    P.ewise(0, a, b, cc, alpha, beta);
    c->op_plan = std::move(P);
    return run_op_plan(c, c->op_plan, 0.0, stream);
  });
}

int ecw_op_unpack(ecw_ctx* c, double alpha, const ecw_tensor* A2, int flags, double beta, const ecw_tensor* C4,
                  void* stream) {
  return guarded_rc(c, [&] {
    require_device();
    Plan P;
    c->ptr[S_A0] = (double*)A2->ptr; c->ptr[S_B0] = (double*)C4->ptr;
    P.unpack(alpha, from_desc(A2, S_A0), flags, beta, from_desc(C4, S_B0));
    c->op_plan = std::move(P);
    return run_op_plan(c, c->op_plan, 0.0, stream);
  });
}

int ecw_op_diag_shift(ecw_ctx* c, const ecw_tensor* Cm, double alpha, const ecw_tensor* fock, int64_t offset,
                      void* stream) {
  return guarded_rc(c, [&] {
    require_device();
    Plan P;
    c->ptr[S_B0] = (double*)Cm->ptr; c->ptr[S_FOCK] = (double*)fock->ptr;
    P.diag_add(from_desc(Cm, S_B0), alpha, from_desc(fock, S_FOCK), offset);
    c->op_plan = std::move(P);
    return run_op_plan(c, c->op_plan, 0.0, stream);
  });
}

int ecw_op_denom(ecw_ctx* c, const ecw_tensor* resid, const ecw_tensor* amp, const ecw_tensor* fock, int nocc,
                 int mode_flags, double alpha, double shift, const ecw_tensor* out, void* stream) {
  return guarded_rc(c, [&] {
    require_device();
    Plan P;
    c->ptr[S_A0] = (double*)resid->ptr; c->ptr[S_A1] = (double*)amp->ptr; c->ptr[S_FOCK] = (double*)fock->ptr;
    c->ptr[S_B0] = (double*)out->ptr;
    Tensor r = from_desc(resid, S_A0);
    const int rank = r.nd == 4 ? 4 : 2;
    P.finish(r, from_desc(amp, S_A1), from_desc(fock, S_FOCK), nocc, rank, (mode_flags & ECW_HAS_ALPHA) ? 1 : 0,
             (mode_flags & ECW_EQUATION) ? 1 : 0, alpha, from_desc(out, S_B0), shift,
             (mode_flags & ECW_SUBDIFF_SINGLES) ? 1 : 0);
    c->op_plan = std::move(P);
    return run_op_plan(c, c->op_plan, alpha, stream);
  });
}

int ecw_op_dot(ecw_ctx* c, double alpha, const ecw_tensor* A, const ecw_tensor* B, double beta, double* out_dev,
               void* stream) {
  return guarded_rc(c, [&] {
    require_device();
    if (!c->ptr[S_SCAL]) throw Fail("slot 'scal' is not bound");
    Plan P;
    c->ptr[S_A0] = (double*)A->ptr; c->ptr[S_A1] = (double*)B->ptr;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (beta != 0.0) ck(cudaMemcpyAsync(c->ptr[S_SCAL] + 1, out_dev, sizeof(double), cudaMemcpyDeviceToDevice, st), "dot in");
    Tensor a = from_desc(A, S_A0), b = from_desc(B, S_A1);
    auto packed = [](const Tensor& t) {                      // row-major without gaps: read in place
      int64_t want = 1;
      for (int i = t.nd - 1; i >= 0; --i) {
        if (t.dim[i] != 1 && t.str[i] != want) return false;
        want *= t.dim[i];
      }
      return true;
    };
    Tensor ad = a, bd = b;
    if (!packed(a)) { ad = P.tmpv(std::vector<int64_t>(a.dim, a.dim + a.nd)); P.axpby(1.0, a, 0.0, ad); }
    if (!packed(b)) { bd = P.tmpv(std::vector<int64_t>(b.dim, b.dim + b.nd)); P.axpby(1.0, b, 0.0, bd); }
    P.dot(alpha, ad, bd, beta, 1);
    c->op_plan = std::move(P);
    int rc = run_op_plan(c, c->op_plan, 0.0, stream);
    if (rc == 0) ck(cudaMemcpyAsync(out_dev, c->ptr[S_SCAL] + 1, sizeof(double), cudaMemcpyDeviceToDevice, st), "dot out");
    return rc;
  });
}

int ecw_conv_check(const double* a, const double* b, const double* prev, double* conv, int64_t n, double* scratch1024,
                   double* sumsq, int accumulate, void* stream) {
  return guarded(nullptr, [&] {
    require_device();
    ck(launch_conv(a, b, prev, conv, n, scratch1024, 1024, sumsq, accumulate ? 1.0 : 0.0, static_cast<cudaStream_t>(stream)),
       "conv_check");
  });
}

int ecw_vexp_mat(const double* rdm1, const double* target, const double* fock, double L, double* vexp, double* fsp,
                 double* stats2, int64_t n, void* stream) {
  return guarded(nullptr, [&] {
    require_device();
    if (!rdm1 || !target || !fock || !vexp || !fsp || !stats2) throw Fail("ecw_vexp_mat: null pointer");
    ck(launch_vexp_mat(rdm1, target, fock, L, vexp, fsp, stats2, n, static_cast<cudaStream_t>(stream)), "vexp_mat");
  });
}

int ecw_ft_aopair(const double* prim, int64_t nprim, const int64_t* ao_first, int nao, const double* G, int64_t nG,
                  double* out, void* stream) {
  return guarded(nullptr, [&] {
    require_device();
    if (!prim || !ao_first || !G || !out) throw Fail("ecw_ft_aopair: null pointer");
    if (nprim < 1 || nao < 1 || nG < 1) throw Fail("ecw_ft_aopair: empty primitive table, basis or G list");
    ck(launch_ft_aopair(prim, nprim, ao_first, nao, G, nG, out, static_cast<cudaStream_t>(stream)), "ft_aopair");
  });
}

namespace {
// ecw_vexp_sf workspace: X / Y [2nao, n] | D [nao, nao] | coef [2 nG] | V_AO [nao, nao], each padded to 32 doubles
struct SfWorkspace {
  int64_t x, d, coef, v, total;
  SfWorkspace(int n, int nao, int64_t nG) {
    auto pad = [](int64_t e) { return (e + 31) / 32 * 32; };
    x = 0;
    d = x + pad(2LL * nao * n);
    coef = d + pad((int64_t)nao * nao);
    v = coef + pad(2 * nG);
    total = v + pad((int64_t)nao * nao);
  }
};
}  // namespace

int64_t ecw_vexp_sf_workspace_bytes(int n, int nao, int64_t nG) {
  if (n < 1 || nao < 1 || nG < 1) return -1;
  return 8 * SfWorkspace(n, nao, nG).total;
}

extern "C++" {
namespace {
// The pipeline shared by the 'F' and 'Fobs' potentials: D = C_a gamma C_a^T + C_b gamma C_b^T, F_calc = planes . vec(D),
// coef_step(F_calc, coef) forms the GEMV coefficients [2 nG], V_AO = planes^T . coef, vexp = C_g^T blockdiag(V_AO,
// V_AO) C_g, fsp = fock - vexp and stats[1] = max |vexp|.  Stream-ordered, no synchronisation.
template <typename CoefStep>
void vexp_planes(const double* rdm1, int n, const double* mo_coeff_g, int nao, const double* ft, int64_t nG,
                 const double* fock, double* vexp, double* fsp, double* F_calc, double* stats, double* workspace,
                 cudaStream_t st, CoefStep coef_step) {
  const SfWorkspace w(n, nao, nG);
  double* X = workspace + w.x;                 // C_g gamma, later blockdiag(V, V) C_g
  double* D = workspace + w.d;
  double* coef = workspace + w.coef;
  double* V = workspace + w.v;
  const int64_t n2 = (int64_t)nao * nao;
  const double* Ca = mo_coeff_g;               // alpha rows of C_g
  const double* Cb = mo_coeff_g + (int64_t)nao * n;
  auto gemm = [&](int ta, int tb, int64_t M, int64_t N, int64_t K, const double* A, int64_t lda, const double* B,
                  int64_t ldb, double beta, double* C, int64_t ldc) {
    GemmArgs g{};
    g.A = A; g.B = B; g.C = C; g.M = M; g.N = N; g.K = K; g.lda = lda; g.ldb = ldb; g.ldc = ldc;
    g.batch = 1; g.splitk = 1; g.kchunk = K; g.ta = ta; g.tb = tb; g.alpha = 1.0; g.beta = beta;
    ck(launch_gemm(g, st), "vexp_sf gemm");
  };
  // D = C_a gamma C_a^T + C_b gamma C_b^T: the spin-summed AO density
  gemm(0, 0, 2LL * nao, n, n, mo_coeff_g, n, rdm1, n, 0.0, X, n);
  gemm(0, 1, nao, nao, n, X, n, Ca, n, 0.0, D, nao);
  gemm(0, 1, nao, nao, n, X + (int64_t)nao * n, n, Cb, n, 1.0, D, nao);
  // F_calc [Re | Im] = planes [2 nG, nao^2] . vec(D)
  gemm(0, 0, 2 * nG, 1, n2, ft, n2, D, 1, 0.0, F_calc, 1);
  coef_step(F_calc, coef);
  // V_AO = planes^T . coef,  vexp = C_g^T blockdiag(V_AO, V_AO) C_g
  gemm(1, 0, n2, 1, 2 * nG, ft, n2, coef, 1, 0.0, V, 1);
  gemm(0, 0, nao, n, nao, V, nao, Ca, n, 0.0, X, n);
  gemm(0, 0, nao, n, nao, V, nao, Cb, n, 0.0, X + (int64_t)nao * n, n);
  gemm(1, 0, n, n, 2LL * nao, mo_coeff_g, n, X, n, 0.0, vexp, n);
  ck(launch_sf_finish(vexp, fock, fsp, stats, (int64_t)n * n, st), "vexp_sf finish");
}
}  // namespace
}  // extern "C++"

int ecw_vexp_sf(const double* rdm1, int n, const double* mo_coeff_g, int nao, const double* ft, int64_t nG,
                const double* F_exp, double L, const double* fock, double* vexp, double* fsp, double* F_calc,
                double* stats2, double* workspace, void* stream) {
  return guarded(nullptr, [&] {
    require_device();
    if (!rdm1 || !mo_coeff_g || !ft || !F_exp || !fock || !vexp || !fsp || !F_calc || !stats2 || !workspace)
      throw Fail("ecw_vexp_sf: null pointer");
    if (n < 1 || nao < 1 || nG < 1) throw Fail("ecw_vexp_sf: empty rdm1, basis or reflection list");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    vexp_planes(rdm1, n, mo_coeff_g, nao, ft, nG, fock, vexp, fsp, F_calc, stats2, workspace, st,
                [&](const double* fc, double* coef) {
                  ck(launch_sf_coef(F_exp, fc, L, coef, stats2, nG, st), "vexp_sf coef");
                });
  });
}

int ecw_ft_aopair_cryst(const double* prim, int64_t nprim, const int64_t* ao_first, const int64_t* ao_atom, int nao,
                        const double* U, int natom, const double* Gs, const double* phase, int nsym, int64_t nG,
                        double* out, void* stream) {
  return guarded(nullptr, [&] {
    require_device();
    if (!prim || !ao_first || !ao_atom || !U || !Gs || !phase || !out) throw Fail("ecw_ft_aopair_cryst: null pointer");
    if (nprim < 1 || nao < 1 || nG < 1 || natom < 1) throw Fail("ecw_ft_aopair_cryst: empty table, basis or hkl list");
    if (nsym < 1 || nsym > 192) throw Fail("ecw_ft_aopair_cryst: nsym must lie in 1..192");
    ck(launch_ft_aopair_cryst(prim, nprim, ao_first, ao_atom, nao, U, natom, Gs, phase, nsym, nG, out,
                              static_cast<cudaStream_t>(stream)), "ft_aopair_cryst");
  });
}

int64_t ecw_vexp_sfobs_workspace_bytes(int n, int nao, int64_t nG) { return ecw_vexp_sf_workspace_bytes(n, nao, nG); }

int ecw_vexp_sfobs(const double* rdm1, int n, const double* mo_coeff_g, int nao, const double* ft, int64_t nG,
                   const double* F_obs, const double* weight, double k_fixed, double L, const double* fock, double* vexp,
                   double* fsp, double* F_calc, double* stats4, double* workspace, void* stream) {
  return guarded(nullptr, [&] {
    require_device();
    if (!rdm1 || !mo_coeff_g || !ft || !F_obs || !weight || !fock || !vexp || !fsp || !F_calc || !stats4 || !workspace)
      throw Fail("ecw_vexp_sfobs: null pointer");
    if (n < 1 || nao < 1 || nG < 1) throw Fail("ecw_vexp_sfobs: empty rdm1, basis or reflection list");
    if (!(k_fixed > 0.0) && nG < 2) throw Fail("ecw_vexp_sfobs: a refined scale needs at least two reflections");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    vexp_planes(rdm1, n, mo_coeff_g, nao, ft, nG, fock, vexp, fsp, F_calc, stats4, workspace, st,
                [&](const double* fc, double* coef) {
                  ck(launch_sfobs_coef(F_obs, weight, fc, L, k_fixed, coef, stats4, nG, st), "vexp_sfobs coef");
                });
  });
}

int64_t ecw_density_grid_workspace_bytes(int nao, int64_t npts) {
  if (nao < 1 || npts < 1) return -1;
  return 8 * density_grid_workspace_elems(nao, npts);
}

int ecw_density_grid(const double* prim, int64_t nprim, const int64_t* ao_first, int nao, const double* dm,
                     const double* box, int n1, int n2, int n3, double* out, double* workspace, void* stream) {
  return guarded(nullptr, [&] {
    require_device();
    if (!prim || !ao_first || !dm || !box || !out || !workspace) throw Fail("ecw_density_grid: null pointer");
    if (nprim < 1 || nao < 1) throw Fail("ecw_density_grid: empty primitive table or basis");
    if (n1 < 1 || n2 < 1 || n3 < 1) throw Fail("ecw_density_grid: grid dimensions must be positive");
    for (int c = 0; c < 12; ++c)
      if (!std::isfinite(box[c])) throw Fail("ecw_density_grid: origin and axes must be finite");
    ck(launch_density_grid(prim, nprim, ao_first, nao, dm, box, n1, n2, n3, out, workspace,
                           static_cast<cudaStream_t>(stream)), "density_grid");
  });
}

int ecw_fourier_map(const int64_t* hkl_half, const double* coef, int64_t N, double F000, double volume_bohr3, int n1,
                    int n2, int n3, double* out, void* stream) {
  return guarded(nullptr, [&] {
    require_device();
    if (!out || (N > 0 && (!hkl_half || !coef))) throw Fail("ecw_fourier_map: null pointer");
    if (N < 0) throw Fail("ecw_fourier_map: negative reflection count");
    if (n1 < 1 || n2 < 1 || n3 < 1 || n1 > FM_MAX_N || n2 > FM_MAX_N || n3 > FM_MAX_N)
      throw Fail("ecw_fourier_map: grid dimensions must lie in 1..512");
    if (!(volume_bohr3 > 0.0) || !std::isfinite(volume_bohr3) || !std::isfinite(F000))
      throw Fail("ecw_fourier_map: the volume must be positive and F000 finite");
    ck(launch_fourier_map(hkl_half, coef, N, F000, volume_bohr3, n1, n2, n3, out, static_cast<cudaStream_t>(stream)),
       "fourier_map");
  });
}

int ecw_profile_enable(ecw_ctx* c, int on) {
  if (!c) return -1;
  c->profile = on != 0;
  return 0;
}

int64_t ecw_profile_dump(ecw_ctx* c, char* buf, int64_t buflen) {
  int64_t r = -1;
  guarded(c, [&] {
    if (!c->last_plan || c->ev.empty()) throw Fail("no profiled run");
    ck(cudaEventSynchronize(c->ev.back()), "cudaEventSynchronize");
    static const char* kn[] = {"gemm", "reduce", "permute", "fill", "tau", "pack", "unpack", "finish",
                               "dot", "scale_dev", "diag_add", "rdm1", "ewise", "allgather", "oz_split", "oz_gemm",
                               "asym4", "alltoall"};
    std::ostringstream o;
    o << "[";
    for (size_t i = 0; i < c->last_plan->ops.size(); ++i) {
      float ms = 0.f;
      cudaEventElapsedTime(&ms, c->ev[i], c->ev[i + 1]);
      const Op& op = c->last_plan->ops[i];
      if (i) o << ",";
      o << "\n{\"kind\":\"" << kn[op.kind] << "\",\"ms\":" << ms << ",\"M\":" << op.M << ",\"N\":" << op.N
        << ",\"K\":" << op.K << ",\"batch\":" << op.batch << ",\"splitk\":" << op.splitk << ",\"elems\":"
        << (op.c.valid() ? op.c.size() : 0) << ",\"note\":\"" << op.note << "\"}";
    }
    o << "\n]";
    std::string s = o.str();
    if ((int64_t)s.size() + 1 > buflen) { r = -(int64_t)(s.size() + 1); return; }
    memcpy(buf, s.c_str(), s.size() + 1);
    r = (int64_t)s.size();
  });
  return r;
}

}  // extern "C"
