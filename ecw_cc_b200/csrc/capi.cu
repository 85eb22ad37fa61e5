// capi.cu — the extern "C" surface declared in include/ecw_b200.h and the NCCL loader; the context's plans run in
// exec.cu.
#include <dlfcn.h>

#include <cmath>
#include <cstring>
#include <sstream>
#include <string>
#include <vector>

#include "exec.h"
#include "kernels.h"

using namespace ecw;

namespace {

int slot_by_name(const char* name) {
  for (int s = 0; s < S_COUNT; ++s)
    if (strcmp(name, slot_name(s)) == 0) return s;
  return -1;
}

int64_t slot_elems(const Sizes& z, int s) {
  const int64_t o = z.nocc, v = z.nvir, n = o + v, po = npair(o), pv = npair(v);
  const int ns = ozaki_digits(z.oz_ns);
  int64_t n0, nsh;                    // this rank's shard of vvvv_p: rows [n0, n0 + nsh) of the packed pair index
  shard_range(pv, z.rank, z.world, &n0, &nsh);
  switch (s) {
    case S_T1: case S_L1: case S_OUT1: return o * v;
    case S_T2: case S_L2: case S_OUT2: case S_OOVV: case S_OOVV_PH: case S_OVOV_PH: return o * o * v * v;
    case S_FSP: case S_FOCK: case S_RDM1: return n * n;
    case S_SCAL: return SC_COUNT;
    case S_OOOO: return o * o * o * o;
    case S_OOOV: return o * o * o * v;
    case S_OVVV: return o * v * v * v;
    case S_OOOO_P: return po * po;
    case S_OOVV_P: return po * pv;
    case S_OVVV_P: return o * v * pv;
    case S_VVVV_P: return nsh * pv;
    case S_VVVV_OZ: return ozaki_plane_elems(nsh, 1, pv, ns);
    case S_VVVV_OZS: return ozaki_stat_elems(nsh, 1);             // [row scales | row sums]
    case S_OVVV_OZ1: return ozaki_plane_elems(o * v, 1, pv, ns);
    case S_OVVV_OZ1S: return ozaki_stat_elems(o * v, 1);
    case S_OVVV_OZ2: return ozaki_plane_elems(pv, o, v, ns);
    case S_OVVV_OZ2S: return ozaki_stat_elems(pv, o);
    default: return -1;
  }
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

// Copies `s` and its terminating NUL into buf: returns the length of s, or minus the buffer size s needs.
int64_t copy_json_out(const std::string& s, char* buf, int64_t buflen) {
  if ((int64_t)s.size() + 1 > buflen) return -(int64_t)(s.size() + 1);
  memcpy(buf, s.c_str(), s.size() + 1);
  return (int64_t)s.size();
}

struct SlotPtr { int slot; const double* p; };

// One call of a cached plan.  `bind` lists exactly the slots the entry point writes: the whole pointer table is part
// of the CUDA-graph key.  result: the plan leaves a scalar in scal[SC_RESULT], copied to *result_out after the call.
int call_plan(ecw_ctx* c, const char* func, int flags, double alpha, std::initializer_list<SlotPtr> bind, bool result,
              double* result_out, void* stream) {
  return guarded_rc(c, [&] {
    require_device();
    for (const SlotPtr& b : bind) c->ptr[b.slot] = const_cast<double*>(b.p);
    if (result) {
      require_slots(c, {S_SCAL});
      c->copy_scal_to = result_out;
    }
    return run_plan(c, get_plan(c, func, flags), alpha, static_cast<cudaStream_t>(stream), true);
  });
}

// The C API's plain GEMM: one product, no split-K.
GemmArgs plain_gemm(int ta, int tb, int64_t M, int64_t N, int64_t K, double alpha, const double* A, int64_t lda,
                    const double* B, int64_t ldb, double beta, double* C, int64_t ldc) {
  GemmArgs g{};
  g.A = A; g.B = B; g.C = C; g.M = M; g.N = N; g.K = K; g.lda = lda; g.ldb = ldb; g.ldc = ldc;
  g.batch = 1; g.splitk = 1; g.kchunk = K; g.ta = ta; g.tb = tb; g.alpha = alpha; g.beta = beta;
  return g;
}

// ecw_tensor -> Tensor in `slot`.  A null descriptor is an absent operand, and so is a null data pointer when
// by_ptr (the ops; the host-only plan dump ignores the pointers).
Tensor from_desc(const ecw_tensor* t, int slot, bool by_ptr = true) {
  Tensor r;
  if (!t || (by_ptr && !t->ptr)) return r;
  if (t->nd < 0 || t->nd > MAXD) throw Fail("ecw_tensor: rank out of range");
  r.slot = slot;
  r.nd = t->nd;
  for (int i = 0; i < t->nd; ++i) { r.dim[i] = t->dim[i]; r.str[i] = t->str[i]; }
  if (r.nd == 0) { r.nd = 1; r.dim[0] = 1; r.str[0] = 1; }
  return r;
}

// The plan of a primitive contraction, configured with the context's GEMM engine; with_override: the engine override
// (ecw_ctx_set_engine_override) takes the INT8 route away.
Plan contract_plan(const ecw_ctx* c, bool with_override) {
  Plan P;
  P.oz_ns = with_override && c->force_dmma ? 0 : c->z.oz_ns;
  P.oz_min_flops = c->z.oz_min_flops;
  P.nocc = c->z.nocc;
  P.nvir = c->z.nvir;
  P.oz_splitk_min_k = c->z.oz_splitk_min_k;
  return P;
}

// Runs the plan of a primitive op, kept as c->op_plan.  Returns -2 with need_ws set when the workspace is too small.
int run_op(ecw_ctx* c, Plan&& P, double alpha_rt, void* stream) {
  c->op_plan = std::move(P);
  if (c->op_plan.workspace_elems() * 8 > c->ws_bytes) {
    c->need_ws = c->op_plan.workspace_elems() * 8;
    c->err = "workspace too small for this op (ecw_op_workspace_needed)";
    return -2;
  }
  return run_plan(c, c->op_plan, alpha_rt, static_cast<cudaStream_t>(stream));
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
    require_slots(c, {S_SCAL});
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (!c->call_has_oz) {          // the last call launched no INT8 product: nothing to read, no synchronisation
      *bound_out = 0.0;
      return;
    }
    ck(cudaMemcpyAsync(bound_out, c->ptr[S_SCAL] + SC_INT8_BOUND, sizeof(double), cudaMemcpyDeviceToHost, st), "read int8 bound");
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
    require_slots(c, {S_VVVV_OZ, S_VVVV_OZS});
    const int64_t pv = npair(c->z.nvir);
    int64_t n0, nsh;
    shard_range(pv, c->z.rank, c->z.world, &n0, &nsh);
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
    require_slots(c, {S_OVVV_P, S_OVVV_OZ1, S_OVVV_OZ1S, S_OVVV_OZ2, S_OVVV_OZ2S});
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
    require_slots(c, {S_OOOO, S_OOOV, S_OOVV, S_OVVV, S_OOVV_PH, S_OVOV_PH, S_OOOO_P, S_OOVV_P, S_OVVV_P, S_VVVV_P});
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
      require_slots(c, {t.slot});
      int64_t r0 = 0, nr = t.rows;
      if (t.slot == S_VVVV_P) shard_range(pv, c->z.rank, c->z.world, &r0, &nr);   // this rank's rows
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
  return call_plan(c, "tupdate", flags, alpha,
                   {{S_T1, t1}, {S_T2, t2}, {S_FSP, fsp}, {S_FOCK, fock}, {S_OUT1, t1new}, {S_OUT2, t2new}}, false,
                   nullptr, stream);
}

int ecw_ccsd_lupdate(ecw_ctx* c, const double* t1, const double* t2, const double* l1, const double* l2,
                     const double* fsp, const double* fock, int flags, double alpha, double* l1new, double* l2new,
                     void* stream) {
  return call_plan(c, "lupdate", flags, alpha,
                   {{S_T1, t1}, {S_T2, t2}, {S_L1, l1}, {S_L2, l2}, {S_FSP, fsp}, {S_FOCK, fock}, {S_OUT1, l1new},
                    {S_OUT2, l2new}},
                   false, nullptr, stream);
}

int ecw_ccsd_gamma(ecw_ctx* c, const double* t1, const double* t2, const double* l1, const double* l2, double* rdm1,
                   void* stream) {
  return call_plan(c, "gamma", 0, 0.0, {{S_T1, t1}, {S_T2, t2}, {S_L1, l1}, {S_L2, l2}, {S_RDM1, rdm1}}, false,
                   nullptr, stream);
}

int ecw_ccsd_energy(ecw_ctx* c, const double* t1, const double* t2, const double* fsp, double* e_out, void* stream) {
  return call_plan(c, "energy", 0, 0.0, {{S_T1, t1}, {S_T2, t2}, {S_FSP, fsp}}, true, e_out, stream);
}

// ---- ECW-CCS intermediates (csrc/ccs_plan.cpp): one cached plan each
int ecw_ccs_t1inter(ecw_ctx* c, const double* ts, const double* fsp, double* F, void* stream) {
  return call_plan(c, "ccs_t1inter", 0, 0.0, {{S_T1, ts}, {S_FSP, fsp}, {S_RDM1, F}}, false, nullptr, stream);
}

int ecw_ccs_l1inter(ecw_ctx* c, const double* ts, const double* fsp, int e_term, double* F, double* W, double* e_out,
                    void* stream) {
  return call_plan(c, "ccs_l1inter", e_term ? 1 : 0, 0.0, {{S_T1, ts}, {S_FSP, fsp}, {S_RDM1, F}, {S_OUT2, W}},
                   e_term != 0, e_out, stream);
}

int ecw_ccs_r1inter(ecw_ctx* c, const double* ts, const double* fsp, const double* vm, double* F, double* W, double* X,
                    double* e_out, void* stream) {
  return call_plan(c, "ccs_r1inter", vm ? 1 : 0, 0.0,
                   {{S_T1, ts}, {S_FSP, fsp}, {S_FOCK, vm}, {S_RDM1, F}, {S_OUT2, W}, {S_OUT1, X}}, true, e_out, stream);
}

int ecw_ccs_esl1inter(ecw_ctx* c, const double* ts, const double* fsp, const double* vm, double* F, double* W, double* X,
                      double* e_out, void* stream) {
  return call_plan(c, "ccs_esl1inter", vm ? 1 : 0, 0.0,
                   {{S_T1, ts}, {S_FSP, fsp}, {S_FOCK, vm}, {S_RDM1, F}, {S_OUT2, W}, {S_OUT1, X}}, true, e_out, stream);
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
  guarded(c, [&] { r = copy_json_out(get_plan(c, func, flags).dump_json(), buf, buflen); });
  return r;
}

int64_t ecw_plan_dump_contract(ecw_ctx* c, double alpha, const ecw_tensor* A, const char* sa, const ecw_tensor* B,
                               const char* sb, double beta, const ecw_tensor* C, const char* sc, char* buf,
                               int64_t buflen) {
  int64_t r = -1;
  guarded(c, [&] {
    // host only: the lowering ecw_op_contract would launch (operands named a0, a1, b0; ptr fields are ignored), with
    // the context's engine: the engine override (ecw_ctx_set_engine_override) is not applied
    Plan P = contract_plan(c, false);
    P.contract(alpha, from_desc(A, S_A0, false), sa, from_desc(B, S_A1, false), sb, beta, from_desc(C, S_B0, false), sc,
               "op");
    r = copy_json_out(P.dump_json(), buf, buflen);
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
    ck(launch_gemm(plain_gemm(ta, tb, M, N, K, alpha, A, lda, B, ldb, beta, C, ldc), static_cast<cudaStream_t>(stream),
                   cfg),
       "dgemm");
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
int64_t ecw_op_workspace_needed(ecw_ctx* c) { return c ? c->need_ws : -1; }

int ecw_op_contract(ecw_ctx* c, double alpha, const ecw_tensor* A, const char* sa, const ecw_tensor* B, const char* sb,
                    double beta, const ecw_tensor* C, const char* sc, void* stream) {
  return guarded_rc(c, [&] {
    require_device();
    Plan P = contract_plan(c, true);
    c->ptr[S_A0] = (double*)A->ptr; c->ptr[S_A1] = (double*)B->ptr; c->ptr[S_B0] = (double*)C->ptr;
    P.contract(alpha, from_desc(A, S_A0), sa, from_desc(B, S_A1), sb, beta, from_desc(C, S_B0), sc, "op");
    return run_op(c, std::move(P), 0.0, stream);
  });
}

int ecw_op_axpby(ecw_ctx* c, double alpha, const ecw_tensor* A, const char* sa, double beta, const ecw_tensor* C,
                 const char* sc, void* stream) {
  return guarded_rc(c, [&] {
    require_device();
    Plan P;
    c->ptr[S_A0] = (double*)A->ptr; c->ptr[S_B0] = (double*)C->ptr;
    P.permute(alpha, from_desc(A, S_A0), sa, beta, from_desc(C, S_B0), sc, "op");
    return run_op(c, std::move(P), 0.0, stream);
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
    return run_op(c, std::move(P), 0.0, stream);
  });
}

int ecw_op_unpack(ecw_ctx* c, double alpha, const ecw_tensor* A2, int flags, double beta, const ecw_tensor* C4,
                  void* stream) {
  return guarded_rc(c, [&] {
    require_device();
    Plan P;
    c->ptr[S_A0] = (double*)A2->ptr; c->ptr[S_B0] = (double*)C4->ptr;
    P.unpack(alpha, from_desc(A2, S_A0), flags, beta, from_desc(C4, S_B0));
    return run_op(c, std::move(P), 0.0, stream);
  });
}

int ecw_op_diag_shift(ecw_ctx* c, const ecw_tensor* Cm, double alpha, const ecw_tensor* fock, int64_t offset,
                      void* stream) {
  return guarded_rc(c, [&] {
    require_device();
    Plan P;
    c->ptr[S_B0] = (double*)Cm->ptr; c->ptr[S_FOCK] = (double*)fock->ptr;
    P.diag_add(from_desc(Cm, S_B0), alpha, from_desc(fock, S_FOCK), offset);
    return run_op(c, std::move(P), 0.0, stream);
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
    return run_op(c, std::move(P), alpha, stream);
  });
}

int ecw_op_dot(ecw_ctx* c, double alpha, const ecw_tensor* A, const ecw_tensor* B, double beta, double* out_dev,
               void* stream) {
  return guarded_rc(c, [&] {
    require_device();
    require_slots(c, {S_SCAL});
    Plan P;
    c->ptr[S_A0] = (double*)A->ptr; c->ptr[S_A1] = (double*)B->ptr;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    double* dot = c->ptr[S_SCAL] + SC_DOT;
    if (beta != 0.0) ck(cudaMemcpyAsync(dot, out_dev, sizeof(double), cudaMemcpyDeviceToDevice, st), "dot in");
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
    P.dot(alpha, ad, bd, beta, SC_DOT);
    int rc = run_op(c, std::move(P), 0.0, stream);
    if (rc == 0) ck(cudaMemcpyAsync(out_dev, dot, sizeof(double), cudaMemcpyDeviceToDevice, st), "dot out");
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
    ck(launch_gemm(plain_gemm(ta, tb, M, N, K, 1.0, A, lda, B, ldb, beta, C, ldc), st), "vexp_sf gemm");
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
    std::ostringstream o;
    o << "[";
    for (size_t i = 0; i < c->last_plan->ops.size(); ++i) {
      float ms = 0.f;
      cudaEventElapsedTime(&ms, c->ev[i], c->ev[i + 1]);
      const Op& op = c->last_plan->ops[i];
      if (i) o << ",";
      o << "\n{\"kind\":\"" << op_kind_name(op.kind) << "\",\"ms\":" << ms << ",\"M\":" << op.M << ",\"N\":" << op.N
        << ",\"K\":" << op.K << ",\"batch\":" << op.batch << ",\"splitk\":" << op.splitk << ",\"elems\":"
        << (op.c.valid() ? op.c.size() : 0) << ",\"note\":\"" << op.note << "\"}";
    }
    o << "\n]";
    r = copy_json_out(o.str(), buf, buflen);
  });
  return r;
}

}  // extern "C"
