// exec.cu — the plan cache and the stream executor of the C API: a plan's ops become kernel launches on the caller's
// stream, optionally captured once into a CUDA graph and replayed.
#include "exec.h"

#include "kernels.h"

namespace ecw {

namespace {

constexpr int kNcclDouble = 8;     // ncclFloat64

double* resolve(ecw_ctx* c, const Tensor& t, bool required = true) {
  if (!t.valid()) {
    if (required) throw Fail("plan references an unset operand");
    return nullptr;
  }
  require_slots(c, {t.slot});
  return c->ptr[t.slot] + t.off;
}

void reset_int8_bound(ecw_ctx* c, cudaStream_t st) {
  if (c->ptr[S_SCAL])
    ck(cudaMemsetAsync(c->ptr[S_SCAL] + SC_INT8_BOUND, 0, sizeof(double), st), "reset int8 bound");
}

}  // namespace

void require_slots(const ecw_ctx* c, std::initializer_list<int> slots) {
  for (int s : slots)
    if (!c->ptr[s]) throw Fail(std::string("slot '") + slot_name(s) + "' is not bound");
}

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
        ck(launch_asym4(resolve(c, op.b, false), op.alpha, resolve(c, op.a), resolve(c, op.c), op.beta,
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
        require_slots(c, {S_SCAL});
        ck(launch_dot(resolve(c, op.a), resolve(c, op.b), op.a.size(), resolve(c, op.c), (int)op.i1,
                      c->ptr[S_SCAL] + op.i0, op.alpha, op.beta, st), "dot");
        break;
      case OP_SCALE_DEV:
        require_slots(c, {S_SCAL});
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
      case OP_EWISE: {
        // out = alpha * a * b + beta * out (strided; a and/or b may be absent)
        Ew2Args e{};
        e.a = resolve(c, op.a, false);
        e.b = resolve(c, op.b, false);
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
        break;
      }
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
                                c->ptr[S_SCAL] + SC_INT8_BOUND, st), "ozaki_bound");
        break;
      }
      default:
        throw Fail("unknown op kind");
    }
    ++c->pc;
    if (c->profile_run) ck(cudaEventRecord(c->ev[c->pc], st), "cudaEventRecord");
  }
  if (c->copy_scal_to) {
    ck(cudaMemcpyAsync(c->copy_scal_to, c->ptr[S_SCAL] + SC_RESULT, sizeof(double), cudaMemcpyDeviceToDevice, st),
       "copy scalar");
    c->copy_scal_to = nullptr;
  }
  c->run_plan_ptr = nullptr;
  return 0;
}

int run_plan(ecw_ctx* c, const Plan& P, double alpha_rt, cudaStream_t st, bool cached_plan) {
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
        reset_int8_bound(c, c->cap_stream);
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
  reset_int8_bound(c, st);
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

}  // namespace ecw
