// plan.cpp — plan container, workspace arena and the binary-contraction
// lowering (TTGT with batch / split-K / layout search).  Host-only C++.
#include "plan.h"
#include "kernels.h"

#include <algorithm>
#include <cmath>
#include <cstring>
#include <map>
#include <sstream>

namespace ecw {

int64_t npair(int64_t n) { return n * (n - 1) / 2; }

const char* slot_name(int s) {
  static const char* names[] = {
      "ws", "t1", "t2", "l1", "l2", "fsp", "fock", "out1", "out2", "rdm1", "scal",
      "oooo", "ooov", "oovv", "oovv_ph", "ovov_ph", "ovvv", "oooo_p", "oovv_p", "ovvv_p", "vvvv_p",
      "vvvv_oz", "vvvv_ozs", "ovvv_oz1", "ovvv_oz1s", "ovvv_oz2", "ovvv_oz2s",
      "a0", "a1", "a2", "a3", "a4", "a5", "a6", "a7", "a8", "a9",
      "b0", "b1", "b2", "b3", "b4", "b5", "b6", "b7"};
  if (s < 0 || s >= S_COUNT) return "?";
  return names[s];
}

Tensor make_tensor(int slot, int64_t off, std::initializer_list<int64_t> dims) {
  Tensor t;
  t.slot = slot;
  t.off = off;
  t.nd = (int)dims.size();
  if (t.nd > MAXD) throw PlanError("tensor rank > MAXD");
  int i = 0;
  for (auto d : dims) t.dim[i++] = d;
  int64_t s = 1;
  for (i = t.nd - 1; i >= 0; --i) { t.str[i] = s; s *= t.dim[i]; }
  return t;
}

static bool is_contig(const Tensor& t) {
  int64_t s = 1;
  for (int i = t.nd - 1; i >= 0; --i) {
    if (t.dim[i] != 1 && t.str[i] != s) return false;
    s *= t.dim[i];
  }
  return true;
}

Tensor reshape(const Tensor& t, std::initializer_list<int64_t> dims) {
  if (!is_contig(t)) throw PlanError("reshape of non-contiguous view");
  Tensor r = make_tensor(t.slot, t.off, dims);
  if (r.size() != t.size()) throw PlanError("reshape size mismatch");
  return r;
}

Tensor block2(const Tensor& m, int64_t r0, int64_t nr, int64_t c0, int64_t nc) {
  if (m.nd != 2) throw PlanError("block2 needs a matrix");
  Tensor r = m;
  r.off = m.off + r0 * m.str[0] + c0 * m.str[1];
  r.dim[0] = nr;
  r.dim[1] = nc;
  return r;
}

Tensor transpose2(const Tensor& m) {
  if (m.nd != 2) throw PlanError("transpose2 needs a matrix");
  Tensor r = m;
  std::swap(r.dim[0], r.dim[1]);
  std::swap(r.str[0], r.str[1]);
  return r;
}

Tensor slice0(const Tensor& t, int64_t i0, int64_t n) {
  Tensor r = t;
  r.off = t.off + i0 * t.str[0];
  r.dim[0] = n;
  return r;
}

Tensor slice_dim(const Tensor& t, int d, int64_t i0, int64_t n) {
  Tensor r = t;
  r.off = t.off + i0 * t.str[d];
  r.dim[d] = n;
  return r;
}

// ---------------------------------------------------------------- arena
int64_t Arena::alloc(int64_t n) {
  n = (n + 31) / 32 * 32;  // 256-byte granularity
  if (n == 0) n = 32;
  for (size_t i = 0; i < blks.size(); ++i) {
    if (!blks[i].used && blks[i].size >= n) {
      if (blks[i].size > n) {
        Blk rest{blks[i].off + n, blks[i].size - n, false};
        blks[i].size = n;
        blks.insert(blks.begin() + i + 1, rest);
      }
      blks[i].used = true;
      return blks[i].off;
    }
  }
  int64_t end = blks.empty() ? 0 : blks.back().off + blks.back().size;
  if (!blks.empty() && !blks.back().used) {  // grow the trailing free block
    blks.back().size = n;
    blks.back().used = true;
    peak = std::max(peak, blks.back().off + n);
    return blks.back().off;
  }
  blks.push_back(Blk{end, n, true});
  peak = std::max(peak, end + n);
  return end;
}

void Arena::release(int64_t off) {
  for (size_t i = 0; i < blks.size(); ++i) {
    if (blks[i].off == off && blks[i].used) {
      blks[i].used = false;
      if (i + 1 < blks.size() && !blks[i + 1].used) {
        blks[i].size += blks[i + 1].size;
        blks.erase(blks.begin() + i + 1);
      }
      if (i > 0 && !blks[i - 1].used) {
        blks[i - 1].size += blks[i].size;
        blks.erase(blks.begin() + i);
      }
      return;
    }
  }
  throw PlanError("arena: release of unknown block");
}

Tensor Plan::tmpv(const std::vector<int64_t>& dims) {
  Tensor t;
  t.slot = S_WS;
  t.nd = (int)dims.size();
  if (t.nd > MAXD) throw PlanError("tensor rank > MAXD");
  int64_t s = 1;
  for (int i = t.nd - 1; i >= 0; --i) { t.dim[i] = dims[i]; t.str[i] = s; s *= dims[i]; }
  t.off = arena.alloc(s);
  return t;
}

Tensor Plan::tmp(std::initializer_list<int64_t> dims) { return tmpv(std::vector<int64_t>(dims)); }

Tensor Plan::tmp_lead_padded(std::initializer_list<int64_t> dims) {
  std::vector<int64_t> d(dims);
  const int64_t lead = d[0];
  d[0] = lead_chunk(lead) * world;
  Tensor t = tmpv(d);
  t.dim[0] = lead;
  return t;
}

void Plan::allgather(const Tensor& chunk, int64_t count, const Tensor& full, const char* note) {
  Op op;
  op.kind = OP_ALLGATHER;
  op.a = chunk;
  op.c = full;
  op.i0 = count;
  op.i1 = world;
  op.i2 = rank;
  op.note = note;
  ops.push_back(op);
}

void Plan::alltoall(const Tensor& send, int64_t count, const Tensor& recv, const char* note) {
  if (world == 1) {
    Tensor a = make_tensor(send.slot, send.off, {count}), c = make_tensor(recv.slot, recv.off, {count});
    permute(1.0, a, "p", 0.0, c, "p", note);
    return;
  }
  Op op;
  op.kind = OP_ALLTOALL;
  op.a = send;
  op.c = recv;
  op.i0 = count;
  op.i1 = world;
  op.i2 = rank;
  op.note = note;
  ops.push_back(op);
}

void Plan::sum_ranks_add(const Tensor& part, const Tensor& C, const char* note) {
  const int64_t n = part.size();
  if (world == 1) {
    axpby(1.0, part, 1.0, C, note);
    return;
  }
  if (part.slot != S_WS) throw PlanError("sum_ranks_add: the partial result must live in the workspace");
  Tensor G = tmp({(int64_t)world, n});
  allgather(part, n, G, note);
  Op r;
  r.kind = OP_REDUCE;
  r.a = G;
  r.i0 = world;
  // C as an M x N matrix: any contiguous C is [n, 1]; a strided 2-D C keeps its own strides
  if (C.nd == 2 && C.size() == n) { r.M = C.dim[0]; r.N = C.dim[1]; r.i1 = C.str[0]; r.i2 = C.str[1]; }
  else { r.M = n; r.N = 1; r.i1 = 1; r.i2 = 0; }
  r.c = C;
  r.alpha = 1.0; r.beta = 1.0;
  r.note = std::string(note) + " [sum over ranks]";
  ops.push_back(r);
  release(G);
}

void Plan::contract_split(double alpha, const Tensor& A, const char* sa, const Tensor& B, const char* sb,
                          const Tensor& C, const char* sc, char lab, const char* note) {
  if (world == 1) {
    contract(alpha, A, sa, B, sb, 1.0, C, sc, note);
    return;
  }
  const char* qa = strchr(sa, lab);
  const char* qb = strchr(sb, lab);
  if (!qa || !qb || strchr(sc, lab)) throw PlanError(std::string("contract_split: label must be contracted in ") + sa + "," + sb);
  const int pa = (int)(qa - sa), pb = (int)(qb - sb);
  const int64_t L = A.dim[pa], chunk = lead_chunk(L);
  const int64_t l0 = std::min<int64_t>(L, rank * chunk), nl = std::min<int64_t>(L, l0 + chunk) - l0;
  const int64_t n = C.size();
  std::vector<int64_t> cd(C.dim, C.dim + C.nd);
  Tensor part = tmpv(cd);
  Tensor G = tmp({(int64_t)world, n});
  if (nl > 0) contract(alpha, slice_dim(A, pa, l0, nl), sa, slice_dim(B, pb, l0, nl), sb, 0.0, part, sc, note);
  else fill(part, 0.0);
  allgather(part, n, G, note);
  Op r;
  r.kind = OP_REDUCE;
  r.a = G;
  r.i0 = world;
  r.M = n; r.N = 1;
  r.c = C;
  r.i1 = 1; r.i2 = 0;
  r.alpha = 1.0; r.beta = 1.0;
  r.note = std::string(note) + " [sum over ranks]";
  ops.push_back(r);
  release(G);
  release(part);
}

void Plan::contract_lead_dist(double alpha, const Tensor& A, const char* sa, const Tensor& B, const char* sb,
                              const Tensor& C, const char* sc, const char* note) {
  if (world == 1) {
    contract(alpha, A, sa, B, sb, 0.0, C, sc, note);
    return;
  }
  if (sa[0] != sc[0]) throw PlanError(std::string("contract_lead_dist: leading labels differ in ") + sa + "->" + sc);
  const int64_t L = C.dim[0], chunk = lead_chunk(L);
  const int64_t l0 = std::min<int64_t>(L, rank * chunk), nl = std::min<int64_t>(L, l0 + chunk) - l0;
  if (nl > 0) contract(alpha, slice0(A, l0, nl), sa, B, sb, 0.0, slice0(C, l0, nl), sc, note);
  Tensor mine = C;
  mine.off = C.off + rank * chunk * C.str[0];
  mine.dim[0] = chunk;
  Tensor full = C;
  full.dim[0] = chunk * world;
  allgather(mine, chunk * C.str[0], full, note);
}

void Plan::release(const Tensor& t) {
  if (t.slot != S_WS) throw PlanError("release of non-workspace tensor");
  if (!cut_cache.empty()) {
    // the planes cut from this buffer go with it (the arena block is the unit: its whole extent)
    int64_t lo = t.off, hi = t.off;
    for (const auto& b : arena.blks)
      if (b.off == t.off && b.used) { hi = b.off + b.size - 1; break; }
    drop_cuts_of(S_WS, lo, hi);
  }
  arena.release(t.off);
}

// ---------------------------------------------------------------- simple ops
void Plan::permute(double alpha, const Tensor& A, const char* sa, double beta, const Tensor& C,
                   const char* sc, const char* note) {
  int n = (int)strlen(sc);
  if ((int)strlen(sa) != n || A.nd != n || C.nd != n) throw PlanError(std::string("permute rank mismatch: ") + sa + "->" + sc);
  Op op;
  op.kind = OP_PERMUTE;
  op.alpha = alpha;
  op.beta = beta;
  op.c = C;
  op.a = A;
  for (int p = 0; p < n; ++p) {
    const char* q = strchr(sa, sc[p]);
    if (!q) throw PlanError(std::string("permute label mismatch: ") + sa + "->" + sc);
    int qi = (int)(q - sa);
    if (A.dim[qi] != C.dim[p]) throw PlanError(std::string("permute dim mismatch: ") + sa + "->" + sc);
    op.a.dim[p] = A.dim[qi];
    op.a.str[p] = A.str[qi];
  }
  op.note = std::string(note) + " [" + sa + "->" + sc + "]";
  perm_bytes += 8.0 * (double)C.size() * (beta != 0.0 ? 3.0 : 2.0);
  ops.push_back(op);
}

void Plan::axpby(double alpha, const Tensor& A, double beta, const Tensor& C, const char* note) {
  static const char* lab = "pqrstu";
  if (A.nd != C.nd) throw PlanError("axpby rank mismatch");
  std::string s(lab, lab + A.nd);
  permute(alpha, A, s.c_str(), beta, C, s.c_str(), note);
}

void Plan::fill(const Tensor& C, double value) {
  Op op;
  op.kind = OP_FILL;
  op.c = C;
  op.alpha = value;
  ops.push_back(op);
}

void Plan::tau(const Tensor& t2, const Tensor& t1, double c1, double c2, const Tensor& out) {
  Op op;
  op.kind = OP_TAU;
  op.a = t2;
  op.b = t1;
  op.c = out;
  op.alpha = c1;
  op.beta = c2;
  ops.push_back(op);
}

void Plan::tau_rows(const Tensor& t2_rows, const Tensor& t1, int64_t i0, double c1, double c2, const Tensor& out_rows) {
  Op op;
  op.kind = OP_TAU;
  op.a = t2_rows;
  op.b = t1;
  op.c = out_rows;
  op.alpha = c1;
  op.beta = c2;
  op.i0 = i0;
  op.i1 = out_rows.dim[0];
  op.i2 = 1;               // row-range form
  ops.push_back(op);
}

void Plan::asym4(double c0, const Tensor* base, const Tensor& z, double beta, const Tensor& out, const char* note) {
  if (z.nd != 4 || out.nd != 4) throw PlanError("asym4: needs [o,o,v,v] tensors");
  Op op;
  op.kind = OP_ASYM4;
  op.a = z;
  if (base) op.b = *base;
  op.c = out;
  op.alpha = base ? c0 : 0.0;
  op.beta = beta;
  op.note = note;
  perm_bytes += 8.0 * (double)out.size() * (2.0 + (base ? 1.0 : 0.0) + (beta != 0.0 ? 1.0 : 0.0));
  ops.push_back(op);
}

void Plan::pack(double alpha, const Tensor& a4, int flags, double beta, const Tensor& c2) {
  if (a4.nd != 4 || c2.nd != 2) throw PlanError("pack: need 4-index source and matrix destination");
  int64_t rows = (flags & 1) ? npair(a4.dim[0]) : a4.dim[0] * a4.dim[1];
  int64_t cols = (flags & 2) ? npair(a4.dim[2]) : a4.dim[2] * a4.dim[3];
  if ((flags & 9) && a4.dim[0] != a4.dim[1]) throw PlanError("pack: first pair dims differ");
  if ((flags & 6) && a4.dim[2] != a4.dim[3]) throw PlanError("pack: second pair dims differ");
  if (rows != c2.dim[0] || cols != c2.dim[1]) throw PlanError("pack: destination shape mismatch");
  Op op;
  op.kind = OP_PACK;
  op.a = a4;
  op.c = c2;
  op.alpha = alpha;
  op.beta = beta;
  op.i0 = flags;
  ops.push_back(op);
}

void Plan::unpack(double alpha, const Tensor& a2, int flags, double beta, const Tensor& c4) {
  if (c4.nd != 4 || a2.nd != 2) throw PlanError("unpack: need matrix source and 4-index destination");
  int64_t rows = (flags & 1) ? npair(c4.dim[0]) : c4.dim[0] * c4.dim[1];
  int64_t cols = (flags & 2) ? npair(c4.dim[2]) : c4.dim[2] * c4.dim[3];
  if (rows != a2.dim[0] || cols != a2.dim[1]) throw PlanError("unpack: source shape mismatch");
  Op op;
  op.kind = OP_UNPACK;
  op.a = a2;
  op.c = c4;
  op.alpha = alpha;
  op.beta = beta;
  op.i0 = flags;
  ops.push_back(op);
}

void Plan::finish(const Tensor& resid, const Tensor& amp, const Tensor& fock, int nocc, int rank,
                  int has_alpha, int equation, double alpha, const Tensor& out, double shift, int sub_singles) {
  Op op;
  op.kind = OP_FINISH;
  op.a = resid;
  op.b = amp;
  op.d = fock;
  op.c = out;
  op.i0 = nocc;
  op.i1 = rank;
  op.i2 = has_alpha;
  op.i3 = equation;
  op.alpha = alpha;
  op.d0 = shift;
  op.d1 = sub_singles;
  ops.push_back(op);
}

void Plan::dot(double alpha, const Tensor& A, const Tensor& B, double beta, int k) {
  if (A.nd != B.nd) throw PlanError("dot rank mismatch");
  for (int i = 0; i < A.nd; ++i) if (A.dim[i] != B.dim[i]) throw PlanError("dot shape mismatch");
  Op op;
  op.kind = OP_DOT;
  op.a = A;
  op.b = B;
  op.alpha = alpha;
  op.beta = beta;
  op.i0 = k;
  // per-block partial sums (deterministic two-stage reduction)
  op.i1 = 1024;
  op.c = tmp({op.i1});
  ops.push_back(op);
  release(op.c);
}

void Plan::scale_dev(const Tensor& C, double d0, double d1, int k) {
  Op op;
  op.kind = OP_SCALE_DEV;
  op.c = C;
  op.d0 = d0;
  op.d1 = d1;
  op.i0 = k;
  ops.push_back(op);
}

void Plan::diag_add(const Tensor& Cmat, double alpha, const Tensor& fock, int64_t foff) {
  Op op;
  op.kind = OP_DIAG_ADD;
  op.c = Cmat;
  op.d = fock;
  op.alpha = alpha;
  op.i0 = foff;
  ops.push_back(op);
}

void Plan::rdm1(const Tensor& doo, const Tensor& dvoT, const Tensor& l1, const Tensor& dvv, const Tensor& out) {
  Op op;
  op.kind = OP_RDM1;
  op.a = doo;
  op.b = dvoT;
  op.d = l1;
  op.e = dvv;
  op.c = out;
  ops.push_back(op);
}

void Plan::ewise(int sub, const Tensor& a, const Tensor& b, const Tensor& c, double alpha, double beta,
                 int64_t i1, int64_t i2) {
  Op op;
  op.kind = OP_EWISE;
  op.a = a;
  op.b = b;
  op.c = c;
  op.alpha = alpha;
  op.beta = beta;
  op.i0 = sub;
  op.i1 = i1;
  op.i2 = i2;
  ops.push_back(op);
}

// ---------------------------------------------------------------- contraction engine
static double oz_time(int ns, int sm_count, int64_t M, int64_t N, int64_t K, int64_t crs, int64_t ccs, double beta,
                      bool* swap_out, int64_t splits = 1);
static int64_t oz_pick_splits(int ns, int sm_count, int64_t M, int64_t N, int64_t K, int64_t min_k);

namespace {

struct Group {
  bool ok = true;
  int64_t dim = 1;
  int64_t str = 0;   // stride of the merged index (0 for an empty group)
};

// Merge the labels `g` (ordered) of tensor T (labels s) into one index.
Group merge(const Tensor& T, const char* s, const std::string& g) {
  Group r;
  int64_t next_str = -1;  // stride the next (more significant) label must have
  for (int k = (int)g.size() - 1; k >= 0; --k) {
    const char* q = strchr(s, g[k]);
    if (!q) { r.ok = false; return r; }
    int p = (int)(q - s);
    if (T.dim[p] == 1) continue;
    if (next_str < 0) {
      r.str = T.str[p];
      r.dim = T.dim[p];
      next_str = T.str[p] * T.dim[p];
    } else {
      if (T.str[p] != next_str) { r.ok = false; return r; }
      r.dim *= T.dim[p];
      next_str = T.str[p] * T.dim[p];
    }
  }
  return r;
}

struct MatView {
  bool rm = false, cm = false;   // row-major (cols contiguous) / col-major (rows contiguous) possible
  int64_t ld_rm = 0, ld_cm = 0;
  int64_t rows = 1, cols = 1;
  bool any = false;              // both groups mergeable (arbitrary strides)
  int64_t sr = 0, scol = 0;
};

MatView mat_view(const Tensor& T, const char* s, const std::string& rows, const std::string& cols) {
  MatView m;
  Group r = merge(T, s, rows), c = merge(T, s, cols);
  if (!r.ok || !c.ok) return m;
  m.any = true;
  m.rows = r.dim;
  m.cols = c.dim;
  m.sr = r.str;
  m.scol = c.str;
  if (c.dim == 1 || c.str == 1) {
    m.rm = true;
    m.ld_rm = (r.dim == 1) ? std::max<int64_t>(c.dim, 1) : r.str;
    if (m.ld_rm < c.dim) m.rm = false;
  }
  if (r.dim == 1 || r.str == 1) {
    m.cm = true;
    m.ld_cm = (c.dim == 1) ? std::max<int64_t>(r.dim, 1) : c.str;
    if (m.ld_cm < r.dim) m.cm = false;
  }
  return m;
}

std::string ordered(const std::string& set, const char* order) {
  std::string r;
  for (const char* p = order; *p; ++p)
    if (set.find(*p) != std::string::npos) r.push_back(*p);
  return r;
}

std::string minus(const std::string& a, const std::string& b) {
  std::string r;
  for (char c : a) if (b.find(c) == std::string::npos) r.push_back(c);
  return r;
}

int64_t dims_of(const std::string& g, const std::map<char, int64_t>& dm) {
  int64_t n = 1;
  for (char c : g) n *= dm.at(c);
  return n;
}

struct Choice {
  double cost = 1e300;
  std::string bt, om, on, ok;
  int bcls = 0;  // 0 none, 1 I, 2 J, 3 K
  bool a_dir = false, b_dir = false, c_dir = false, c_swap = false;
  int ta = 0, tb = 0;
  int64_t lda = 0, ldb = 0, ldc = 0, sA = 0, sB = 0, sC = 0;
  int64_t c_sr = 0, c_sc = 0;   // strided-C target for the reduce path
};

}  // namespace

void Plan::contract(double alpha, const Tensor& A, const char* sa, const Tensor& B, const char* sb,
                    double beta, const Tensor& C, const char* sc, const char* note) {
  std::string tag = std::string(sa) + "," + sb + "->" + sc;
  if ((int)strlen(sa) != A.nd || (int)strlen(sb) != B.nd || (int)strlen(sc) != C.nd)
    throw PlanError("contract rank mismatch: " + tag);
  std::map<char, int64_t> dm;
  auto reg = [&](const Tensor& T, const char* s) {
    for (int i = 0; i < T.nd; ++i) {
      auto it = dm.find(s[i]);
      if (it == dm.end()) dm[s[i]] = T.dim[i];
      else if (it->second != T.dim[i]) throw PlanError("contract dim mismatch for '" + std::string(1, s[i]) + "' in " + tag);
    }
  };
  reg(A, sa); reg(B, sb); reg(C, sc);
  std::string I, J, K;
  for (auto& kv : dm) {
    bool ia = strchr(sa, kv.first), ib = strchr(sb, kv.first), ic = strchr(sc, kv.first);
    if (ia && ic && !ib) I.push_back(kv.first);
    else if (ib && ic && !ia) J.push_back(kv.first);
    else if (ia && ib && !ic) K.push_back(kv.first);
    else throw PlanError("contract: unsupported label pattern in " + tag);
  }
  const int64_t szA = A.size(), szB = B.size(), szC = C.size();

  // candidate batch sets
  std::vector<std::string> cands{""};
  for (auto& kv : dm) cands.push_back(std::string(1, kv.first));
  for (int p = 0; p + 1 < C.nd; ++p) {
    char x = sc[p], y = sc[p + 1];
    bool bi = I.find(x) != std::string::npos && I.find(y) != std::string::npos;
    bool bj = J.find(x) != std::string::npos && J.find(y) != std::string::npos;
    if (bi || bj) cands.push_back(std::string{x, y});
  }

  Choice best, best0;          // best0: best lowering without a batch index (the only form the INT8 route takes)
  for (auto& bt : cands) {
    int bcls = 0;
    if (!bt.empty()) bcls = I.find(bt[0]) != std::string::npos ? 1 : (J.find(bt[0]) != std::string::npos ? 2 : 3);
    int64_t nb = dims_of(bt, dm);
    if (!bt.empty() && nb == 1) continue;
    // batch strides
    Group gA, gB, gC;
    if (bcls == 1 || bcls == 3) { gA = merge(A, sa, bt); if (!gA.ok) continue; }
    if (bcls == 2 || bcls == 3) { gB = merge(B, sb, bt); if (!gB.ok) continue; }
    if (bcls == 1 || bcls == 2) { gC = merge(C, sc, bt); if (!gC.ok) continue; }
    std::string Ir = minus(I, bt), Jr = minus(J, bt), Kr = minus(K, bt);
    int64_t Md = dims_of(Ir, dm), Nd = dims_of(Jr, dm);
    for (int m = 0; m < 2; ++m)
      for (int n = 0; n < 2; ++n)
        for (int k = 0; k < 2; ++k) {
          Choice ch;
          ch.bt = bt;
          ch.bcls = bcls;
          ch.om = ordered(Ir, m ? sc : sa);
          ch.on = ordered(Jr, n ? sc : sb);
          ch.ok = ordered(Kr, k ? sb : sa);
          MatView va = mat_view(A, sa, ch.om, ch.ok);
          MatView vb = mat_view(B, sb, ch.ok, ch.on);
          MatView vc = mat_view(C, sc, ch.om, ch.on);
          double cost = 0.0;
          if (va.rm) { ch.a_dir = true; ch.ta = 0; ch.lda = va.ld_rm; }
          else if (va.cm) { ch.a_dir = true; ch.ta = 1; ch.lda = va.ld_cm; }
          else cost += 2.0 * szA;
          if (vb.rm) { ch.b_dir = true; ch.tb = 0; ch.ldb = vb.ld_rm; }
          else if (vb.cm) { ch.b_dir = true; ch.tb = 1; ch.ldb = vb.ld_cm; }
          else cost += 2.0 * szB;
          if (bcls == 3) {
            // reduce path: any strided C target works
            if (vc.any) { ch.c_dir = true; ch.c_sr = vc.sr; ch.c_sc = vc.scol; }
            else cost += 3.0 * szC;
            cost += 2.0 * (double)nb * Md * Nd + 0.5;
          } else {
            if (vc.rm) { ch.c_dir = true; ch.ldc = vc.ld_rm; ch.c_sr = vc.sr; ch.c_sc = vc.scol; }
            else if (vc.cm) { ch.c_dir = true; ch.c_swap = true; ch.ldc = vc.ld_cm; ch.c_sr = vc.sr; ch.c_sc = vc.scol; }
            else cost += (beta != 0.0 ? 3.0 : 2.0) * szC;
            if (vc.any && !ch.c_dir) { ch.c_sr = vc.sr; ch.c_sc = vc.scol; }
            if (bcls != 0) cost += 0.25;
            // many tiny batched GEMMs are slow: discourage when the per-batch problem is small
            if (bcls != 0 && (double)Md * Nd < 1024.0) cost += 1e3 * (double)nb;
          }
          ch.sA = (bcls == 1 || bcls == 3) ? gA.str : 0;
          ch.sB = (bcls == 2 || bcls == 3) ? gB.str : 0;
          ch.sC = (bcls == 1 || bcls == 2) ? gC.str : 0;
          ch.cost = cost;
          if (cost < best.cost) best = ch;
          if (bcls == 0 && cost < best0.cost) best0 = ch;
        }
  }
  if (best.cost >= 1e299) throw PlanError("contract: no lowering for " + tag);

  // A batched DMMA lowering that avoids a permute may still lose against ONE large INT8 product plus that permute
  // (e.g. 'ijbc,ca->ijab': 1600 products of 400^3 at 18 TFLOP/s vs one 640000 x 400 x 400 product and a transposed
  // accumulate of the result): compare the two with the same cost models as below.
  if (oz_ns > 0 && oz_min_flops >= 0.0 && best.bcls != 0 && best0.cost < 1e299) {
    const int64_t M0 = dims_of(best0.om, dm), N0 = dims_of(best0.on, dm), K0 = dims_of(best0.ok, dm);
    const double fl0 = 2.0 * (double)M0 * (double)N0 * (double)K0;
    const bool plain = (K0 + 31) / 32 <= 65535 && A.slot != S_VVVV_P && B.slot != S_VVVV_P && A.slot != S_OVVV_P &&
                       B.slot != S_OVVV_P;
    if (plain && fl0 >= oz_min_flops) {
      MatView vc0 = mat_view(C, sc, best0.om, best0.on);
      const double perm0 = 8.0 * best0.cost / 2.5e12, perm1 = 8.0 * best.cost / 2.5e12;
      const double cut = (8.0 + 2.0 * oz_ns) * ((double)M0 + (double)N0) * (double)K0 / 5e12;
      const double t_oz = oz_time(oz_ns, sm_count, M0, N0, K0, vc0.any ? vc0.sr : N0, vc0.any ? vc0.scol : 1,
                                  vc0.any ? beta : 0.0, nullptr) + cut + perm0 + 2e-5;
      const double t_dmma = fl0 / 1.8e13 + perm1;
      if (t_oz < 0.7 * t_dmma) best = best0;
    }
  }
  const Choice& ch = best;
  const int64_t nb = ch.bt.empty() ? 1 : dims_of(ch.bt, dm);
  const int64_t Md = dims_of(ch.om, dm), Nd = dims_of(ch.on, dm), Kd = dims_of(ch.ok, dm);
  auto dimvec = [&](const std::string& g) {
    std::vector<int64_t> v;
    for (char c : g) v.push_back(dm.at(c));
    return v;
  };
  std::vector<Tensor> to_free;

  Op g;
  g.kind = OP_GEMM;
  g.M = Md; g.N = Nd; g.K = Kd;
  g.batch = nb;
  g.alpha = alpha;
  g.note = std::string(note) + " [" + tag + "]";

  // ---- INT8 tensor-core route (ozaki.cu): one unbatched GEMM, operands cut into digit planes
  {
    const bool const_a = (vvvv_planes && A.slot == S_VVVV_P) || (ovvv_planes && A.slot == S_OVVV_P);
    const bool const_b = (vvvv_planes && B.slot == S_VVVV_P) || (ovvv_planes && B.slot == S_OVVV_P);
    const bool const_planes = const_a || const_b;
    const double fl = 2.0 * (double)Md * (double)Nd * (double)Kd;
    bool oz = oz_ns > 0 && ch.bcls == 0 && Kd >= 1 && (Kd + 31) / 32 <= 65535;
    const int64_t S = (oz && !const_planes) ? oz_pick_splits(oz_ns, sm_count, Md, Nd, Kd, oz_splitk_min_k) : 1;
    if (oz && oz_min_flops >= 0.0) {
      // INT8 route (model in oz_time) + cutting the operands (8 B read + ns B written and re-read) against the
      // DMMA route at 30 TFLOP/s: skinny, few-tile or short-K products stay on the DMMA kernels
      MatView vcm = mat_view(C, sc, ch.om, ch.on);
      const double cut = (8.0 + 2.0 * oz_ns) * ((const_a ? 0.0 : (double)Md) + (const_b ? 0.0 : (double)Nd)) * (double)Kd / 5e12;
      const double t_oz = oz_time(oz_ns, sm_count, Md, Nd, Kd, vcm.any ? vcm.sr : Nd, vcm.any ? vcm.scol : 1, beta, nullptr, S) +
                          cut + 2e-5;
      // the DMMA kernels reach ~30 TFLOP/s on large plain GEMMs, ~18 on split-K / few-tile shapes
      oz = fl >= oz_min_flops && t_oz < 0.8 * fl / (S > 1 ? 1.8e13 : 3.0e13);
    } else if (oz && oz_min_flops < -1.5) {
      // test configuration: a pure flop threshold -oz_min_flops without the time model, so that small shapes can be
      // given the routing the benchmark shape has (ladders, rings, R4/R6/R9 on the INT8 pipe, the rest on DMMA)
      oz = fl >= -oz_min_flops;
    }
    if (const_planes && !(oz_ns > 0 && ch.bcls == 0 && ch.a_dir && ch.b_dir))
      throw PlanError("contract: an operand is bound as digit planes but the contraction is not a plain GEMM: " + tag);
    if (oz || const_planes) {
      Tensor tA = A, tB = B;
      int64_t ars, aks, brs, bks;
      if (ch.a_dir) { ars = ch.ta ? 1 : ch.lda; aks = ch.ta ? ch.lda : 1; }
      else {
        std::vector<int64_t> dv = dimvec(ch.om + ch.ok);
        tA = tmpv(dv);
        permute(1.0, A, sa, 0.0, tA, (ch.om + ch.ok).c_str(), "engine:A");
        to_free.push_back(tA);
        ars = std::max<int64_t>(Kd, 1); aks = 1;
      }
      if (ch.b_dir) { brs = ch.tb ? ch.ldb : 1; bks = ch.tb ? 1 : ch.ldb; }
      else {
        std::vector<int64_t> dv = dimvec(ch.ok + ch.on);
        tB = tmpv(dv);
        permute(1.0, B, sb, 0.0, tB, (ch.ok + ch.on).c_str(), "engine:B");
        to_free.push_back(tB);
        brs = 1; bks = std::max<int64_t>(Nd, 1);
      }
      MatView vc = mat_view(C, sc, ch.om, ch.on);
      const std::string nt = std::string(note) + " [" + tag + "]";
      if (S > 1) {
        // split-K: S products over the chunks of a two-level index, partial results summed in a fixed order
        OzSet a = oz_cut(tA, Md, ars, S, (Kd / S) * aks, Kd / S, aks, nt);
        OzSet b = oz_cut(tB, Nd, brs, S, (Kd / S) * bks, Kd / S, bks, nt);
        Tensor part = tmp({S, Md, Nd});
        OzSel sel;
        sel.k1b = 1; sel.nk1 = 1;
        oz_mm(alpha, a, sel, b, sel, Md, Nd, S, 0.0, part, Nd, 1, Md * Nd, nt + " [split-K]");
        oz_release(b);
        oz_release(a);
        Op r;
        r.kind = OP_REDUCE;
        r.a = part;
        r.i0 = S;
        r.M = Md; r.N = Nd;
        r.alpha = 1.0;
        r.note = nt;
        if (vc.any) {
          r.c = C; r.beta = beta; r.i1 = Md == 1 ? 0 : vc.sr; r.i2 = Nd == 1 ? 0 : vc.scol;
          ops.push_back(r);
        } else {
          std::string lay = ch.om + ch.on;
          Tensor tC = tmpv(dimvec(lay));
          r.c = tC; r.beta = 0.0; r.i1 = Nd; r.i2 = 1;
          ops.push_back(r);
          permute(1.0, tC, lay.c_str(), beta, C, sc, "engine:C");
          release(tC);
        }
        release(part);
      } else if (vc.any) {
        emit_oz(alpha, tA, ars, aks, tB, brs, bks, Md, Nd, Kd, beta, C, Md == 1 ? 0 : vc.sr, Nd == 1 ? 0 : vc.scol, nt);
      } else {
        std::string lay = ch.om + ch.on;
        Tensor tC = tmpv(dimvec(lay));
        emit_oz(alpha, tA, ars, aks, tB, brs, bks, Md, Nd, Kd, 0.0, tC, Nd, 1, nt);
        permute(1.0, tC, lay.c_str(), beta, C, sc, "engine:C");
        release(tC);
      }
      for (auto& t : to_free) release(t);
      return;
    }
  }

  // ---- A operand
  if (ch.a_dir) {
    g.a = A; g.ta = ch.ta; g.lda = ch.lda; g.sA = ch.sA;
  } else {
    std::string lay = ((ch.bcls == 1 || ch.bcls == 3) ? ch.bt : std::string()) + ch.om + ch.ok;
    std::vector<int64_t> dv = dimvec(lay);
    if (dv.empty()) dv.push_back(1);
    Tensor tA = tmpv(dv);
    if (lay.empty()) lay = "";  // scalar case cannot occur (A has rank>=1)
    permute(1.0, A, sa, 0.0, tA, lay.c_str(), "engine:A");
    to_free.push_back(tA);
    g.a = tA; g.ta = 0; g.lda = std::max<int64_t>(Kd, 1);
    g.sA = (ch.bcls == 1 || ch.bcls == 3) ? Md * Kd : 0;
  }
  // ---- B operand
  if (ch.b_dir) {
    g.b = B; g.tb = ch.tb; g.ldb = ch.ldb; g.sB = ch.sB;
  } else {
    std::string lay = ((ch.bcls == 2 || ch.bcls == 3) ? ch.bt : std::string()) + ch.ok + ch.on;
    Tensor tB = tmpv(dimvec(lay));
    permute(1.0, B, sb, 0.0, tB, lay.c_str(), "engine:B");
    to_free.push_back(tB);
    g.b = tB; g.tb = 0; g.ldb = std::max<int64_t>(Nd, 1);
    g.sB = (ch.bcls == 2 || ch.bcls == 3) ? Kd * Nd : 0;
  }

  // ---- split-K decision (only when there is no free-index batch)
  int64_t R = (ch.bcls == 3) ? nb : 1;
  int64_t S = 1;
  if (ch.bcls == 0 || ch.bcls == 3) {
    int bm = 128, bn = 128;
    gemm_tile_of(Md, Nd, Kd, &bm, &bn);
    bm = std::max(bm, 48);                       // the small Gram tiles keep the split count of the 48-wide ones
    bn = std::max(bn, 48);
    int64_t tiles = ((Md + bm - 1) / bm) * ((Nd + bn - 1) / bn) * R;
    if (tiles < 2 * sm_count && Kd >= 1024) {
      S = std::min<int64_t>((2 * sm_count + tiles - 1) / tiles, Kd / 512);
      while (S > 1 && (double)S * R * Md * Nd * 8.0 > 512e6) --S;
      if (S < 2) S = 1;
    }
  }

  if (R * S > 1) {
    // GEMM into partials [R*S, M, N], then reduce into the target
    Tensor part = tmp({R * S, Md, Nd});
    g.c = part; g.ldc = std::max<int64_t>(Nd, 1); g.sC = Md * Nd; g.beta = 0.0;
    g.batch = R * S;
    g.splitk = S;
    g.kchunk = S > 1 ? ((Kd + S - 1) / S + 15) / 16 * 16 : Kd;
    if (S > 1) {  // chunks may not be empty for any s
      while (S > 1 && (S - 1) * g.kchunk >= Kd) { --S; }
      g.splitk = S; g.batch = R * S;
    }
    gemm_flops += 2.0 * (double)Md * Nd * Kd * (double)R;
    ops.push_back(g);
    Op r;
    r.kind = OP_REDUCE;
    r.a = part;
    r.i0 = R * S;
    r.M = Md; r.N = Nd;
    r.alpha = 1.0;
    r.note = g.note;
    if (ch.c_dir) {
      r.c = C; r.beta = beta; r.i1 = ch.c_sr; r.i2 = ch.c_sc;
      if (Md == 1) r.i1 = 0;
      if (Nd == 1) r.i2 = 0;
      ops.push_back(r);
    } else {
      std::string lay = ch.om + ch.on;
      std::vector<int64_t> dv = dimvec(lay);
      if (dv.empty()) dv.push_back(1);
      Tensor tC = tmpv(dv);
      r.c = tC; r.beta = 0.0; r.i1 = Nd; r.i2 = 1;
      ops.push_back(r);
      permute(1.0, tC, lay.c_str(), beta, C, sc, "engine:C");
      release(tC);
    }
    release(part);
  } else {
    if (ch.c_dir) {
      g.c = C; g.ldc = ch.ldc; g.sC = ch.sC; g.beta = beta;
      if (ch.c_swap) {  // compute C^T = B^T A^T
        std::swap(g.a, g.b);
        std::swap(g.M, g.N);
        std::swap(g.sA, g.sB);
        int ta = g.ta, tb = g.tb;
        int64_t lda = g.lda, ldb = g.ldb;
        g.ta = !tb; g.tb = !ta; g.lda = ldb; g.ldb = lda;
      }
      gemm_flops += 2.0 * (double)Md * Nd * Kd * (double)nb;
      ops.push_back(g);
    } else {
      std::string lay = ((ch.bcls == 1 || ch.bcls == 2) ? ch.bt : std::string()) + ch.om + ch.on;
      std::vector<int64_t> dv = dimvec(lay);
      if (dv.empty()) dv.push_back(1);
      Tensor tC = tmpv(dv);
      g.c = tC; g.ldc = std::max<int64_t>(Nd, 1); g.sC = Md * Nd; g.beta = 0.0;
      gemm_flops += 2.0 * (double)Md * Nd * Kd * (double)nb;
      ops.push_back(g);
      permute(1.0, tC, lay.c_str(), beta, C, sc, "engine:C");
      release(tC);
    }
  }
  for (auto& t : to_free) release(t);
}

// ---------------------------------------------------------------- INT8-pipe GEMM

// Seconds (model) of one INT8-route GEMM for both role assignments; tile = 128 rows of the first operand x TN rows
// of the second.  Main loop: padded product at ~100 TFLOP/s FP64-equivalent for 7 digits (scaled by the digit-pair
// count), derated when fewer tiles than SMs; epilogue: the C tile is written (and read when beta != 0) by one thread
// per tile row — coalesced when the tile rows are contiguous in C, 16-byte pieces otherwise.
static double oz_time(int ns, int sm_count, int64_t M, int64_t N, int64_t K, int64_t crs, int64_t ccs, double beta,
                      bool* swap_out, int64_t splits) {
  auto pad = [](int64_t x, int64_t g) { return (x + g - 1) / g * g; };
  const int TN = ozaki_tile_n(ns);
  const double rate = 1.0e14 * 28.0 / (0.5 * ns * (ns + 1));
  double best = 1e300;
  for (int sw = 0; sw < 2; ++sw) {
    const int64_t m = sw ? N : M, n = sw ? M : N, rs = sw ? ccs : crs;
    const double tiles = (double)(pad(m, 128) / 128) * (double)(pad(n, TN) / TN) * (double)splits;
    const double waves = std::ceil(tiles / (double)sm_count);
    const double eff = tiles / (waves * (double)sm_count);
    const double main = 2.0 * (double)K * (double)pad(m, 128) * (double)pad(n, TN) / (rate * eff);
    const double epi = 8.0 * (double)M * (double)N * (beta != 0.0 ? 2.0 : 1.0) / (rs == 1 ? 3.0e12 : 0.5e12);
    if (main + epi < best) { best = main + epi; if (swap_out) *swap_out = sw != 0; }
  }
  return best;
}

// Few output tiles and a long contraction index: cut K into S equal chunks (a two-level index, one product per
// chunk, partial results summed by a reduce op).  S = the divisor of K/32 up to 64 that fills the SMs best.
static int64_t oz_pick_splits(int ns, int sm_count, int64_t M, int64_t N, int64_t K, int64_t min_k) {
  auto pad = [](int64_t x, int64_t g) { return (x + g - 1) / g * g; };
  const int TN = ozaki_tile_n(ns);
  const int64_t tiles = std::min((pad(M, 128) / 128) * (pad(N, TN) / TN), (pad(N, 128) / 128) * (pad(M, TN) / TN));
  if (min_k <= 0 || K < min_k || K % 32 != 0 || tiles * 2 > sm_count) return 1;
  int64_t best = 1;
  double best_eff = (double)tiles / (double)sm_count;
  for (int64_t S = 2; S <= 64; ++S) {
    if ((K / 32) % S != 0) continue;
    const double items = (double)(tiles * S);
    const double eff = items / (std::ceil(items / (double)sm_count) * (double)sm_count);
    if (eff > best_eff + 0.02) { best_eff = eff; best = S; }
  }
  return best;
}

namespace {
// element range [lo, hi] a strided view can touch
void view_range(const Tensor& t, int64_t* lo, int64_t* hi) {
  int64_t a = t.off, b = t.off;
  for (int i = 0; i < t.nd; ++i) {
    if (t.dim[i] <= 0) { *lo = t.off; *hi = t.off - 1; return; }
    const int64_t span = (t.dim[i] - 1) * t.str[i];
    if (span >= 0) b += span; else a += span;
  }
  *lo = a; *hi = b;
}
}  // namespace

// has any op after `op_index` written into [lo, hi] of `slot`?  (conservative: ranges of strided views)
bool Plan::written_since(size_t op_index, int slot, int64_t lo, int64_t hi) const {
  auto hits = [&](const Tensor& t, int64_t extra = 0) {
    if (!t.valid() || t.slot != slot) return false;
    int64_t a, b;
    view_range(t, &a, &b);
    b += extra;
    return !(b < lo || a > hi);
  };
  for (size_t k = op_index + 1; k < ops.size(); ++k) {
    const Op& op = ops[k];
    switch (op.kind) {
      case OP_OZ_SPLIT: if (hits(op.c) || hits(op.d)) return true; break;
      case OP_DOT: break;                                   // writes only its scratch partials (released at once) and scal
      case OP_GEMM: {                                       // batched / split-K outputs: batch * sC beyond the first matrix
        Tensor c = op.c;
        int64_t a, b;
        view_range(c, &a, &b);
        const int64_t ext = (op.M - 1) * std::max<int64_t>(op.ldc, 1) + op.N - 1 + (op.batch - 1) * op.sC;
        if (c.slot == slot && !(a + std::max<int64_t>(ext, b - a) < lo || a > hi)) return true;
        break;
      }
      case OP_OZ_GEMM: {
        if (op.c.slot != slot) break;
        const int64_t a = op.c.off;
        const int64_t ext = (op.M - 1) * std::max<int64_t>(op.i1, 0) + (op.N - 1) * std::max<int64_t>(op.i2, 0) +
                            (op.batch - 1) * op.sC;
        if (!(a + ext < lo || a > hi)) return true;
        break;
      }
      case OP_REDUCE: {
        if (op.c.slot != slot) break;
        const int64_t a = op.c.off, ext = (op.M - 1) * op.i1 + (op.N - 1) * op.i2;
        if (!(a + ext < lo || a > hi)) return true;
        break;
      }
      case OP_ALLGATHER: case OP_ALLTOALL:
        if (op.c.slot == slot && !(op.c.off + op.i0 * op.i1 - 1 < lo || op.c.off > hi)) return true;
        break;
      default:
        if (hits(op.c)) return true;
    }
  }
  return false;
}

// entry i leaves the cache: its planes are freed now, or — when a product that was handed the set has not been
// emitted yet (oz_cut without its oz_release) — by that oz_release
void Plan::retire_cut(size_t i) {
  CutEntry& e = cut_cache[i];
  if (e.users > 0) {
    cut_orphans.push_back(e);
  } else {
    arena.release(e.set.stats.off);
    arena.release(e.set.planes.off);
  }
  cut_cache.erase(cut_cache.begin() + i);
}

void Plan::drop_cuts_of(int slot, int64_t lo, int64_t hi) {
  for (size_t i = 0; i < cut_cache.size();) {
    CutEntry& e = cut_cache[i];
    if (e.slot == slot && !(e.hi < lo || e.lo > hi)) retire_cut(i);
    else ++i;
  }
}

OzSet Plan::oz_cut(const Tensor& X, int64_t R, int64_t rs, int64_t K1, int64_t ks1, int64_t K2, int64_t ks2,
                   const std::string& note) {
  if (oz_ns <= 0) throw PlanError("oz_cut: the INT8 engine is off");
  // the element range the cut reads
  int64_t lo = X.off, hi = X.off + (R - 1) * rs + (K1 - 1) * ks1 + (K2 - 1) * ks2;
  const bool cacheable = R * K1 * K2 >= cut_cache_min_elems && rs >= 0 && ks1 >= 0 && ks2 >= 0;
  if (cacheable) {
    for (CutEntry& e : cut_cache) {
      if (e.slot == X.slot && e.off == X.off && e.R == R && e.rs == rs && e.K1 == K1 && e.ks1 == (K1 > 1 ? ks1 : e.ks1) &&
          e.K2 == K2 && e.ks2 == ks2 && e.ns == oz_ns && !written_since(e.op_index, e.slot, e.lo, e.hi)) {
        ++cut_cache_hits;
        ++e.users;
        return e.set;
      }
    }
    // a stale entry of the same source is useless from now on
    for (size_t i = 0; i < cut_cache.size();) {
      CutEntry& e = cut_cache[i];
      if (e.slot == X.slot && !(e.hi < lo || e.lo > hi) && written_since(e.op_index, e.slot, e.lo, e.hi)) retire_cut(i);
      else ++i;
    }
  }
  OzSet s;
  s.R = R; s.K1 = K1; s.K2 = K2;
  s.owned = !cacheable;
  s.cached = cacheable;
  s.planes = tmp({ozaki_plane_elems(R, K1, K2, oz_ns)});
  s.stats = tmp({ozaki_stat_elems(R, K1)});
  Op sp;
  sp.kind = OP_OZ_SPLIT;
  sp.a = X;
  sp.c = s.planes;
  sp.d = s.stats;
  sp.M = R; sp.K = K2; sp.i1 = K1;
  sp.lda = rs; sp.ldb = ks2; sp.ldc = ks1;
  sp.i0 = oz_ns;
  sp.note = note;
  ops.push_back(sp);
  if (cacheable) {
    CutEntry e{X.slot, X.off, R, rs, K1, ks1, K2, ks2, oz_ns, lo, hi, ops.size() - 1, s, 1};
    cut_cache.push_back(e);
  }
  return s;
}

void Plan::oz_release(const OzSet& s) {
  if (s.owned) {
    release(s.stats);
    release(s.planes);
    return;
  }
  if (!s.cached) return;                     // constant plane sets
  for (CutEntry& e : cut_cache)
    if (e.set.planes.off == s.planes.off) {
      if (e.users > 0) --e.users;
      return;
    }
  for (size_t i = 0; i < cut_orphans.size(); ++i) {
    CutEntry& e = cut_orphans[i];
    if (e.set.planes.off != s.planes.off) continue;
    if (--e.users <= 0) {
      arena.release(e.set.stats.off);
      arena.release(e.set.planes.off);
      cut_orphans.erase(cut_orphans.begin() + i);
    }
    return;
  }
}

OzSet Plan::oz_const_vvvv(int64_t rows) const {
  const int64_t pv = npair(nvir);
  OzSet s;
  s.R = rows; s.K1 = 1; s.K2 = pv;
  s.planes = make_tensor(S_VVVV_OZ, 0, {ozaki_plane_elems(rows, 1, pv, oz_ns)});
  s.stats = make_tensor(S_VVVV_OZS, 0, {ozaki_stat_elems(rows, 1)});
  return s;
}
OzSet Plan::oz_const_ovvv1() const {
  const int64_t pv = npair(nvir);
  OzSet s;
  s.R = nocc * nvir; s.K1 = 1; s.K2 = pv;
  s.planes = make_tensor(S_OVVV_OZ1, 0, {ozaki_plane_elems(s.R, 1, pv, oz_ns)});
  s.stats = make_tensor(S_OVVV_OZ1S, 0, {ozaki_stat_elems(s.R, 1)});
  return s;
}
OzSet Plan::oz_const_ovvv2() const {
  const int64_t pv = npair(nvir);
  OzSet s;
  s.R = pv; s.K1 = nocc; s.K2 = nvir;
  s.planes = make_tensor(S_OVVV_OZ2, 0, {ozaki_plane_elems(pv, nocc, nvir, oz_ns)});
  s.stats = make_tensor(S_OVVV_OZ2S, 0, {ozaki_stat_elems(pv, nocc)});
  return s;
}

void Plan::oz_mm(double alpha, const OzSet& A, const OzSel& a, const OzSet& B, const OzSel& b, int64_t M, int64_t N,
                 int64_t batch, double beta, const Tensor& C, int64_t crs, int64_t ccs, int64_t c_b,
                 const std::string& note) {
  const int64_t ank1 = a.nk1 > 0 ? a.nk1 : A.K1, bnk1 = b.nk1 > 0 ? b.nk1 : B.K1;
  if (A.K2 != B.K2 || ank1 != bnk1) throw PlanError("oz_mm: contraction ranges differ in " + note);
  if ((ank1 != A.K1 && ank1 != 1) || (bnk1 != B.K1 && bnk1 != 1))
    throw PlanError("oz_mm: a partial k1 range must be a single k1 in " + note);
  if (((a.row0 | a.rowb | b.row0 | b.rowb) & 7) != 0) throw PlanError("oz_mm: row offsets must be multiples of 8 in " + note);
  const int64_t K = ank1 * A.K2;
  Op g;
  g.kind = OP_OZ_GEMM;
  g.alpha = alpha; g.beta = beta;
  g.c = C;
  g.K = K;
  g.i0 = oz_ns;
  g.batch = batch;
  g.sC = c_b;
  g.note = note;
  bool swap = false;
  oz_time(oz_ns, sm_count, M, N, K, crs, ccs, beta, &swap);
  const OzSet& X = swap ? B : A;
  const OzSet& Y = swap ? A : B;
  const OzSel& x = swap ? b : a;
  const OzSel& y = swap ? a : b;
  g.a = X.planes; g.d = X.stats; g.lda = X.R;
  g.b = Y.planes; g.e = Y.stats; g.ldb = Y.R;
  g.M = swap ? N : M; g.N = swap ? M : N;
  g.i1 = swap ? ccs : crs; g.i2 = swap ? crs : ccs;
  auto fill = [&](const OzSet& S, const OzSel& e, int64_t nk1, int64_t* row0, int64_t* rowb, int64_t* kb0, int64_t* kbb,
                  int64_t* t0, int64_t* tb) {
    *row0 = e.row0; *rowb = e.rowb;
    *kb0 = e.k10 * S.nkb2(); *kbb = e.k1b * S.nkb2();
    if (nk1 == S.K1) { *t0 = S.rp(); *tb = 0; }                          // whole-index row sums
    else { *t0 = (2 + e.k10) * S.rp(); *tb = e.k1b * S.rp(); }          // sums of one k1
  };
  fill(X, x, ank1, &g.oz[0], &g.oz[1], &g.oz[4], &g.oz[5], &g.oz[8], &g.oz[9]);
  fill(Y, y, ank1, &g.oz[2], &g.oz[3], &g.oz[6], &g.oz[7], &g.oz[10], &g.oz[11]);
  g.oz[12] = ank1 * A.nkb2();
  ops.push_back(g);
  gemm_flops += 2.0 * (double)M * N * K * (double)batch;
  oz_flops += 2.0 * (double)M * N * K * (double)batch;
}

void Plan::emit_oz(double alpha, const Tensor& A, int64_t ars, int64_t aks, const Tensor& B, int64_t brs, int64_t bks,
                   int64_t M, int64_t N, int64_t K, double beta, const Tensor& C, int64_t crs, int64_t ccs,
                   const std::string& note) {
  const int64_t pv = npair(nvir);
  // the (m, a) contraction index of the constant ovvv plane set OZ2 is two-level (a padded per m): the other
  // operand of such a product is cut with the same structure
  auto is_oz2 = [&](const Tensor& X, int64_t R, int64_t rs, int64_t ks) {
    return ovvv_planes && X.slot == S_OVVV_P && X.off == 0 && rs == 1 && ks == pv && R == pv && K == nocc * nvir;
  };
  const bool two_level = is_oz2(A, M, ars, aks) || is_oz2(B, N, brs, bks);
  const int64_t K1 = two_level ? nocc : 1, K2 = two_level ? nvir : K;
  struct Side { OzSet set; OzSel sel; };
  auto prepare = [&](const Tensor& X, int64_t R, int64_t rs, int64_t ks) {
    Side s;
    if (vvvv_planes && X.slot == S_VVVV_P) {
      // the constant row shard of the packed vvvv: [R, K] with K contiguous, cut once at upload time
      // (a one-row shard has no meaningful row stride, and the engine may read it as a column)
      if (X.off != 0 || K != pv || (R > 1 && (ks != 1 || rs != K)))
        throw PlanError("vvvv_p digit planes: unexpected operand view in " + note);
      s.set = oz_const_vvvv(R);
      return s;
    }
    if (ovvv_planes && X.slot == S_OVVV_P) {
      if (is_oz2(X, R, rs, ks)) { s.set = oz_const_ovvv2(); return s; }
      if (ks == 1 && rs == pv && K == pv && X.off % pv == 0 && (X.off / pv) % 8 == 0 && X.off / pv + R <= nocc * nvir) {
        s.set = oz_const_ovvv1();
        s.sel.row0 = X.off / pv;       // a range of (m,a) rows
        return s;
      }
      throw PlanError("ovvv_p digit planes: unexpected operand view in " + note);
    }
    s.set = oz_cut(X, R, rs, K1, K2 * ks, K2, ks, note);
    return s;
  };
  Side a = prepare(A, M, ars, aks), b = prepare(B, N, brs, bks);
  oz_mm(alpha, a.set, a.sel, b.set, b.sel, M, N, 1, beta, C, crs, ccs, 0, note);
  oz_release(b.set);
  oz_release(a.set);
}

// ---------------------------------------------------------------- dump
static void dump_tensor(std::ostringstream& o, const char* key, const Tensor& t) {
  o << "\"" << key << "\":";
  if (!t.valid()) { o << "null"; return; }
  o << "{\"slot\":\"" << slot_name(t.slot) << "\",\"off\":" << t.off << ",\"dim\":[";
  for (int i = 0; i < t.nd; ++i) o << (i ? "," : "") << t.dim[i];
  o << "],\"str\":[";
  for (int i = 0; i < t.nd; ++i) o << (i ? "," : "") << t.str[i];
  o << "]}";
}

const char* op_kind_name(int kind) {
  static const char* names[] = {"gemm", "reduce", "permute", "fill", "tau", "pack", "unpack", "finish",
                                "dot", "scale_dev", "diag_add", "rdm1", "ewise", "allgather", "oz_split", "oz_gemm",
                                "asym4", "alltoall"};
  static_assert(sizeof(names) / sizeof(names[0]) == OP_ALLTOALL + 1, "one name per OpKind");
  if (kind < 0 || kind > OP_ALLTOALL) return "?";
  return names[kind];
}

std::string Plan::dump_json() const {
  std::ostringstream o;
  o.precision(17);
  o << "{\"workspace_elems\":" << arena.peak << ",\"gemm_flops\":" << gemm_flops << ",\"oz_flops\":" << oz_flops
    << ",\"perm_bytes\":" << perm_bytes << ",\"ops\":[";
  for (size_t i = 0; i < ops.size(); ++i) {
    const Op& p = ops[i];
    if (i) o << ",";
    o << "\n{\"kind\":\"" << op_kind_name(p.kind) << "\",";
    dump_tensor(o, "a", p.a); o << ",";
    dump_tensor(o, "b", p.b); o << ",";
    dump_tensor(o, "c", p.c); o << ",";
    dump_tensor(o, "d", p.d); o << ",";
    dump_tensor(o, "e", p.e); o << ",";
    o << "\"alpha\":" << p.alpha << ",\"beta\":" << p.beta << ",\"M\":" << p.M << ",\"N\":" << p.N
      << ",\"K\":" << p.K << ",\"lda\":" << p.lda << ",\"ldb\":" << p.ldb << ",\"ldc\":" << p.ldc
      << ",\"sA\":" << p.sA << ",\"sB\":" << p.sB << ",\"sC\":" << p.sC << ",\"batch\":" << p.batch
      << ",\"ta\":" << p.ta << ",\"tb\":" << p.tb << ",\"splitk\":" << p.splitk << ",\"kchunk\":" << p.kchunk
      << ",\"i0\":" << p.i0 << ",\"i1\":" << p.i1 << ",\"i2\":" << p.i2 << ",\"i3\":" << p.i3
      << ",\"d0\":" << p.d0 << ",\"d1\":" << p.d1 << ",\"oz\":[";
    for (int q = 0; q < 13; ++q) o << (q ? "," : "") << p.oz[q];
    o << "],\"note\":\"" << p.note << "\"}";
  }
  o << "\n]}";
  return o.str();
}

}  // namespace ecw
