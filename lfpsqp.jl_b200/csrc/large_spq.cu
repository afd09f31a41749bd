// large_spq.cu -- LFPSQP_FAM_SPARSE_QCQP: validation of the lfpsqp_sparse_qcqp descriptor and the canonical structures the
// device kernels read (large_families.cuh), built once on the host in a fixed order and uploaded at setup.
#include <cuda_runtime.h>
#include <math.h>
#include <algorithm>
#include <vector>

#include "ctx.h"
#include "large_state.h"

namespace {

constexpr int64_t kMax32 = (int64_t)1 << 31;

struct Ent {
  int32_t mat;   // constraint index (0 for P and Ac)
  int64_t key;   // row * ncols + col
  double val;
  bool operator<(const Ent &o) const { return mat != o.mat ? mat < o.mat : key < o.key; }
};

// reads one coordinate list: every check of the header, then the entries sorted by (mat, row, col) without duplicates
int read_coo(lfpsqp_ctx *c, const char *name, const lfpsqp_coo &A, bool stacked, int64_t nrows, int64_t ncols, int64_t nmat,
             std::vector<Ent> &out) {
  const int64_t nnz = A.nnz;
  if (nnz < 0 || nnz >= kMax32) return c->fail(LFPSQP_ERR_ARG, "sparse QCQP: %s.nnz = %lld; it must be in [0, 2^31)", name, (long long)nnz);
  if (nnz > 0 && (!A.row || !A.col || !A.val || (stacked && !A.mat)))
    return c->fail(LFPSQP_ERR_ARG, "sparse QCQP: %s has nnz = %lld but a NULL %s array", name, (long long)nnz,
                   !A.row ? "row" : !A.col ? "col" : !A.val ? "val" : "mat");
  if (!stacked && A.mat) return c->fail(LFPSQP_ERR_ARG, "sparse QCQP: %s.mat must be NULL (only Qc is a stack)", name);
  out.resize((size_t)nnz);
  for (int64_t k = 0; k < nnz; k++) {
    const int64_t r = A.row[k], cc = A.col[k], mt = stacked ? A.mat[k] : 0;
    const double v = A.val[k];
    if (r < 0 || r >= nrows || cc < 0 || cc >= ncols)
      return c->fail(LFPSQP_ERR_ARG, "sparse QCQP: %s entry %lld: index (%lld, %lld) out of range for %lld x %lld", name, (long long)k,
                     (long long)r, (long long)cc, (long long)nrows, (long long)ncols);
    if (mt < 0 || mt >= nmat)
      return c->fail(LFPSQP_ERR_ARG, "sparse QCQP: %s entry %lld: constraint index %lld not in [0, m = %lld)", name, (long long)k,
                     (long long)mt, (long long)nmat);
    if (!isfinite(v)) return c->fail(LFPSQP_ERR_ARG, "sparse QCQP: %s entry %lld is not finite", name, (long long)k);
    out[(size_t)k] = Ent{(int32_t)mt, r * ncols + cc, v};
  }
  std::sort(out.begin(), out.end());
  for (size_t k = 1; k < out.size(); k++)
    if (out[k].mat == out[k - 1].mat && out[k].key == out[k - 1].key)
      return c->fail(LFPSQP_ERR_ARG, "sparse QCQP: %s has a duplicate entry (matrix %d, %lld, %lld)", name, out[k].mat,
                     (long long)(out[k].key / ncols), (long long)(out[k].key % ncols));
  return 0;
}

// every off-diagonal entry (r, c) of each n x n matrix has its mirror (c, r) with exactly the same value
int check_symmetric(lfpsqp_ctx *c, const char *name, const std::vector<Ent> &e, int64_t n) {
  for (const Ent &a : e) {
    const int64_t r = a.key / n, cc = a.key % n;
    if (r == cc) continue;
    const Ent probe{a.mat, cc * n + r, 0.0};
    auto it = std::lower_bound(e.begin(), e.end(), probe);
    const bool found = it != e.end() && it->mat == a.mat && it->key == probe.key;
    if (!found || it->val != a.val)
      return c->fail(LFPSQP_ERR_ARG, "sparse QCQP: %s (matrix %d) is not exactly symmetric: entry (%lld, %lld) = %.17g, (%lld, %lld) = %.17g",
                     name, a.mat, (long long)r, (long long)cc, a.val, (long long)cc, (long long)r, found ? it->val : 0.0);
  }
  return 0;
}

int check_vector(lfpsqp_ctx *c, const char *name, const double *v, int64_t len) {
  if (!v) return 0;
  for (int64_t k = 0; k < len; k++)
    if (!isfinite(v[k])) return c->fail(LFPSQP_ERR_ARG, "sparse QCQP: %s[%lld] is not finite", name, (long long)k);
  return 0;
}

template <class T> bool upload(LargeState &S, const T **dst, const std::vector<T> &h) {
  void *p = nullptr;
  if (cudaMalloc(&p, std::max<size_t>(h.size(), 1) * sizeof(T)) != cudaSuccess) { cudaGetLastError(); return false; }
  S.owned.push_back(p);
  if (!h.empty() && cudaMemcpyAsync(p, h.data(), h.size() * sizeof(T), cudaMemcpyHostToDevice, S.stream) != cudaSuccess) return false;
  *dst = (const T *)p;
  return true;
}

}  // namespace

int spq_build(lfpsqp_ctx *c, const lfpsqp_sparse_qcqp *D, int64_t n, int64_t m, SpqHost &H) {
  if (n >= kMax32) return c->fail(LFPSQP_ERR_ARG, "sparse QCQP: n must be < 2^31");
  std::vector<Ent> P, Q, A;
  int rc;
  if ((rc = read_coo(c, "P", D->P, false, n, n, 1, P))) return rc;
  if ((rc = read_coo(c, "Qc", D->Qc, true, n, n, m, Q))) return rc;
  if ((rc = read_coo(c, "Ac", D->Ac, false, m, n, 1, A))) return rc;
  if ((rc = check_symmetric(c, "P", P, n))) return rc;
  if ((rc = check_symmetric(c, "Qc", Q, n))) return rc;
  if ((rc = check_vector(c, "q", D->q, n)) || (rc = check_vector(c, "bc", D->bc, m)) || (rc = check_vector(c, "r", &D->r, 1))) return rc;
  if ((int64_t)P.size() + (int64_t)Q.size() >= kMax32)
    return c->fail(LFPSQP_ERR_ARG, "sparse QCQP: nnz(P) + nnz(Qc) must be < 2^31 (sources of the Lagrangian Hessian)");
  H.n = n; H.m = (int)m; H.r = D->r;
  H.q.assign((size_t)n, 0.0); if (D->q) std::copy(D->q, D->q + n, H.q.begin());
  H.bc.assign((size_t)m, 0.0); if (D->bc) std::copy(D->bc, D->bc + m, H.bc.begin());
  // CSR of P (f, grad)
  H.prow.assign((size_t)n + 1, 0);
  for (const Ent &e : P) { H.prow[(size_t)(e.key / n) + 1]++; H.pcol.push_back((int)(e.key % n)); H.pval.push_back(e.val); }
  for (int64_t i = 0; i < n; i++) H.prow[(size_t)i + 1] += H.prow[(size_t)i];
  // constraint segments (i, r): row r of Qc_i merged with Ac[i, r]; Q and A are sorted by (i, r, col) and (i, r)
  H.con_ptr.assign((size_t)m + 1, 0);
  H.seg_ptr.push_back(0);
  size_t kq = 0, ka = 0;
  for (int64_t i = 0; i < m; i++) {
    while ((kq < Q.size() && Q[kq].mat == i) || (ka < A.size() && A[ka].key / n == i)) {
      const int64_t rq = (kq < Q.size() && Q[kq].mat == i) ? Q[kq].key / n : n;
      const int64_t ra = (ka < A.size() && A[ka].key / n == i) ? A[ka].key % n : n;
      const int64_t r = std::min(rq, ra);
      double a = 0.0;
      if (ra == r) a = A[ka++].val;
      while (kq < Q.size() && Q[kq].mat == i && Q[kq].key / n == r) { H.seg_col.push_back((int)(Q[kq].key % n)); H.seg_val.push_back(Q[kq].val); kq++; }
      if ((int64_t)H.seg_row.size() + 1 >= kMax32) return c->fail(LFPSQP_ERR_ARG, "sparse QCQP: more than 2^31 constraint segments");
      H.seg_row.push_back((int)r); H.seg_a.push_back(a); H.seg_ptr.push_back((int)H.seg_col.size());
    }
    H.con_ptr[(size_t)i + 1] = (int)H.seg_row.size();
  }
  // union pattern of H = P + sum_i lam_i Qc_i; the sources of each entry: the P entry first, then constraints in index order
  struct Src { int64_t key; int32_t con; double val; };
  std::vector<Src> all;
  all.reserve(P.size() + Q.size());
  for (const Ent &e : P) all.push_back(Src{e.key, -1, e.val});
  for (const Ent &e : Q) all.push_back(Src{e.key, e.mat, e.val});
  std::sort(all.begin(), all.end(), [](const Src &a, const Src &b) { return a.key != b.key ? a.key < b.key : a.con < b.con; });
  H.hrow.assign((size_t)n + 1, 0);
  H.hsrc_ptr.push_back(0);
  for (size_t k = 0; k < all.size(); k++) {
    if (k == 0 || all[k].key != all[k - 1].key) {
      if (k > 0) H.hsrc_ptr.push_back((int)k);
      H.hrow[(size_t)(all[k].key / n) + 1]++;
      H.hcol.push_back((int)(all[k].key % n));
    }
    H.hsrc_con.push_back(all[k].con); H.hsrc_val.push_back(all[k].val);
  }
  if (!all.empty()) H.hsrc_ptr.push_back((int)all.size());
  for (int64_t i = 0; i < n; i++) H.hrow[(size_t)i + 1] += H.hrow[(size_t)i];
  return 0;
}

// lanes per CSR row: 4 for short rows (stencils, diagonals), a whole warp for long ones
static int lanes_for(int64_t nnz, int64_t n) { return nnz > 16 * n ? 32 : 4; }

bool spq_upload(LargeState &S, const SpqHost &H) {
  lfpsqp::SpqDev &D = S.spq;
  D.n = H.n; D.m = H.m; D.r = H.r; D.nh = (int64_t)H.hcol.size();
  D.gp = lanes_for((int64_t)H.pcol.size(), H.n); D.gh = lanes_for(D.nh, H.n);
  bool ok = upload(S, &D.q, H.q) && upload(S, &D.bc, H.bc) && upload(S, &D.prow, H.prow) && upload(S, &D.pcol, H.pcol) &&
            upload(S, &D.pval, H.pval) && upload(S, &D.hrow, H.hrow) && upload(S, &D.hcol, H.hcol) &&
            upload(S, &D.hsrc_ptr, H.hsrc_ptr) && upload(S, &D.hsrc_con, H.hsrc_con) && upload(S, &D.hsrc_val, H.hsrc_val) &&
            upload(S, &D.con_ptr, H.con_ptr) && upload(S, &D.seg_row, H.seg_row) && upload(S, &D.seg_a, H.seg_a) &&
            upload(S, &D.seg_ptr, H.seg_ptr) && upload(S, &D.seg_col, H.seg_col) && upload(S, &D.seg_val, H.seg_val);
  void *hv = nullptr;
  ok = ok && cudaMalloc(&hv, (size_t)std::max<int64_t>(D.nh, 1) * sizeof(double)) == cudaSuccess;
  if (!ok) { cudaGetLastError(); return false; }
  S.owned.push_back(hv); D.hval = (double *)hv;
  ok = cudaMemsetAsync(hv, 0, (size_t)std::max<int64_t>(D.nh, 1) * sizeof(double), S.stream) == cudaSuccess;
  // the host vectors are the caller's: the copies must have landed before it returns
  return ok && cudaStreamSynchronize(S.stream) == cudaSuccess;
}

bool spj_upload(LargeState &S, const SpqHost &H) {
  const int m = H.m;
  const int64_t n = H.n, nnz = (int64_t)H.seg_row.size();   // < 2^31: spq_build refuses more segments
  // CSC by a counting sort over the CSR order: the rows of every column come out increasing
  std::vector<int> cptr((size_t)n + 1, 0), crow((size_t)nnz), csc_of((size_t)nnz);
  for (int64_t s = 0; s < nnz; s++) cptr[(size_t)H.seg_row[(size_t)s] + 1]++;
  for (int64_t j = 0; j < n; j++) cptr[(size_t)j + 1] += cptr[(size_t)j];
  {
    std::vector<int> next(cptr.begin(), cptr.end() - 1);
    for (int i = 0; i < m; i++)
      for (int s = H.con_ptr[(size_t)i]; s < H.con_ptr[(size_t)i + 1]; s++) {
        const int p = next[(size_t)H.seg_row[(size_t)s]]++;
        crow[(size_t)p] = i; csc_of[(size_t)s] = p;
      }
  }
  // chunks of the rows longer than SPJ_CHUNK segments: a function of the pattern alone
  std::vector<int> row_slot((size_t)m + 1, 0), slot_row, slot_beg, slot_end, long_row;
  for (int i = 0; i < m; i++) {
    const int b = H.con_ptr[(size_t)i], e = H.con_ptr[(size_t)i + 1];
    if (e - b > lfpsqp::SPJ_CHUNK) {
      long_row.push_back(i);
      for (int s = b; s < e; s += lfpsqp::SPJ_CHUNK) {
        slot_row.push_back(i); slot_beg.push_back(s); slot_end.push_back((int)std::min<int64_t>((int64_t)s + lfpsqp::SPJ_CHUNK, e));
      }
    }
    row_slot[(size_t)i + 1] = (int)slot_row.size();
  }
  lfpsqp::SpjDev &P = S.spj;
  P.m = m; P.nnz = nnz; P.nslot = (int)slot_row.size(); P.nlong = (int)long_row.size();
  bool ok = upload(S, &P.cptr, cptr) && upload(S, &P.crow, crow) && upload(S, &P.csc_of, csc_of) && upload(S, &P.row_slot, row_slot) &&
            upload(S, &P.slot_row, slot_row) && upload(S, &P.slot_beg, slot_beg) && upload(S, &P.slot_end, slot_end) &&
            upload(S, &P.long_row, long_row);
  double **bufs[] = {&P.jr, &P.jc, &S.spj_part, &S.spj_gpart};
  const size_t cnt[] = {(size_t)nnz, (size_t)nnz, (size_t)P.nslot, (size_t)P.nslot * (size_t)m};
  for (int k = 0; ok && k < 4; k++) {
    void *p = nullptr;
    ok = cudaMalloc(&p, std::max<size_t>(cnt[k], 1) * sizeof(double)) == cudaSuccess;
    if (ok) { S.owned.push_back(p); *bufs[k] = (double *)p; }
  }
  if (!ok) { cudaGetLastError(); return false; }
  return cudaStreamSynchronize(S.stream) == cudaSuccess;
}
