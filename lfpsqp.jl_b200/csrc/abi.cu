// abi.cu -- extern "C" entry points of liblfpsqp_b200.so (see include/lfpsqp_b200.h) and the batched-mode launcher.
#include <cuda_runtime.h>
#include <math.h>
#include <stdio.h>
#include <string.h>
#include <string>
#include <vector>
#include <algorithm>

#include "ctx.h"
#include "batched_tiny.cuh"
#include "batched_warp.cuh"
#include "launch.cuh"

using namespace lfpsqp;

int launch_batched_reg(lfpsqp_ctx *c, lfpsqp::BatchedArgs &A);  // batched_reg.cu
int solve_batched_multi(lfpsqp_ctx *c, int family, int64_t n, int64_t m, int64_t p, int64_t B, const double *fam_params,
                        int64_t fam_stride, const double *x0, const double *xl, const double *xu, const lfpsqp_params *prm,
                        double *x_out, double *obj_hist, int64_t H, int64_t *obj_len, double *lambda, lfpsqp_term *term,
                        lfpsqp_stats *stats);   // multi.cu

static_assert(sizeof(lfpsqp_params) == 160, "lfpsqp_params layout is part of the ABI");
static_assert(sizeof(lfpsqp_term) == 40, "TerminationInfo is {Int32, pad, 3 x Float64, Int64} = 40 B");
static_assert(sizeof(lfpsqp_stats) == 80, "lfpsqp_stats layout is part of the ABI");
static thread_local std::string g_create_error;

int lfpsqp_ctx::fail(int code, const char *fmt, ...) {
  char buf[512];
  va_list ap; va_start(ap, fmt); vsnprintf(buf, sizeof(buf), fmt, ap); va_end(ap);
  err = buf;
  return code;
}
int lfpsqp_ctx::cuda_fail(cudaError_t e, const char *what) {
  cudaGetLastError();
  return fail(LFPSQP_ERR_CUDA, "CUDA error in %s: %s", what, cudaGetErrorString(e));
}
void *lfpsqp_ctx::arena(int slot, size_t bytes) {
  if (slot >= (int)bufs.size()) { bufs.resize(slot + 1, nullptr); caps.resize(slot + 1, 0); }
  if (bytes == 0) bytes = 8;
  if (caps[slot] < bytes) {
    if (bufs[slot]) cudaFree(bufs[slot]);
    bufs[slot] = nullptr; caps[slot] = 0;
    size_t want = bytes + bytes / 8;
    if (cudaMalloc(&bufs[slot], want) != cudaSuccess) { cudaGetLastError(); return nullptr; }
    caps[slot] = want;
  }
  return bufs[slot];
}

extern "C" const char *lfpsqp_version(void) { return "lfpsqp_b200 0.1.0 (sm_100a)"; }

extern "C" void lfpsqp_default_params(lfpsqp_params *p) {  // src/LFPSQP.jl:57-81
  memset(p, 0, sizeof(*p));
  p->alpha = 1.0; p->beta = 0.0; p->t_beta = 0; p->s = 0.5; p->sigma = 1e-4; p->eps_c = 1e-6; p->eps_f = 1e-6;
  p->eps_x = 0.0; p->eps_kkt = 1e-6; p->eps_rank = 1e-10; p->maxiter = 10000; p->maxiter_retract = 100;
  p->maxiter_pcg = 100; p->mu0 = 1e-2; p->disable_linesearch = 0; p->do_project_retract = 1; p->disp = 1;
  p->linesearch = 0; p->do_newton = 1; p->tn_maxiter = 10000; p->tn_kappa = 0.5; p->callback_period = 100;
}

extern "C" int lfpsqp_ctx_create(int device, lfpsqp_ctx **out) {
  *out = nullptr;
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev == 0) {
    cudaGetLastError();
    g_create_error = std::string("lfpsqp_ctx_create: no CUDA device (") + cudaGetErrorString(e) +
                     "); this library has no CPU fallback";
    return LFPSQP_ERR_CUDA;
  }
  if (device < 0 || device >= ndev) { g_create_error = "lfpsqp_ctx_create: bad device index"; return LFPSQP_ERR_ARG; }
  cudaSetDevice(device);
  lfpsqp_ctx *c = new lfpsqp_ctx();
  c->device = device;
  cudaDeviceProp prop;
  cudaGetDeviceProperties(&prop, device);
  c->sm_count = prop.multiProcessorCount;
  c->smem_optin = (int)prop.sharedMemPerBlockOptin;
  if (prop.major < 10) {
    g_create_error = "lfpsqp_ctx_create: device is not sm_100 (Blackwell); this build carries sm_100a code only";
    delete c; return LFPSQP_ERR_CUDA;
  }
  if (cudaStreamCreateWithFlags(&c->own_stream, cudaStreamNonBlocking) != cudaSuccess ||
      cudaEventCreate(&c->ev0) != cudaSuccess || cudaEventCreate(&c->ev1) != cudaSuccess ||
      cudaMalloc(&c->work_counter, 256) != cudaSuccess) {
    g_create_error = "lfpsqp_ctx_create: stream/event creation failed";
    delete c; cudaGetLastError(); return LFPSQP_ERR_CUDA;
  }
  c->stream = c->own_stream;
  *out = c;
  return LFPSQP_OK;
}

extern "C" void lfpsqp_ctx_destroy(lfpsqp_ctx *c) {
  if (!c) return;
  for (lfpsqp_ctx *ch : c->children) lfpsqp_ctx_destroy(ch);
  c->children.clear();
  cudaSetDevice(c->device);
  lfpsqp_large_release(c);
  lfpsqp_comm_destroy(c);
  for (void *b : c->bufs) if (b) cudaFree(b);
  if (c->work_counter) cudaFree(c->work_counter);
  for (int i = 0; i < 3; i++) if (c->pipe[i]) cudaStreamDestroy(c->pipe[i]);
  if (c->ev0) cudaEventDestroy(c->ev0);
  if (c->ev1) cudaEventDestroy(c->ev1);
  if (c->own_stream) cudaStreamDestroy(c->own_stream);
  delete c;
}

extern "C" const char *lfpsqp_last_error(lfpsqp_ctx *c) { return c ? c->err.c_str() : g_create_error.c_str(); }

extern "C" int lfpsqp_ctx_set_stream(lfpsqp_ctx *c, void *s) {
  if (!c) return LFPSQP_ERR_ARG;
  c->stream = s ? (cudaStream_t)s : c->own_stream;
  return LFPSQP_OK;
}
extern "C" int lfpsqp_ctx_set_noise(lfpsqp_ctx *c, const double *noise, int64_t T, int64_t N, int64_t B) {
  if (!c) return LFPSQP_ERR_ARG;
  if (noise && (T < 1 || N < 1 || B < 1)) return c->fail(LFPSQP_ERR_ARG, "lfpsqp_ctx_set_noise: bad sizes");
  c->noise_host = noise; c->noise_T = noise ? T : 0; c->noise_N = noise ? N : 0; c->noise_B = noise ? B : 0;
  return LFPSQP_OK;
}
extern "C" double lfpsqp_last_kernel_ms(lfpsqp_ctx *c) { return c ? c->last_ms : -1.0; }
extern "C" int64_t lfpsqp_last_launches(lfpsqp_ctx *c) { return c ? c->last_launches : 0; }
extern "C" int lfpsqp_last_kernel(lfpsqp_ctx *c, int *out4) {
  if (!c || !out4) return LFPSQP_ERR_ARG;
  memcpy(out4, c->last_kernel, sizeof(c->last_kernel));
  return LFPSQP_OK;
}

// ------------------------------------------------------------------ family registry
namespace {

int64_t fam_param_count(int family, int64_t n, int64_t m, int64_t p) {
  (void)p;
  switch (family) {
    case LFPSQP_FAM_README_INEQ: return n;
    case LFPSQP_FAM_DIAGQUAD: return 2 * m * n + m + 2 * n;
    case LFPSQP_FAM_SIN: return n;
    case LFPSQP_FAM_BOXQUAD: return 2 * n + 1;
    default: return 0;
  }
}

bool fam_valid(int family, int64_t n, int64_t m, int64_t p) {
  switch (family) {
    case LFPSQP_FAM_ROSENBROCK: return FamRosenbrock::valid(n, m, p);
    case LFPSQP_FAM_README_EQ: return FamReadmeEq::valid(n, m, p);
    case LFPSQP_FAM_README_INEQ: return FamReadmeIneq::valid(n, m, p);
    case LFPSQP_FAM_THOMSON: return FamThomson::valid(n, m, p);
    case LFPSQP_FAM_DIAGQUAD: return FamDiagQuad::valid(n, m, p);
    case LFPSQP_FAM_SIN: return FamSin::valid(n, m, p);
    case LFPSQP_FAM_BOXQUAD: return FamBoxQuad::valid(n, m, p);
    case LFPSQP_FAM_QCQP: return FamQCQP::valid(n, m, p);
    default: return false;
  }
}

// lfpsqp_qcqp viewed as its nine {pointer, batch stride} pairs, in declaration order
struct QcqpField { const double *ptr; int64_t stride; };
static_assert(sizeof(lfpsqp_qcqp) == 9 * sizeof(QcqpField), "lfpsqp_qcqp is nine {pointer, stride} pairs");
const char *const kQcqpNames[9] = {"P", "q", "r", "Qc", "Ac", "bc", "Qd", "Ad", "bd"};

// element count of each array and how many n x n matrices it stacks
void qcqp_counts(int64_t n, int64_t m, int64_t p, int64_t cnt[9], int64_t nmat[9]) {
  const int64_t c[9] = {n * n, n, 1, m * n * n, m * n, m, p * n * n, p * n, p}, k[9] = {1, 0, 0, m, 0, 0, p, 0, 0};
  for (int i = 0; i < 9; i++) { cnt[i] = c[i]; nmat[i] = k[i]; }
}

// Argument checks of the QCQP descriptor shared by both entry points.  out = the descriptor with the arrays of
// zero elements (Qc when m = 0, ...) set to NULL, so that nothing downstream reads them.
int qcqp_check(lfpsqp_ctx *c, const double *fam_params, int64_t fam_stride, int64_t n, int64_t m, int64_t p,
               lfpsqp_qcqp &out) {
  if (!fam_params) return c->fail(LFPSQP_ERR_ARG, "LFPSQP_FAM_QCQP: fam_params must point to a lfpsqp_qcqp descriptor");
  if (fam_stride != 0) return c->fail(LFPSQP_ERR_ARG, "LFPSQP_FAM_QCQP: fam_stride must be 0 (each array has its own stride)");
  out = *(const lfpsqp_qcqp *)fam_params;
  QcqpField *F = (QcqpField *)&out;
  int64_t cnt[9], nmat[9];
  qcqp_counts(n, m, p, cnt, nmat);
  for (int i = 0; i < 9; i++) {
    if (cnt[i] == 0) { F[i].ptr = nullptr; F[i].stride = 0; continue; }
    if (F[i].ptr && (F[i].stride < 0 || (F[i].stride != 0 && F[i].stride < cnt[i])))
      return c->fail(LFPSQP_ERR_ARG, "LFPSQP_FAM_QCQP: %s_stride = %lld; it must be 0 (shared) or >= %lld", kQcqpNames[i],
                     (long long)F[i].stride, (long long)cnt[i]);
  }
  if (m > 0 && !out.Qc && !out.Ac) return c->fail(LFPSQP_ERR_ARG, "LFPSQP_FAM_QCQP: m > 0 needs Qc or Ac");
  if (p > 0 && !out.Qd && !out.Ad) return c->fail(LFPSQP_ERR_ARG, "LFPSQP_FAM_QCQP: p > 0 needs Qd or Ad");
  return LFPSQP_OK;
}

// exact symmetry of every n x n matrix the host entry point stages (instances [0, B) of a per-instance array)
int qcqp_check_symmetric(lfpsqp_ctx *c, const lfpsqp_qcqp &qp, int64_t n, int64_t m, int64_t p, int64_t B) {
  const QcqpField *F = (const QcqpField *)&qp;
  int64_t cnt[9], nmat[9];
  qcqp_counts(n, m, p, cnt, nmat);
  for (int i = 0; i < 9; i++) {
    if (!F[i].ptr || nmat[i] == 0) continue;
    const int64_t copies = F[i].stride ? B : 1;
    for (int64_t k = 0; k < copies; k++)
      for (int64_t t = 0; t < nmat[i]; t++) {
        const double *M = F[i].ptr + k * F[i].stride + t * n * n;
        for (int64_t a = 1; a < n; a++)
          for (int64_t b = 0; b < a; b++)
            if (!(M[a * n + b] == M[b * n + a]))
              return c->fail(LFPSQP_ERR_ARG, "LFPSQP_FAM_QCQP: %s is not symmetric (instance %lld, matrix %lld, entry %lld,%lld)",
                             kQcqpNames[i], (long long)k, (long long)t, (long long)a, (long long)b);
      }
  }
  return LFPSQP_OK;
}

// InequalityData (src/inequality_helper.jl:39-85) for the slack-augmented bound vectors (optimize.jl:30-36).
// Layout: [kind | q | r | s | t], each NA doubles.  Returns ineq (optimize.jl:151), or <0 on bound errors.
int build_bounds(int64_t n, int64_t p, const double *xl, const double *xu, std::vector<double> &bnd) {
  const int64_t NA = n + p;
  bool ineq = p > 0;  // du = 0 is finite => the bounds branch is always active on the d! path (SURVEY A.2)
  if (xl && xu) {
    bool alll = true, allu = true;
    for (int64_t i = 0; i < n; i++) {
      if (!(xl[i] == -INFINITY)) alll = false;
      if (!(xu[i] == INFINITY)) allu = false;
      if (xl[i] > xu[i]) return LFPSQP_ERR_BOUNDS;
    }
    if (!(alll && allu)) ineq = true;
  } else if (xl || xu) return LFPSQP_ERR_ARG;
  if (!ineq) return 0;
  bnd.assign(5 * NA, 0.0);
  double *kind = bnd.data(), *q = kind + NA, *r = q + NA, *s = r + NA, *t = s + NA;
  for (int64_t i = 0; i < NA; i++) {
    double lo = (i < n) ? (xl ? xl[i] : -INFINITY) : -INFINITY;
    double hi = (i < n) ? (xu ? xu[i] : INFINITY) : 0.0;
    bool linf = isinf(lo), uinf = isinf(hi);
    if (linf && uinf) { kind[i] = 0; }
    else if (!linf && uinf) { kind[i] = 1; q[i] = 0; r[i] = lo; s[i] = -1.0; t[i] = lo; }
    else if (linf && !uinf) { kind[i] = 1; q[i] = 0; r[i] = hi; s[i] = 1.0; t[i] = hi; }
    else { kind[i] = 2; q[i] = 1.0; r[i] = (hi + lo) / 2; s[i] = 1.0; t[i] = (hi - lo) * (hi - lo) / 4; }
  }
  return 1;
}

template <class Fam>
int launch_warp(lfpsqp_ctx *c, BatchedArgs &A, int use_nr) {
  WarpLayout L(A.n, A.m, A.p, A.ineq, use_nr, (A.prm.linesearch != 0 && !A.prm.disable_linesearch) ? 1 : 0);
  const size_t bnd_bytes = (size_t)(((A.ineq ? 5 * L.NA : 0) + 1) & ~1) * 8;
  const size_t per_warp = (size_t)L.total * 8;
  const size_t cap = (size_t)c->smem_optin;
  if (bnd_bytes + per_warp > cap)
    return c->fail(LFPSQP_ERR_NOMEM,
                   "batched mode: one instance needs %zu B of shared memory (> %zu); use lfpsqp_solve_large",
                   bnd_bytes + per_warp, cap);
  int maxw = (int)((cap - bnd_bytes) / per_warp);
  if (maxw > 8) maxw = 8;
  auto kern = batched_warp_kernel<Fam>;
  cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(bnd_bytes + maxw * per_warp));
  if (e != cudaSuccess) return c->cuda_fail(e, "cudaFuncSetAttribute");
  // pick the CTA width that keeps the most warps resident per SM (shared memory AND registers, via the occupancy API)
  int warps = maxw, resident = 0, best = 0;
  for (int w = maxw; w >= 1; w--) {
    int r = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&r, kern, w * 32, bnd_bytes + w * per_warp) != cudaSuccess) { cudaGetLastError(); continue; }
    if (r * w > best) { best = r * w; warps = w; resident = r; }
  }
  if (resident < 1) return c->fail(LFPSQP_ERR_CUDA, "batched_warp_kernel cannot be made resident");
  const size_t smem = bnd_bytes + warps * per_warp;
  const int64_t grid = persistent_grid(c, A, resident, warps);
  return launch_batched_kernel(c, kern, grid, warps * 32, smem, {1, 32, 0, 0}, "batched_warp_kernel launch", A, use_nr);
}

template <class Fam, int NT>
int launch_tiny(lfpsqp_ctx *c, BatchedArgs &A) {   // one thread per instance, not persistent
  const int threads = 128;
  return launch_batched_kernel(c, batched_tiny_kernel<Fam, NT>, (A.B + threads - 1) / threads, threads, 0, {0, 1, 0, 0},
                               "batched_tiny_kernel launch", A);
}

int dispatch_batched(lfpsqp_ctx *c, BatchedArgs &A) {
  const int use_nr = A.prm.do_project_retract ? 0 : 1;
  {  // separable families with a register-resident instantiation (batched_reg.cuh)
    int rc = launch_batched_reg(c, A);
    if (rc <= 0) return rc;
  }
  switch (A.family) {
    case LFPSQP_FAM_ROSENBROCK:
      if (!A.ineq && !(A.prm.linesearch != 0 && !A.prm.disable_linesearch)) return launch_tiny<FamRosenbrock, 2>(c, A);
      return launch_warp<FamRosenbrock>(c, A, use_nr);
    case LFPSQP_FAM_README_EQ: return launch_warp<FamReadmeEq>(c, A, use_nr);
    case LFPSQP_FAM_README_INEQ: return launch_warp<FamReadmeIneq>(c, A, use_nr);
    case LFPSQP_FAM_THOMSON: return launch_warp<FamThomson>(c, A, use_nr);
    case LFPSQP_FAM_DIAGQUAD: return launch_warp<FamDiagQuad>(c, A, use_nr);
    case LFPSQP_FAM_SIN: return launch_warp<FamSin>(c, A, use_nr);
    case LFPSQP_FAM_BOXQUAD: return launch_warp<FamBoxQuad>(c, A, use_nr);
    case LFPSQP_FAM_QCQP: return launch_warp<FamQCQP>(c, A, use_nr);   // not separable: no register-resident solver
    default: return c->fail(LFPSQP_ERR_FAMILY, "unknown family %d", A.family);
  }
}

int check_common(lfpsqp_ctx *c, int family, int64_t n, int64_t m, int64_t p, int64_t B, const lfpsqp_params *prm,
                 int64_t H) {
  if (!c) return LFPSQP_ERR_ARG;
  if (!prm) return c->fail(LFPSQP_ERR_ARG, "params is NULL");
  if (n < 1 || m < 0 || p < 0 || B < 0 || H < 1) return c->fail(LFPSQP_ERR_ARG, "bad sizes n=%lld m=%lld p=%lld B=%lld H=%lld",
                                                                  (long long)n, (long long)m, (long long)p, (long long)B, (long long)H);
  if (n > (1 << 24)) return c->fail(LFPSQP_ERR_ARG, "n too large");
  if (!fam_valid(family, n, m, p)) return c->fail(LFPSQP_ERR_FAMILY, "family %d does not support n=%lld m=%lld p=%lld", family,
                                                  (long long)n, (long long)m, (long long)p);
  if (prm->beta > 0) {
    if (!c->noise_host) return c->fail(LFPSQP_ERR_UNSUPPORTED, "beta>0 (stochastic perturbation, optimize.jl:264-273) needs the caller's noise "
                                                               "sequence: lfpsqp_ctx_set_noise (device families) or the randn callback (lfpsqp_solve_host)");
    if (c->noise_B != B || c->noise_T < 1) return c->fail(LFPSQP_ERR_ARG, "lfpsqp_ctx_set_noise: noise was supplied for %lld instances, the batch has %lld",
                                                           (long long)c->noise_B, (long long)B);
  }
  return LFPSQP_OK;
}

}  // namespace

int build_bounds_public(int64_t n, int64_t p, const double *xl, const double *xu, std::vector<double> &bnd) { return build_bounds(n, p, xl, xu, bnd); }

// argument checks + bound embedding data shared by both batched entry points; fills A except the per-batch pointers
static int prepare_batched(lfpsqp_ctx *c, int family, int64_t n, int64_t m, int64_t p, int64_t B, const double *xl,
                           const double *xu, const lfpsqp_params *prm, int64_t H, BatchedArgs &A) {
  int rc = check_common(c, family, n, m, p, B, prm, H);
  if (rc) return rc;
  c->last_kernel[0] = -1; c->last_kernel[1] = c->last_kernel[2] = c->last_kernel[3] = 0;
  cudaSetDevice(c->device);
  std::vector<double> &bnd = c->bnd_host;   // kept for the launcher (kernel selection looks at the bound kinds)
  bnd.clear();
  int ineq = build_bounds(n, p, xl, xu, bnd);
  if (ineq == LFPSQP_ERR_BOUNDS) return c->fail(ineq, "Infeasible: lower bounds cannot be greater than upper bounds");
  if (ineq < 0) return c->fail(ineq, "xl, xu, and x0 must all be the same length (both or neither may be NULL)");
  memset(&A, 0, sizeof(A));
  A.family = family; A.n = (int)n; A.m = (int)m; A.p = (int)p; A.ineq = ineq; A.B = B; A.prm = *prm; A.H = H;
  if (prm->beta > 0) {
    const int64_t Nw = (ineq ? 2 : 1) * (n + p);      // the working dimension the reference draws randn! for (optimize.jl:172, :265)
    if (c->noise_N != Nw) return c->fail(LFPSQP_ERR_ARG, "lfpsqp_ctx_set_noise: rows of %lld entries, the working dimension is %lld", (long long)c->noise_N, (long long)Nw);
  }
  if (ineq && B > 0) {
    double *dbnd = (double *)c->arena(0, bnd.size() * 8);
    if (!dbnd) return c->fail(LFPSQP_ERR_NOMEM, "device allocation failed");
    cudaMemcpyAsync(dbnd, bnd.data(), bnd.size() * 8, cudaMemcpyHostToDevice, c->stream);
    A.bnd = dbnd;
  }
  return LFPSQP_OK;
}

extern "C" int lfpsqp_solve_batched_dev(lfpsqp_ctx *c, int family, int64_t n, int64_t m, int64_t p, int64_t B,
                                        const double *fam_params_dev, int64_t fam_stride, const double *x0_dev,
                                        const double *xl, const double *xu, const lfpsqp_params *prm, double *x_out_dev,
                                        double *obj_hist_dev, int64_t H, int64_t *obj_len_dev, double *lambda_dev,
                                        lfpsqp_term *term_dev, lfpsqp_stats *stats_dev) {
  BatchedArgs A;
  int rc = prepare_batched(c, family, n, m, p, B, xl, xu, prm, H, A);
  if (rc) return rc;
  c->last_ms = 0; c->last_launches = 0;
  if (family == LFPSQP_FAM_QCQP) {   // descriptor in host memory, arrays in device memory (symmetry is a precondition)
    rc = qcqp_check(c, fam_params_dev, fam_stride, n, m, p, A.qcqp);
    if (rc) return rc;
    fam_params_dev = nullptr;
  }
  if (B == 0) return LFPSQP_OK;
  if (fam_param_count(family, n, m, p) > 0 && !fam_params_dev) return c->fail(LFPSQP_ERR_ARG, "family needs a parameter blob");
  A.fam_params = fam_params_dev; A.fam_stride = fam_stride; A.x0 = x0_dev;
  A.x_out = x_out_dev; A.obj_hist = obj_hist_dev; A.obj_len = obj_len_dev; A.lambda = lambda_dev;
  A.term = term_dev; A.stats = stats_dev;
  if (prm->beta > 0) {
    const size_t nb = (size_t)c->noise_B * c->noise_T * c->noise_N * 8;
    double *d_noise = (double *)c->arena(9, nb);
    if (!d_noise) return c->fail(LFPSQP_ERR_NOMEM, "device allocation failed");
    cudaMemcpyAsync(d_noise, c->noise_host, nb, cudaMemcpyHostToDevice, c->stream);
    A.noise = d_noise; A.noise_T = c->noise_T;
  }
  cudaMemsetAsync(obj_hist_dev, 0xff, (size_t)H * B * 8, c->stream);   // NaN-fill the unused tail of the history, as the host entry does
  rc = dispatch_batched(c, A);
  if (rc) return rc;
  cudaError_t e = cudaStreamSynchronize(c->stream);
  if (e != cudaSuccess) return c->cuda_fail(e, "batched solve");
  float ms = 0; cudaEventElapsedTime(&ms, c->ev0, c->ev1);
  c->last_ms = ms;
  return LFPSQP_OK;
}

// Host-buffer entry point.  Large batches are cut into chunks that flow through a 3-stream pipeline
// (H2D of chunk i+1 and D2H of chunk i-1 overlap the kernel of chunk i; needs pinned host buffers to really overlap).
extern "C" int lfpsqp_solve_batched(lfpsqp_ctx *c, int family, int64_t n, int64_t m, int64_t p, int64_t B,
                                    const double *fam_params, int64_t fam_stride, const double *x0, const double *xl,
                                    const double *xu, const lfpsqp_params *prm, double *x_out, double *obj_hist,
                                    int64_t H, int64_t *obj_len, double *lambda, lfpsqp_term *term, lfpsqp_stats *stats) {
  if (c && !c->children.empty())   // multi-GPU ctx: contiguous instance ranges per device, one host thread each (multi.cu)
    return solve_batched_multi(c, family, n, m, p, B, fam_params, fam_stride, x0, xl, xu, prm, x_out, obj_hist, H, obj_len, lambda, term, stats);
  BatchedArgs A0;
  int rc = prepare_batched(c, family, n, m, p, B, xl, xu, prm, H, A0);
  if (rc) return rc;
  // QCQP: host arrays of the descriptor; qf = the device copies (arena slots 10..18, same batch strides as the caller's)
  lfpsqp_qcqp qh{}, qd{};
  QcqpField *qf = (QcqpField *)&qd;
  const QcqpField *hf = (const QcqpField *)&qh;
  int64_t qcnt[9] = {0}, qmat[9];
  if (family == LFPSQP_FAM_QCQP) {
    rc = qcqp_check(c, fam_params, fam_stride, n, m, p, qh);
    if (rc) return rc;
    rc = qcqp_check_symmetric(c, qh, n, m, p, B);
    if (rc) return rc;
    fam_params = nullptr;
    qcqp_counts(n, m, p, qcnt, qmat);
  }
  if (B == 0) return LFPSQP_OK;
  for (int i = 0; i < 9; i++) {
    if (!hf[i].ptr) continue;
    const int64_t elems = hf[i].stride ? (B - 1) * hf[i].stride + qcnt[i] : qcnt[i];   // never reads past the last instance
    qf[i].ptr = (const double *)c->arena(10 + i, (size_t)elems * 8);
    qf[i].stride = hf[i].stride;
    if (!qf[i].ptr) return c->fail(LFPSQP_ERR_NOMEM, "device allocation failed");
  }
  const int64_t npar = fam_param_count(family, n, m, p);
  if (npar > 0 && !fam_params) return c->fail(LFPSQP_ERR_ARG, "family needs a parameter blob");
  if (npar > 0 && fam_stride != 0 && fam_stride < npar) return c->fail(LFPSQP_ERR_ARG, "fam_stride smaller than the family's blob");
  const size_t par_bytes = npar ? (size_t)(fam_stride ? fam_stride * B : npar) * 8 : 0;
  const int64_t ME = m + p;
  double *d_par = (double *)c->arena(1, par_bytes), *d_x0 = (double *)c->arena(2, (size_t)n * B * 8),
         *d_x = (double *)c->arena(3, (size_t)n * B * 8), *d_obj = (double *)c->arena(4, (size_t)H * B * 8),
         *d_lam = (double *)c->arena(6, (size_t)ME * B * 8);
  int64_t *d_len = (int64_t *)c->arena(5, (size_t)B * 8);
  lfpsqp_term *d_term = (lfpsqp_term *)c->arena(7, (size_t)B * sizeof(lfpsqp_term));
  lfpsqp_stats *d_stats = stats ? (lfpsqp_stats *)c->arena(8, (size_t)B * sizeof(lfpsqp_stats)) : nullptr;
  const size_t noise_row = (prm->beta > 0) ? (size_t)c->noise_T * c->noise_N : 0;    // doubles per instance
  double *d_noise = noise_row ? (double *)c->arena(9, noise_row * B * 8) : nullptr;
  if (!d_par || !d_x0 || !d_x || !d_obj || !d_lam || !d_len || !d_term || (stats && !d_stats) || (noise_row && !d_noise))
    return c->fail(LFPSQP_ERR_NOMEM, "device allocation failed");
  // chunking: keep every chunk big enough to fill the GPU several times over.  The first chunk's H2D and the last chunk's
  // D2H are the only copies the kernels cannot hide, so those two chunks are half the size of the others (measured at C2,
  // 65,536 instances: 8 equal chunks 2.050 ms, halved ends 2.009 ms, 16 chunks 2.06-2.09 ms, 4 chunks 2.24 ms;
  // device-resident kernel 1.74 ms).  Chunks cut in whole rounds of the persistent kernels (resident CTAs x instances per
  // CTA) measured slower (2.11 ms): a partly filled last round costs nothing, because the idle CTAs exit and the next
  // chunk's CTAs take their place, while whole rounds end all CTAs at once and expose the launch gap.
  int nchunk = 1;
  if (B >= 16384) nchunk = (int)std::min<int64_t>(8, B / 8192);
  const int NS = 3;
  if (nchunk > 1 && !c->pipe[0]) {
    for (int i = 0; i < NS; i++) if (cudaStreamCreateWithFlags(&c->pipe[i], cudaStreamNonBlocking) != cudaSuccess) { cudaGetLastError(); nchunk = 1; break; }
  }
  // chunk ci = instances [cut[ci], cut[ci + 1]); chunk sizes in the ratio 1/2 : 1 : ... : 1 : 1/2 (two halves when nchunk = 2)
  std::vector<int64_t> cut(nchunk + 1, B);
  cut[0] = 0;
  for (int ci = 1; ci < nchunk; ci++) cut[ci] = (int64_t)(B * ((ci - 0.5) / (nchunk - 1)) + 0.5);
  cudaStream_t user_stream = c->stream;
  unsigned long long *counter0 = c->work_counter;
  if (nchunk > 1) cudaStreamSynchronize(user_stream);   // earlier work on the caller's stream is done before the pipeline starts
  if (npar && fam_stride == 0) cudaMemcpyAsync(d_par, fam_params, par_bytes, cudaMemcpyHostToDevice, user_stream), cudaStreamSynchronize(user_stream);
  {  // QCQP arrays shared by the batch: copied once, before any chunk's kernel
    bool any = false;
    for (int i = 0; i < 9; i++)
      if (hf[i].ptr && !hf[i].stride) { cudaMemcpyAsync((void *)qf[i].ptr, hf[i].ptr, (size_t)qcnt[i] * 8, cudaMemcpyHostToDevice, user_stream); any = true; }
    if (any) cudaStreamSynchronize(user_stream);
  }
  c->last_launches = 0;
  int64_t launches = 0;
  for (int ci = 0; ci < nchunk && rc == 0; ci++) {
    const int64_t lo = cut[ci], hi = cut[ci + 1], nb = hi - lo;
    cudaStream_t s = (nchunk > 1) ? c->pipe[ci % NS] : user_stream;
    if (npar && fam_stride) cudaMemcpyAsync(d_par + lo * fam_stride, fam_params + lo * fam_stride, (size_t)nb * fam_stride * 8, cudaMemcpyHostToDevice, s);
    cudaMemcpyAsync(d_x0 + lo * n, x0 + lo * n, (size_t)n * nb * 8, cudaMemcpyHostToDevice, s);
    cudaMemsetAsync(d_obj + lo * H, 0xff, (size_t)H * nb * 8, s);  // NaN-fill the unused tail of the history
    BatchedArgs A = A0;
    A.B = nb;
    QcqpField *af = (QcqpField *)&A.qcqp;
    for (int i = 0; i < 9; i++) {
      af[i] = qf[i];
      if (!hf[i].ptr || !hf[i].stride) continue;
      const int64_t off = lo * hf[i].stride;   // per-instance array: this chunk's instances, rebased to the chunk
      cudaMemcpyAsync((void *)(qf[i].ptr + off), hf[i].ptr + off, (size_t)((nb - 1) * hf[i].stride + qcnt[i]) * 8, cudaMemcpyHostToDevice, s);
      af[i].ptr = qf[i].ptr + off;
    }
    if (noise_row) {
      cudaMemcpyAsync(d_noise + lo * noise_row, c->noise_host + lo * noise_row, noise_row * nb * 8, cudaMemcpyHostToDevice, s);
      A.noise = d_noise + lo * noise_row; A.noise_T = c->noise_T;
    }
    A.fam_params = npar ? (fam_stride ? d_par + lo * fam_stride : d_par) : nullptr; A.fam_stride = fam_stride;
    A.x0 = d_x0 + lo * n; A.x_out = d_x + lo * n; A.obj_hist = d_obj + lo * H; A.obj_len = d_len + lo;
    A.lambda = d_lam + lo * ME; A.term = d_term + lo; A.stats = d_stats ? d_stats + lo : nullptr;
    c->stream = s; c->work_counter = counter0 + (ci % 32);   // 256 B = 32 counters: one per chunk in flight
    rc = dispatch_batched(c, A);
    launches += c->last_launches;
    if (rc) break;
    cudaMemcpyAsync(x_out + lo * n, d_x + lo * n, (size_t)n * nb * 8, cudaMemcpyDeviceToHost, s);
    cudaMemcpyAsync(obj_hist + lo * H, d_obj + lo * H, (size_t)H * nb * 8, cudaMemcpyDeviceToHost, s);
    cudaMemcpyAsync(obj_len + lo, d_len + lo, (size_t)nb * 8, cudaMemcpyDeviceToHost, s);
    if (ME) cudaMemcpyAsync(lambda + lo * ME, d_lam + lo * ME, (size_t)ME * nb * 8, cudaMemcpyDeviceToHost, s);
    cudaMemcpyAsync(term + lo, d_term + lo, (size_t)nb * sizeof(lfpsqp_term), cudaMemcpyDeviceToHost, s);
    if (stats) cudaMemcpyAsync(stats + lo, d_stats + lo, (size_t)nb * sizeof(lfpsqp_stats), cudaMemcpyDeviceToHost, s);
  }
  c->stream = user_stream; c->work_counter = counter0;
  c->last_launches = launches;
  cudaError_t e = cudaSuccess;
  if (nchunk > 1) { for (int i = 0; i < NS; i++) { cudaError_t ei = cudaStreamSynchronize(c->pipe[i]); if (ei != cudaSuccess) e = ei; } }
  else e = cudaStreamSynchronize(user_stream);
  if (rc) return rc;
  if (e != cudaSuccess) return c->cuda_fail(e, "batched solve (pipeline)");
  return LFPSQP_OK;
}
