// large_fused.cu -- persistent, grid-synchronised projcg! (src/projcg.jl:71-112) and pcg! (src/retractions.jl:179-246)
// for the large-n mode, with the cross-GPU all-reduces of the column-sharded mode done inside the kernels.
//
// The unfused path (large.cu::projcg) spends 8 dependent launches per CG iteration (11 with the cross-GPU all-reduces);
// at C5 that is ~25 us of launch/drain gaps on top of 334 us of HBM time, and at 8 GPUs (41 us of HBM time per
// iteration) the gaps dominate.  Here ONE cooperative kernel (one CTA per SM, 512 threads) runs a whole chunk of
// iterations; the data dependencies between the phases of an iteration are grid barriers (cooperative launch, one
// release-add / acquire-spin counter), the CG
// scalars are re-reduced redundantly by every CTA from per-CTA partials in a fixed order (bitwise identical on every
// CTA => control flow stays grid-uniform), and projcg's exits (negative curvature, rg <= 0, ||g|| < tol, iteration
// cap) are taken on the device exactly as in the unfused kernels.
//
// Phases of iteration k (B = grid barrier):
//   P1  Ad = H d (diagonal Lagrangian Hessian: hd .* d), partial d.Ad            [owned columns]
//   B   alpha = rg / d.Ad ; x += alpha d ; rp = r + alpha Ad                      [owned columns]       (projcg.jl:74-93)
//   B   t = J rp                                                                  [owned rows, whole rows streamed]  (:96)
//   B   u = G^-1 t  (explicit G^-1 = L^-T L^-1, one m x m pass)                    [owned rows]
//   B   gp = rp - J' u ; partials rp.gp, gp.gp                                    [owned columns, all m rows streamed] (:97-99)
//   B   beta = rp.gp / rg ; d = beta d - gp ; r = gp ; convergence tests          [owned columns]       (:98-111)
// Algorithmic HBM bytes per iteration are those of the unfused path (16 m N + 8 m^2 + ~100 N); J is streamed with
// 128-bit ld.global.nc.L1::no_allocate loads, vectors written inside the kernel are only read with coherent loads.
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>

#include "large_device.cuh"
#include "large_state.h"

using namespace lfpsqp;

namespace {

constexpr int FT = 512;      // threads per CTA
constexpr int TR = 16;       // rows per sweep of the triangular phases
constexpr int CU = 16;       // 128-bit loads in flight per thread in the streaming phases
constexpr int RCH = 2048;    // column pairs per shared-memory chunk of rp in the row phase (2 buffers x 32 KB)
constexpr size_t SMEM_MAX = 220 * 1024;   // dynamic shared memory opted in for every fused kernel (larger m: not eligible)

struct FusedArgs {
  int64_t n, ldj, ldm;       // local columns (even), leading dimensions
  int m;
  const double *J, *Ginv, *hd, *Linv, *XT;
  double *xs, *dc, *r, *Ad, *rp, *gp, *tm, *tu, *ty;
  int *abort_flag;           // column-sharded: raised by a CTA whose peer-memory exchange timed out (see GridBar)
  double *part;              // 3 x gridDim partials: d.Ad | rp.gp | gp.gp
  const double *lp_rg;       // first chunk: partials of r.r from cg_init (loop slot 3)
  int np_rg, first, max_iters;
  LargeCtrl *ctrl;
  double *prof;              // nullptr, or 8 doubles: ns per phase summed over the chunk (debug)
  // column-sharded mode (world > 1): the exported peer regions (push mailboxes, large_ctrl.h FZ_*), this rank, and the
  // device-resident exchange counter (same sequence on every rank: the CG scalars are bitwise identical everywhere)
  double *peer[PC_RANKS];
  int rank, world;
  unsigned long long *epoch;
  unsigned *bar;             // grid-barrier arrival counter
  // zero-slab map of J (large_gemm.cuh::zero_slab_map_kernel: 64 rows x 16 columns per byte) for the SKIP instantiation of the
  // pcg! kernel: loads of all-zero slabs are not issued (same threads, same order: bit-identical to the dense streaming)
  const unsigned char *nz = nullptr;
  int64_t nz_ld = 0;
};

// ---- in-kernel all-reduce over NVLink: push model with flag-in-data mailboxes (the "LL" idea: every 16-byte entry
// carries {value, exchange number} and is written with ONE 128-bit store, which the fabric delivers atomically; the
// consumer spins on the entry itself).  No fence, no separate flag, no extra grid barrier: an exchange costs one
// one-way NVLink latency.  Every rank (including the sender itself) receives a copy in its own region, so consumers
// only read local memory; sums are taken in rank order => bitwise identical on every rank and CTA.
// Reuse is safe without double buffering: a rank overwrites its entries of kind K only after it has consumed a later
// exchange from every peer, and a peer sends that later exchange only behind a grid barrier that follows all of its
// reads of kind K.
struct __align__(16) LLEntry { unsigned long long w0, w1; };   // {lo32(value) | e32 << 32}, {hi32(value) | e32 << 32}
__device__ __forceinline__ void ll_store(LLEntry *p, double v, unsigned long long e) {
  const unsigned long long b = (unsigned long long)__double_as_longlong(v), f = (e & 0xffffffffULL) << 32;
  asm volatile("st.relaxed.sys.global.v2.b64 [%0], {%1, %2};" ::"l"(p), "l"((b & 0xffffffffULL) | f), "l"((b >> 32) | f) : "memory");
}
// one poll: true when both words carry the same exchange number >= e (32-bit wrap-around compare)
__device__ __forceinline__ bool ll_try(const LLEntry *p, unsigned long long e, double &v) {
  unsigned long long a, b;
  asm volatile("ld.relaxed.sys.global.v2.b64 {%0, %1}, [%2];" : "=l"(a), "=l"(b) : "l"(p) : "memory");
  const unsigned fa = (unsigned)(a >> 32), fb = (unsigned)(b >> 32);
  if (fa == fb && (int)(fa - (unsigned)e) >= 0) { v = __longlong_as_double((long long)((a & 0xffffffffULL) | (b << 32))); return true; }
  return false;
}
// spin until the entry carries exchange >= e; false after ~4 s (a peer died: do not hang the GPU)
__device__ __forceinline__ bool ll_load(const LLEntry *p, unsigned long long e, double &v) {
  const long long t0 = clock64();
  do {
    if (ll_try(p, e, v)) return true;
    __nanosleep(40);
  } while (clock64() - t0 < 8000000000LL);
  v = 0.0;
  return false;
}
// raw poll of one entry (no retry): the two words and whether they validate for exchange e
__device__ __forceinline__ void ll_raw(const LLEntry *p, unsigned long long &a, unsigned long long &b) {
  asm volatile("ld.relaxed.sys.global.v2.b64 {%0, %1}, [%2];" : "=l"(a), "=l"(b) : "l"(p) : "memory");
}
__device__ __forceinline__ bool ll_valid(unsigned long long a, unsigned long long b, unsigned long long e, double &v) {
  const unsigned fa = (unsigned)(a >> 32), fb = (unsigned)(b >> 32);
  v = __longlong_as_double((long long)((a & 0xffffffffULL) | (b << 32)));
  return fa == fb && (int)(fa - (unsigned)e) >= 0;
}
__device__ __forceinline__ LLEntry *ll_vec(double *region, int src_rank) { return reinterpret_cast<LLEntry *>(region + FZ_VEC) + (size_t)src_rank * PC_MAX; }
__device__ __forceinline__ LLEntry *ll_scal(double *region, int kind, int src_rank) { return reinterpret_cast<LLEntry *>(region + FZ_SCAL) + kind * PC_RANKS + src_rank; }
__device__ __forceinline__ LLEntry *ll_u(double *region) { return reinterpret_cast<LLEntry *>(region + FZ_U); }
// rank-ordered sum over the world mailbox rows of entry i (exchange e): all loads are issued before any is checked (the
// entries have normally arrived behind the barrier: one L2 round trip instead of `world` dependent ones); a late entry is
// then spun on individually.
// (not inlined: its 2 x PC_RANKS live words must not add to the register pressure of the streaming phases)
__device__ __noinline__ double ll_sum_ranks(double *region, int world, int i, unsigned long long e, bool &ok) {
  unsigned long long a[PC_RANKS], b[PC_RANKS];
#pragma unroll
  for (int r = 0; r < PC_RANKS; r++) if (r < world) ll_raw(ll_vec(region, r) + i, a[r], b[r]);
  double s = 0.0;
#pragma unroll
  for (int r = 0; r < PC_RANKS; r++) {
    if (r < world) {
      double w;
      if (!ll_valid(a[r], b[r], e, w) && !ll_load(ll_vec(region, r) + i, e, w)) ok = false;
      s += w;
    }
  }
  return s;
}

// all-reduce of nv <= 2 scalars of kinds kind0, kind0+1: `loc` is this rank's value (identical in every CTA).  CTA 0
// pushes, every CTA polls its local mailboxes (threads r < world) and sums in rank order through shared memory.
__device__ __forceinline__ bool fz_allreduce_scal(const FusedArgs &a, unsigned long long e, int kind0, const double *loc, int nv,
                                                  double *out, double *shm /* >= 2 * PC_RANKS + 1 doubles */) {
  __syncthreads();
  if (threadIdx.x == 0) shm[2 * PC_RANKS] = 0.0;
  if (blockIdx.x == 0 && (int)threadIdx.x < a.world)
    for (int k = 0; k < nv; k++) ll_store(ll_scal(a.peer[threadIdx.x], kind0 + k, a.rank), loc[k], e);
  __syncthreads();
  if ((int)threadIdx.x < a.world) {
    for (int k = 0; k < nv; k++) {
      double v;
      if (!ll_load(ll_scal(a.peer[a.rank], kind0 + k, threadIdx.x), e, v)) shm[2 * PC_RANKS] = 1.0;
      shm[k * PC_RANKS + threadIdx.x] = v;
    }
  }
  __syncthreads();
  for (int k = 0; k < nv; k++) { double s = 0.0; for (int r = 0; r < a.world; r++) s += shm[k * PC_RANKS + r]; out[k] = s; }
  return shm[2 * PC_RANKS] == 0.0;
}

__device__ __forceinline__ double cta_sum_fixed(const double *p, int np, double *sh) {  // fixed-order sum, valid in every thread
  double s = 0.0;
  for (int i = threadIdx.x; i < np; i += blockDim.x) s += p[i];
  return block_sum(s, sh);
}

// NV independent CTA-wide sums with ONE barrier pair: warp butterflies (independent => latencies overlap), per-warp
// partials through shared memory, thread q < NV ends up with the total of value q in v[0] (fixed order).
template <int NV>
__device__ __forceinline__ void cta_sum_multi(double (&v)[NV], double *shm /* (FT/32) * NV doubles */) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int q = 0; q < NV; q++) v[q] = warp_sum(v[q]);
  __syncthreads();
  if (lane == 0) {
#pragma unroll
    for (int q = 0; q < NV; q++) shm[warp * NV + q] = v[q];
  }
  __syncthreads();
  if (threadIdx.x < NV) {
    double s = 0.0;
    for (int w = 0; w < FT / 32; w++) s += shm[w * NV + threadIdx.x];
    v[0] = s;
  }
}

// ---- row phase shared by the fused projcg and pcg kernels: t[i] = J[i] . v for the rows of this CTA.  One WARP per
// row (rows i = c + w G of warp w: every row of the CTA is streamed concurrently, so the bytes in flight stay constant
// over the whole phase and all CTAs finish together); v goes through double-buffered shared-memory chunks (one L2
// read per CTA instead of one per row); CU x 128-bit loads in flight per lane.  Single GPU: t -> a.tm.  Column-sharded:
// {partial t_i, exchange number e} is pushed into every rank's mailbox row [my rank] with one 128-bit store per peer.
// The main loop runs over whole blocks of CU x 32 pairs and keeps its loads free of bounds tests: with a predicate on each
// load ptxas interleaves the loads with their uses (runs of 1-5 in flight instead of CU).  A partial block goes through the
// tail loop, in the same per-lane summation order.
template <bool SKIP = false>
__device__ __forceinline__ void fz_rows(const FusedArgs &a, const double *v, double2 *vch, bool multi, unsigned long long e) {
  const int G = gridDim.x, c = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, m = a.m;
  const int64_t n2 = a.n >> 1;
  const double2 *rp2 = reinterpret_cast<const double2 *>(v);
  for (int pass0 = 0; c + (int64_t)pass0 * (FT / 32) * G < m; pass0++) {
    const int i = c + (pass0 * (FT / 32) + warp) * G;
    const bool act = i < m;
    const double *row = a.J + (int64_t)(act ? i : 0) * a.ldj;
    const unsigned char *nzr = SKIP ? a.nz + (int64_t)((act ? i : 0) >> 6) * a.nz_ld : nullptr;
    const int nch = (int)((n2 + RCH - 1) / RCH);
    double acc = 0.0;
    __syncthreads();
    for (int p = tid; p < (int)min((int64_t)RCH, n2); p += FT) vch[p] = rp2[p];
    __syncthreads();
    for (int ch = 0; ch < nch; ch++) {
      const double2 *cur = vch + (ch & 1) * RCH;
      double2 *nxt = vch + ((ch + 1) & 1) * RCH;
      const int64_t base = (int64_t)ch * RCH;
      const int len = (int)min((int64_t)RCH, n2 - base);
      if (ch + 1 < nch) {
        const int nlen = (int)min((int64_t)RCH, n2 - base - RCH);
        for (int p = tid; p < nlen; p += FT) nxt[p] = rp2[base + RCH + p];
      }
      if (act) {
        const double *rb = row + 2 * base;
        int p = lane;
        for (; p + (CU - 1) * 32 < len; p += 32 * CU) {
          double2 q[CU];
#pragma unroll
          for (int k = 0; k < CU; k++) { const int pp = p + k * 32; q[k] = (!SKIP || nzr[(base + pp) >> 3]) ? ld_stream2(rb + 2 * pp) : make_double2(0.0, 0.0); }
#pragma unroll
          for (int k = 0; k < CU; k++) { const double2 w = cur[p + k * 32]; acc += q[k].x * w.x + q[k].y * w.y; }
        }
        for (; p < len; p += 32) {
          const double2 q = (!SKIP || nzr[(base + p) >> 3]) ? ld_stream2(rb + 2 * p) : make_double2(0.0, 0.0);
          const double2 w = cur[p]; acc += q.x * w.x + q.y * w.y;
        }
      }
      __syncthreads();
    }
    acc = warp_sum(acc);
    if (lane == 0 && act) {
      if (!multi) a.tm[i] = acc;
      else for (int r = 0; r < a.world; r++) ll_store(ll_vec(a.peer[r], a.rank) + i, acc, e);
    }
  }
}

// ---- column phase shared by both kernels: s_j = sum_i J[i][j] u[i] over ALL m rows for the column pairs [p0, p1) this
// CTA owns (u staged in shared memory `us`); thread groups split the rows, `fin(p, s0, s1)` is called once per pair by
// its owner thread with the finished sums.
template <bool SKIP = false, class F>
__device__ __forceinline__ void fz_cols(const FusedArgs &a, const double *us, double2 *red, int64_t p0, int64_t p1, F fin) {
  const int tid = threadIdx.x, m = a.m;
  for (int64_t pc = p0; pc < p1; pc += FT) {
    const int PW = (int)min((int64_t)FT, p1 - pc);
    const int RG = FT / PW;                       // row groups sharing one column pair
    const int g = tid / PW, pl = tid - g * PW;
    double a0 = 0.0, a1 = 0.0;
    if (g < RG) {
      const double *base = a.J + 2 * (pc + pl);
      const unsigned char *nzc = SKIP ? a.nz + ((pc + pl) >> 3) : nullptr;
      int i = g;
      for (; i + (CU - 1) * RG < m; i += CU * RG) {
        double2 q[CU];
#pragma unroll
        for (int k = 0; k < CU; k++) q[k] = (!SKIP || nzc[(int64_t)((i + k * RG) >> 6) * a.nz_ld]) ? ld_stream2(base + (int64_t)(i + k * RG) * a.ldj) : make_double2(0.0, 0.0);
        asm volatile("" ::: "memory");
#pragma unroll
        for (int k = 0; k < CU; k++) { const double w = us[i + k * RG]; a0 += q[k].x * w; a1 += q[k].y * w; }
      }
      for (; i < m; i += RG) {
        const double2 q = (!SKIP || nzc[(int64_t)(i >> 6) * a.nz_ld]) ? ld_stream2(base + (int64_t)i * a.ldj) : make_double2(0.0, 0.0);
        const double w = us[i]; a0 += q.x * w; a1 += q.y * w;
      }
    }
    __syncthreads();
    red[tid] = make_double2(a0, a1);
    __syncthreads();
    if (g == 0) {
      double s0 = 0.0, s1 = 0.0;
      for (int k = 0; k < RG; k++) { const double2 w = red[k * PW + pl]; s0 += w.x; s1 += w.y; }
      fin(pc + pl, s0, s1);
    }
  }
}

// Grid barrier of the cooperative launch: one monotone arrival counter (zeroed by the host before every launch);
// thread 0 of each CTA arrives with a release-add at gpu scope and spins with acquire loads until everybody of this
// generation has arrived.  Co-residency of all CTAs is guaranteed by cudaLaunchCooperativeKernel.
// sync() also returns the ABORT flag (column-sharded mode): a CTA whose peer-memory exchange timed out raises it and
// keeps running with substitute values up to the next barrier, where EVERY CTA reads the same flag value and leaves --
// no CTA is ever left spinning in a barrier the others will not reach.
struct GridBar {
  unsigned *ctr; unsigned gen, nblk; int *abort_flag; int *s_abort;
  __device__ __forceinline__ bool sync() {
    __syncthreads();
    if (threadIdx.x == 0) {
      gen++;
      const unsigned target = gen * nblk;
      asm volatile("red.release.gpu.global.add.u32 [%0], %1;" ::"l"(ctr), "r"(1u) : "memory");
      unsigned v;
      do { asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(ctr) : "memory"); } while (v < target);
      *s_abort = abort_flag ? *reinterpret_cast<volatile int *>(abort_flag) : 0;
    }
    __syncthreads();
    return *s_abort != 0;
  }
  __device__ __forceinline__ void raise() { if (abort_flag) atomicExch(abort_flag, 1); }
};

// ---- dense m x m matvec phase: out[i] = sum_k M[i][k] in[k] for the rows c, c + G, ... of this CTA, TR rows at once (every
// thread takes the same k-slices of all TR rows: TR x 128-bit loads in flight, one CTA-wide reduction per sweep).  `in` is
// a plain m-vector, or (mail) the rank-ordered sum of the t mailboxes of exchange ep.
// (not inlined, scalar arguments only: keeps its registers out of the streaming phases' budget)
__device__ __forceinline__ bool fz_matvec(const double *M, int64_t ldm, int m, const double *in, double *region, int world,
                                       unsigned long long ep, double *out, double *red_d) {
  const int G = gridDim.x, c = blockIdx.x, tid = threadIdx.x;
  const bool mail = region != nullptr;
  const int m2 = (m + 1) >> 1;
  bool ok = true;
  for (int i0 = c; i0 < m; i0 += G * TR) {
    double acc[TR];
#pragma unroll
    for (int q = 0; q < TR; q++) acc[q] = 0.0;
    for (int k2 = tid; k2 < m2; k2 += FT) {
      const int k = 2 * k2;
      const bool has1 = k + 1 < m;
      double v0, v1;
      if (mail) {
        v0 = ll_sum_ranks(region, world, k, ep, ok);
        v1 = has1 ? ll_sum_ranks(region, world, k + 1, ep, ok) : 0.0;
      } else { v0 = in[k]; v1 = has1 ? in[k + 1] : 0.0; }
#pragma unroll
      for (int q = 0; q < TR; q++) {
        const int row = i0 + q * G;
        const bool inr = row < m;
        const double2 w = *reinterpret_cast<const double2 *>(M + (inr ? (int64_t)row * ldm + k : 0));
        acc[q] += (inr ? w.x * v0 : 0.0) + ((inr && has1) ? w.y * v1 : 0.0);
      }
    }
    cta_sum_multi<TR>(acc, red_d);
    if (tid < TR && i0 + tid * G < m) out[i0 + tid * G] = acc[0];
  }
  return ok;
}

// ---- column-sharded solve: rank r owns the rows [r mb, (r+1) mb) of u = G^-1 t (mb = ceil(m / world)): 1/world of the
// G^-1 traffic and of the dot products per GPU instead of a replicated solve.  One warp per owned row; the CTAs that hold
// such rows first stage t (rank-ordered sum of the t mailboxes) in shared memory, then every finished u_i is pushed into
// the u mailbox of every rank (exchange eu).
__device__ __noinline__ bool fz_solve_sharded(const double *Ginv, int64_t ldm, int m, int rank, int world, double *const *peer,
                                              unsigned long long et, unsigned long long eu, double *tsh) {
  const int c = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, W = FT / 32;
  const int mb = (m + world - 1) / world, lo = rank * mb, hi = min(m, lo + mb);
  bool ok = true;
  if (lo + c * W >= hi) return ok;                                   // this CTA owns no row
  for (int i = tid; i < m; i += FT) tsh[i] = ll_sum_ranks(peer[rank], world, i, et, ok);
  __syncthreads();
  for (int row = lo + c * W + warp; row < hi; row += gridDim.x * W) {
    const double *g = Ginv + (int64_t)row * ldm;
    double acc = 0.0;
    for (int k = 2 * lane; k < m; k += 64) {
      const double2 w = *reinterpret_cast<const double2 *>(g + k);
      acc += w.x * tsh[k] + ((k + 1 < m) ? w.y * tsh[k + 1] : 0.0);
    }
    acc = warp_sum(acc);
    if (lane < world) ll_store(ll_u(peer[lane]) + row, acc, eu);
  }
  return ok;
}

// MULTI = column-sharded (world > 1); TRI = the two triangular solve phases (large.cu::factorize's explicit-inverse guard)
// instead of one phase with the explicit G^-1.  Each instantiation carries only its own solve and exchange code.
template <bool MULTI, bool TRI>
__global__ void __launch_bounds__(FT, 1) fused_projcg_kernel(FusedArgs a) {
  __shared__ int s_abort;
  GridBar grid{a.bar, 0u, gridDim.x, MULTI ? a.abort_flag : nullptr, &s_abort};
  extern __shared__ __align__(16) double fsm[];            // [m] staged u | [FT] double2 scratch for the column phase
  __shared__ double sh[33];
  const int G = gridDim.x, c = blockIdx.x, tid = threadIdx.x;
  const int64_t n2 = a.n >> 1;
  const int64_t P = (n2 + G - 1) / G;        // owned column pairs [p0, p1)
  const int64_t p0 = min((int64_t)c * P, n2), p1 = min(p0 + P, n2);
  const int m = a.m;
  double *pA = a.part, *pB = a.part + G, *pC = a.part + 2 * G;
  double *red_d = fsm + ((m + 1) & ~1);      // scratch after the staged u: FT double2
  double2 *vch = reinterpret_cast<double2 *>(red_d + 2 * FT);   // 2 x RCH double2: rp chunks of the row phase
  LargeCtrl *ctrl = a.ctrl;
  double rg = a.first ? cta_sum_fixed(a.lp_rg, a.np_rg, sh) : ctrl->gg;
  const double tol = ctrl->tol;
  const int lim = ctrl->lim;
  int iter = ctrl->iter, status = ctrl->status;
  // dAd / alpha / beta / rp.gp / |g| are reported through the control block by CTA 0 as soon as they are known, so that no
  // thread keeps them live across the streaming phases (whose loads in flight need the registers)
  const bool reporter = c == 0 && tid == 0;
  double gg = ctrl->gg;
  constexpr bool multi = MULTI;
  unsigned long long ep = multi ? *a.epoch : 0ULL;   // exchanges completed so far (every CTA counts the same sequence)
  __shared__ double *s_peer[PC_RANKS];
  if (tid == 0) s_abort = 0;
  if (tid < PC_RANKS) s_peer[tid] = a.peer[tid];
  __syncthreads();
  grid.sync();                               // every CTA has read the control block before anyone may rewrite it
  // optional phase profile (LFPSQP_FUSED_PROF=1): CTA 0 / thread 0 accumulates globaltimer deltas per phase
  // (accumulated in global memory by the one profiling thread: no registers are held across the phases for it)
  const bool prof = a.prof != nullptr && c == 0 && tid == 0;
  auto tick = [&](int ph) {
    if (prof) {
      unsigned long long now; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(now));
      if (ph >= 0) a.prof[ph] += (double)(now - (unsigned long long)a.prof[8]);
      else for (int q = 0; q < 8; q++) a.prof[q] = 0.0;
      a.prof[8] = (double)now;
    }
  };
  tick(-1);

  for (int k = 0; k < a.max_iters && status == 0; k++) {
    // ---- P1: Ad = hd .* d ; partial d.Ad
    {
      double s = 0.0;
      for (int64_t p = p0 + tid; p < p1; p += FT) {
        const double2 d2 = *reinterpret_cast<const double2 *>(a.dc + 2 * p);
        const double2 h2 = *reinterpret_cast<const double2 *>(a.hd + 2 * p);
        const double2 v = make_double2(h2.x * d2.x, h2.y * d2.y);
        *reinterpret_cast<double2 *>(a.Ad + 2 * p) = v;
        s += d2.x * v.x + d2.y * v.y;
      }
      s = block_sum(s, sh);
      if (tid == 0) pA[c] = s;
    }
    if (grid.sync()) { status = 5; break; }
    tick(0);
    // ---- update1 (projcg.jl:74-93).  The exits of :77-89 are taken BEHIND the next barrier, so that a CTA whose exchange
    // timed out (substitute dAd = 1) and the CTAs that see the true value leave the loop at the same barrier.
    double dAd = cta_sum_fixed(pA, G, sh);
    if (multi) { double o; if (fz_allreduce_scal(a, ++ep, 0, &dAd, 1, &o, red_d)) dAd = o; else { grid.raise(); dAd = 1.0; } }
    iter++;
    const int exit_st = (dAd <= 0.0) ? 2 : ((rg <= 0.0) ? 3 : 0);
    if (reporter) ctrl->dAd = dAd;
    if (!exit_st) {
      const double alpha = rg / dAd;
      if (reporter) ctrl->alpha = alpha;
      for (int64_t p = p0 + tid; p < p1; p += FT) {
        const double2 d2 = *reinterpret_cast<const double2 *>(a.dc + 2 * p);
        const double2 r2 = *reinterpret_cast<const double2 *>(a.r + 2 * p);
        const double2 A2 = *reinterpret_cast<const double2 *>(a.Ad + 2 * p);
        double2 x2 = *reinterpret_cast<double2 *>(a.xs + 2 * p);
        x2.x += alpha * d2.x; x2.y += alpha * d2.y;
        *reinterpret_cast<double2 *>(a.xs + 2 * p) = x2;
        *reinterpret_cast<double2 *>(a.rp + 2 * p) = make_double2(r2.x + alpha * A2.x, r2.y + alpha * A2.y);
      }
    }
    if (grid.sync()) { status = 5; break; }
    if (exit_st) { status = exit_st; break; }
    tick(1);
    // ---- rows: t = J rp (fz_rows: one warp per row; column-sharded: partials pushed into every rank's mailboxes)
    fz_rows(a, a.rp, vch, multi, ep + 1);
    // t is complete behind a grid barrier; column-sharded, the remote partials are already on their way (no fence, no flag
    // round trip) and the solve phase checks the per-entry exchange numbers.  (Without this barrier the early CTAs'
    // polling competes with the CTAs still streaming J: measured slower.)
    if (grid.sync()) { status = 5; break; }
    if (multi) ++ep;
    tick(2);
    // ---- u = G^-1 t.  Well-conditioned factor: the explicit symmetric inverse G^-1 = L^-T L^-1 (formed once per
    // factorisation by a DMMA GEMM) makes this ONE grid phase -- sharded over the ranks when column-sharded (each rank
    // solves m / world rows and pushes its slice of u).  Otherwise (TRI, large.cu::factorize's explicit-inverse guard):
    // two dependent triangular phases y = L^-1 t, u = L^-T y with the accuracy of a triangular solve.
    if constexpr (TRI) {
      if (!fz_matvec(a.Linv, a.ldm, m, a.tm, multi ? s_peer[a.rank] : nullptr, a.world, ep, a.ty, red_d)) grid.raise();
      if (grid.sync()) { status = 5; break; }
      fz_matvec(a.XT, a.ldm, m, a.ty, nullptr, 1, 0ULL, a.tu, red_d);
    } else if constexpr (MULTI) {
      if (!fz_solve_sharded(a.Ginv, a.ldm, m, a.rank, a.world, s_peer, ep, ep + 1, fsm)) grid.raise();
      ++ep;
    } else {
      fz_matvec(a.Ginv, a.ldm, m, a.tm, nullptr, 1, 0ULL, a.tu, red_d);
    }
    if (grid.sync()) { status = 5; break; }
    tick(3);
    // ---- cols: gp = rp - J' u on the owned columns ; partials rp.gp, gp.gp
    {
      if constexpr (MULTI && !TRI) {
        bool ok = true;
        const LLEntry *ub = ll_u(a.peer[a.rank]);
        for (int i0 = tid; i0 < m; i0 += 4 * FT) {       // 4 independent polls in flight per thread
          unsigned long long wa[4], wb[4];
#pragma unroll
          for (int q = 0; q < 4; q++) if (i0 + q * FT < m) ll_raw(ub + i0 + q * FT, wa[q], wb[q]);
#pragma unroll
          for (int q = 0; q < 4; q++) {
            const int i = i0 + q * FT;
            if (i < m) { double w; if (!ll_valid(wa[q], wb[q], ep, w) && !ll_load(ub + i, ep, w)) ok = false; fsm[i] = w; }
          }
        }
        if (!ok) grid.raise();
      } else for (int i = tid; i < m; i += FT) fsm[i] = a.tu[i];
      __syncthreads();
      double sb = 0.0, sc = 0.0;
      fz_cols(a, fsm, reinterpret_cast<double2 *>(red_d), p0, p1, [&](int64_t p, double s0, double s1) {
        const double2 rp2 = *reinterpret_cast<const double2 *>(a.rp + 2 * p);
        const double2 g2 = make_double2(rp2.x - s0, rp2.y - s1);
        *reinterpret_cast<double2 *>(a.gp + 2 * p) = g2;
        sb += rp2.x * g2.x + rp2.y * g2.y; sc += g2.x * g2.x + g2.y * g2.y;
      });
      sb = block_sum(sb, sh); sc = block_sum(sc, sh);
      if (tid == 0) { pB[c] = sb; pC[c] = sc; }
    }
    if (grid.sync()) { status = 5; break; }
    tick(5);
    // ---- update3 (projcg.jl:98-111)
    double rpgp = cta_sum_fixed(pB, G, sh);
    gg = cta_sum_fixed(pC, G, sh);
    if (multi) {
      double loc[2] = {rpgp, gg}, o[2];
      if (fz_allreduce_scal(a, ++ep, 1, loc, 2, o, red_d)) { rpgp = o[0]; gg = o[1]; } else grid.raise();
    }
    const double beta = rpgp / rg;
    for (int64_t p = p0 + tid; p < p1; p += FT) {
      const double2 g2 = *reinterpret_cast<const double2 *>(a.gp + 2 * p);
      double2 d2 = *reinterpret_cast<double2 *>(a.dc + 2 * p);
      d2.x = beta * d2.x - g2.x; d2.y = beta * d2.y - g2.y;
      *reinterpret_cast<double2 *>(a.dc + 2 * p) = d2;
      *reinterpret_cast<double2 *>(a.r + 2 * p) = g2;
    }
    const double nr = sqrt(gg);
    rg = gg;                                    // r == g after every projection (:100-101)
    if (nr < tol) status = 1; else if (iter >= lim) status = 4;
    if (reporter) { ctrl->beta = beta; ctrl->rpgp = rpgp; ctrl->nr = nr; }
    tick(6);
    // no barrier: the next P1 touches only this CTA's own columns; pA is next written after every CTA has passed the
    // barrier that follows its last read of pB/pC
  }
  // column-sharded: one more barrier before leaving (unless the abort was already seen at a barrier), so that a CTA that lost
  // its last exchange -- and therefore went on into another iteration -- meets the others at a barrier and all leave together
  if (multi && status != 5 && grid.sync()) status = 5;
  if (c == 0 && tid == 0) {
    if (multi) *a.epoch = ep;
    if (status == 5) ctrl->commfail = 1;
    ctrl->iter = iter; ctrl->status = status; ctrl->gg = gg; ctrl->rg = rg;
  }
}


// ================================================================== persistent pcg! (src/retractions.jl:179-246, M! = copy)
// CG on (J'J + mu I) dx = r inside ProjPenalty's Gauss-Newton step: the other HBM-bound loop of the large-n mode (two
// passes over J per iteration, no solve).  Same building blocks as the projcg kernel; the whole pcg! call (at most
// maxiter_pcg <= 128 iterations) is ONE launch.  Vector roles in FusedArgs: xs = dx, r = r, dc = p, Ad = z.
//   rho_k = r.r ; exit tests (||r|| <= tol, iteration cap) ; p = r + (rho_k / rho_{k-1}) p      [owned columns]   (:207-216)
//   B   t = J p                                                                                  [owned rows]      (:221)
//   B   z = J' t + mu p ; partial p.z                                                            [owned columns]   (:222-226)
//   B   alpha = rho / p.z ; dx += alpha p ; r -= alpha z ; partial r.r                           [owned columns]   (:229-235)
//   B
template <bool MULTI, bool SKIP = false>
__global__ void __launch_bounds__(FT, 1) fused_pcg_kernel(FusedArgs a) {
  __shared__ int s_abort;
  GridBar grid{a.bar, 0u, gridDim.x, MULTI ? a.abort_flag : nullptr, &s_abort};
  extern __shared__ __align__(16) double fsm[];
  __shared__ double sh[33];
  const int G = gridDim.x, c = blockIdx.x, tid = threadIdx.x, m = a.m;
  const int64_t n2 = a.n >> 1;
  const int64_t P = (n2 + G - 1) / G;
  const int64_t p0 = min((int64_t)c * P, n2), p1 = min(p0 + P, n2);
  double *pA = a.part, *pB = a.part + G;
  double *red_d = fsm + ((m + 1) & ~1);
  double2 *vch = reinterpret_cast<double2 *>(red_d + 2 * FT);
  LargeCtrl *ctrl = a.ctrl;
  constexpr bool multi = MULTI;
  unsigned long long ep = multi ? *a.epoch : 0ULL;
  const double tol = ctrl->tol, mu = ctrl->mu;
  const int lim = ctrl->pcg_lim;
  int iter = 0, status = 0;
  double rho = cta_sum_fixed(a.lp_rg, a.np_rg, sh), rho_prev = 1.0, norm_res = INFINITY, pz = 0.0, alpha = 0.0;
  __shared__ double *s_peer[PC_RANKS];
  if (tid == 0) s_abort = 0;
  if (tid < PC_RANKS) s_peer[tid] = a.peer[tid];
  __syncthreads();
  grid.sync();
  if (multi) { double o; if (fz_allreduce_scal(a, ++ep, 1, &rho, 1, &o, red_d)) rho = o; else grid.raise(); }
  while (status == 0) {
    // ---- :207-216 ; the exits are taken behind the next barrier (see fused_projcg_kernel)
    const int exit_st = (!(norm_res > tol)) ? 1 : ((iter >= lim) ? 4 : 0);
    if (!exit_st) {
      const double beta = rho / rho_prev;
      for (int64_t p = p0 + tid; p < p1; p += FT) {
        const double2 r2 = *reinterpret_cast<const double2 *>(a.r + 2 * p);
        double2 d2 = *reinterpret_cast<double2 *>(a.dc + 2 * p);
        d2.x = r2.x + beta * d2.x; d2.y = r2.y + beta * d2.y;
        *reinterpret_cast<double2 *>(a.dc + 2 * p) = d2;
      }
    }
    if (grid.sync()) { status = 5; break; }
    if (exit_st) { status = exit_st; break; }
    // ---- t = J p
    fz_rows<SKIP>(a, a.dc, vch, multi, ep + 1);
    if (grid.sync()) { status = 5; break; }
    if (multi) ++ep;
    // ---- z = J' t + mu p ; partial p.z
    {
      bool late = false;
      for (int i = tid; i < m; i += FT) {
        bool okk = true;
        fsm[i] = multi ? ll_sum_ranks(a.peer[a.rank], a.world, i, ep, okk) : a.tm[i];
        if (!okk) late = true;
      }
      if (late) grid.raise();
      __syncthreads();
      double sp = 0.0;
      fz_cols<SKIP>(a, fsm, reinterpret_cast<double2 *>(red_d), p0, p1, [&](int64_t p, double s0, double s1) {
        const double2 d2 = *reinterpret_cast<const double2 *>(a.dc + 2 * p);
        const double2 z2 = make_double2(s0 + mu * d2.x, s1 + mu * d2.y);
        *reinterpret_cast<double2 *>(a.Ad + 2 * p) = z2;
        sp += d2.x * z2.x + d2.y * z2.y;
      });
      sp = block_sum(sp, sh);
      if (tid == 0) pA[c] = sp;
    }
    if (grid.sync()) { status = 5; break; }
    pz = cta_sum_fixed(pA, G, sh);
    if (multi) { double o; if (fz_allreduce_scal(a, ++ep, 0, &pz, 1, &o, red_d)) pz = o; else grid.raise(); }
    // ---- :229-235
    alpha = rho / pz;
    {
      double sr = 0.0;
      for (int64_t p = p0 + tid; p < p1; p += FT) {
        const double2 d2 = *reinterpret_cast<const double2 *>(a.dc + 2 * p);
        const double2 z2 = *reinterpret_cast<const double2 *>(a.Ad + 2 * p);
        double2 x2 = *reinterpret_cast<double2 *>(a.xs + 2 * p);
        double2 r2 = *reinterpret_cast<double2 *>(a.r + 2 * p);
        x2.x += alpha * d2.x; x2.y += alpha * d2.y;
        r2.x -= alpha * z2.x; r2.y -= alpha * z2.y;
        *reinterpret_cast<double2 *>(a.xs + 2 * p) = x2;
        *reinterpret_cast<double2 *>(a.r + 2 * p) = r2;
        sr += r2.x * r2.x + r2.y * r2.y;
      }
      sr = block_sum(sr, sh);
      if (tid == 0) pB[c] = sr;
    }
    if (grid.sync()) { status = 5; break; }
    rho_prev = rho;
    rho = cta_sum_fixed(pB, G, sh);
    if (multi) { double o; if (fz_allreduce_scal(a, ++ep, 1, &rho, 1, &o, red_d)) rho = o; else grid.raise(); }
    norm_res = sqrt(rho);
    iter++;
  }
  if (c == 0 && tid == 0) {
    if (multi) *a.epoch = ep;
    if (status == 5) ctrl->commfail = 1;
    ctrl->pcg_iter = iter; ctrl->pcg_status = status; ctrl->norm_res = norm_res; ctrl->rho = rho; ctrl->pz = pz; ctrl->alpha = alpha;
  }
}

}  // namespace

// Returns 0 when the chunk was enqueued, 1 when this configuration is not eligible (the caller uses the unfused path).
int fused_projcg_chunk(LargeState &S, int iters, int first, double *xs, double *r, double *dc, double *Ad, double *rp, double *gp) {
  if (S.ineq || S.family != LFPSQP_FAM_DIAGQUAD || (S.n_loc & 1) || S.m < 1 || !S.fused_ok || !S.Ginv) return 1;
  if (S.world > 1 && !(S.comm && S.comm->peer_ready && S.m <= PC_MAX && S.world <= PC_RANKS)) return 1;
  const bool multi = S.world > 1, tri = !S.explicit_inverse_ok;
  FusedArgs a;
  for (int r = 0; r < PC_RANKS; r++) a.peer[r] = (S.world > 1) ? S.comm->peer_map[r] : nullptr;
  a.rank = S.rank; a.world = S.world; a.epoch = (S.world > 1) ? reinterpret_cast<unsigned long long *>(S.comm->peer_local + FZ_FLAG + PC_RANKS) : nullptr;   // lives with the region
  a.n = S.n_loc; a.ldj = S.ldj; a.ldm = S.ldm; a.m = S.m;
  a.J = S.J; a.Ginv = S.Ginv; a.hd = S.hdiag; a.Linv = S.Linv; a.XT = S.XT;
  a.xs = xs; a.dc = dc; a.r = r; a.Ad = Ad; a.rp = rp; a.gp = gp; a.tm = S.tm; a.tu = S.tu; a.ty = S.ty;
  a.abort_flag = reinterpret_cast<int *>(S.fused_part + 3 * (size_t)S.fused_grid + 14);
  a.part = S.fused_part; a.lp_rg = S.lp + 3 * (size_t)MAXP; a.np_rg = S.np_loop; a.first = first; a.max_iters = iters;
  a.ctrl = S.ctrl;
  a.bar = reinterpret_cast<unsigned *>(S.fused_part + 3 * (size_t)S.fused_grid + 12);
  cudaMemsetAsync(a.bar, 0, 4 * sizeof(double), S.stream);   // barrier counter (+12) + abort flag (+14)
  static const bool want_prof = getenv("LFPSQP_FUSED_PROF") != nullptr;
  a.prof = want_prof ? S.fused_part + 3 * (size_t)S.fused_grid : nullptr;
  const size_t smem = ((size_t)((S.m + 1) & ~1) + 2 * FT + 4 * RCH) * sizeof(double);
  void *args[] = {&a};
  void *kern = multi ? (tri ? (void *)fused_projcg_kernel<true, true> : (void *)fused_projcg_kernel<true, false>)
                     : (tri ? (void *)fused_projcg_kernel<false, true> : (void *)fused_projcg_kernel<false, false>);
  cudaError_t e = cudaLaunchCooperativeKernel(kern, dim3(S.fused_grid), dim3(FT), args, smem, S.stream);
  if (e != cudaSuccess) { cudaGetLastError(); S.fused_ok = false; return 1; }
  S.launches++;
  S.disp[multi || tri ? LARGE_DISP_FUSED_GENERAL : LARGE_DISP_FUSED_SINGLE]++;
  S.disp[LARGE_DISP_SOLVE] |= tri ? (int64_t)LARGE_SOLVE_TRIANGULAR : large_ginv_form(S);
  if (want_prof) {
    double h[8];
    cudaMemcpyAsync(h, a.prof, sizeof(h), cudaMemcpyDeviceToHost, S.stream);
    cudaStreamSynchronize(S.stream);
    fprintf(stderr, "[fused projcg] %d iterations max; us per phase over the chunk: hess %.1f | update1 %.1f | rows %.1f | solve %.1f | (unused %.1f) | cols %.1f | update3 %.1f\n",
            iters, h[0] / 1e3, h[1] / 1e3, h[2] / 1e3, h[3] / 1e3, h[4] / 1e3, h[5] / 1e3, h[6] / 1e3);
  }
  return 0;
}

// The whole pcg! call as one launch (state as large.cu::run_pcg: dx = S.w3, r = S.w0, p = S.w1 zeroed, z = S.w2, r.r partials of
// the start residual in loop slot 5; tol / mu / pcg_lim already in the device control block).  Returns 1 when not eligible.
int fused_pcg(LargeState &S, double *dx, double *r, double *pv, double *z) {
  if (S.ineq || (S.n_loc & 1) || S.m < 1 || !S.fused_ok) return 1;
  if (S.world > 1 && !(S.comm && S.comm->peer_ready && S.m <= PC_MAX && S.world <= PC_RANKS)) return 1;
  FusedArgs a;
  for (int q = 0; q < PC_RANKS; q++) a.peer[q] = (S.world > 1) ? S.comm->peer_map[q] : nullptr;
  a.rank = S.rank; a.world = S.world;
  a.epoch = (S.world > 1) ? reinterpret_cast<unsigned long long *>(S.comm->peer_local + FZ_FLAG + PC_RANKS) : nullptr;
  a.n = S.n_loc; a.ldj = S.ldj; a.ldm = S.ldm; a.m = S.m;
  a.J = S.J; a.Ginv = nullptr; a.hd = nullptr; a.Linv = nullptr; a.XT = nullptr;
  a.xs = dx; a.dc = pv; a.r = r; a.Ad = z; a.rp = nullptr; a.gp = nullptr; a.tm = S.tm; a.tu = S.tu; a.ty = S.ty;
  a.abort_flag = reinterpret_cast<int *>(S.fused_part + 3 * (size_t)S.fused_grid + 14);
  a.part = S.fused_part; a.lp_rg = S.lp + 5 * (size_t)MAXP; a.np_rg = S.np_loop_raw; a.first = 1; a.max_iters = 0;
  a.ctrl = S.ctrl; a.prof = nullptr;
  a.bar = reinterpret_cast<unsigned *>(S.fused_part + 3 * (size_t)S.fused_grid + 12);
  cudaMemsetAsync(a.bar, 0, 4 * sizeof(double), S.stream);   // barrier counter (+12) + abort flag (+14)
  const size_t smem = ((size_t)((S.m + 1) & ~1) + 2 * FT + 4 * RCH) * sizeof(double);
  void *args[] = {&a};
  // block-sparse J whose zero-slab map is current (large.cu::gram_syrk): the instantiation that does not load all-zero slabs
  const bool skip = S.world <= 1 && S.jmap_valid && S.gram_mode == 1 && S.nzmap;
  if (skip) { a.nz = S.nzmap; a.nz_ld = S.nz_ld; }
  void *kern = S.world > 1 ? (void *)fused_pcg_kernel<true> : (skip ? (void *)fused_pcg_kernel<false, true> : (void *)fused_pcg_kernel<false>);
  cudaError_t e = cudaLaunchCooperativeKernel(kern, dim3(S.fused_grid), dim3(FT), args, smem, S.stream);
  if (e != cudaSuccess) { cudaGetLastError(); return 1; }
  S.launches++;
  S.disp[LARGE_DISP_FUSED_PCG]++;
  return 0;
}

// one-time eligibility probe: cooperative launch support, co-residency of one CTA per SM with the dynamic shared memory
void fused_projcg_init(LargeState &S, int device) {
  S.fused_ok = false;
  int coop = 0;
  if (cudaDeviceGetAttribute(&coop, cudaDevAttrCooperativeLaunch, device) != cudaSuccess || !coop) { cudaGetLastError(); return; }
  const size_t smem = ((size_t)((S.m + 1) & ~1) + 2 * FT + 4 * RCH) * sizeof(double);
  if (smem > SMEM_MAX) return;
  // the attribute is per kernel and process-wide: opting in to the eligibility limit (not this context's size) keeps a
  // context with a larger m launchable after a smaller one was set up
  const void *kernels[] = {(const void *)fused_projcg_kernel<false, false>, (const void *)fused_projcg_kernel<false, true>,
                           (const void *)fused_projcg_kernel<true, false>, (const void *)fused_projcg_kernel<true, true>,
                           (const void *)fused_pcg_kernel<false>, (const void *)fused_pcg_kernel<false, true>, (const void *)fused_pcg_kernel<true>};
  for (const void *k : kernels)
    if (cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SMEM_MAX) != cudaSuccess) { cudaGetLastError(); return; }
  int per_sm = 0;
  if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, fused_projcg_kernel<true, false>, FT, smem) != cudaSuccess || per_sm < 1) { cudaGetLastError(); return; }
  S.fused_grid = S.sm_count;
  void *p = nullptr;
  if (cudaMalloc(&p, (3 * (size_t)S.fused_grid + 16) * sizeof(double)) != cudaSuccess) { cudaGetLastError(); return; }   // partials | 9 prof | barrier | abort
  cudaMemset(p, 0, (3 * (size_t)S.fused_grid + 16) * sizeof(double));
  S.owned.push_back(p); S.fused_part = (double *)p;
  if (S.family == LFPSQP_FAM_DIAGQUAD) {   // explicit G^-1 is only needed by the fused projcg (diagonal Hessians); pcg needs no factor
    void *gi = nullptr;
    if (cudaMalloc(&gi, (size_t)S.m * S.ldm * sizeof(double)) != cudaSuccess) { cudaGetLastError(); return; }
    S.owned.push_back(gi); S.Ginv = (double *)gi;
  }
  S.fused_ok = true;
}
