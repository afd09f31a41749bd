// large_fused_single.cu -- the single-GPU, explicit-inverse instance of the persistent fused projcg kernel, kept as its own
// translation unit: it is the kernel behind the "large-n projcg iterations/s" metric (C5: 2930 it/s = 0.98 of the measured HBM
// peak), and ptxas only keeps all 16 x 128-bit loads of the row phase in flight while the kernel around the streaming loops is
// this small (with the column-sharded mailbox code, the sharded solve and the triangular fallback compiled into the same
// kernel the row phase ran 17 % slower: 185 vs 158 us at C5).  large_fused.cu holds the general kernel (column-sharded,
// two-phase solve) and pcg!; both files implement the same phases -- see the header of large_fused.cu.
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

struct FusedArgs {
  int64_t n, ldj, ldm;       // local columns (even), leading dimensions
  int m;
  const double *J, *Ginv, *hd;
  double *xs, *dc, *r, *Ad, *rp, *gp, *tm, *tu;
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
};

// ---- in-kernel all-reduce over NVLink: push model with flag-in-data mailboxes (the "LL" idea: every 16-byte entry
// carries {value, exchange number} and is written with ONE 128-bit store, which the fabric delivers atomically; the
// consumer spins on the entry itself).  No fence, no separate flag, no extra grid barrier: an exchange costs one
// one-way NVLink latency.  Every rank (including the sender itself) receives a copy in its own region, so consumers
// only read local memory; sums are taken in rank order => bitwise identical on every rank and CTA.
// Reuse is safe without double buffering: a rank overwrites its entries of kind K only after it has consumed a later
// exchange from every peer, and a peer sends that later exchange only behind a grid barrier that follows all of its
// reads of kind K.
struct __align__(16) LLEntry { double v; unsigned long long e; };
__device__ __forceinline__ void ll_store(LLEntry *p, double v, unsigned long long e) {
  asm volatile("st.relaxed.sys.global.v2.b64 [%0], {%1, %2};" ::"l"(p), "l"(__double_as_longlong(v)), "l"(e) : "memory");
}
// spin until the entry carries exchange >= e; false after ~4 s (a peer died: do not hang the GPU)
__device__ __forceinline__ bool ll_load(const LLEntry *p, unsigned long long e, double &v) {
  long long bits; unsigned long long f;
  const long long t0 = clock64();
  do {
    asm volatile("ld.relaxed.sys.global.v2.b64 {%0, %1}, [%2];" : "=l"(bits), "=l"(f) : "l"(p) : "memory");
    if (f >= e) { v = __longlong_as_double(bits); return true; }
    __nanosleep(40);
  } while (clock64() - t0 < 8000000000LL);
  v = 0.0;
  return false;
}
__device__ __forceinline__ LLEntry *ll_vec(double *region, int src_rank) { return reinterpret_cast<LLEntry *>(region + FZ_VEC) + (size_t)src_rank * PC_MAX; }
__device__ __forceinline__ LLEntry *ll_scal(double *region, int kind, int src_rank) { return reinterpret_cast<LLEntry *>(region + FZ_SCAL) + kind * PC_RANKS + src_rank; }

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
__device__ __forceinline__ void fz_rows(const FusedArgs &a, const double *v, double2 *vch, bool multi, unsigned long long e) {
  const int G = gridDim.x, c = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, m = a.m;
  const int64_t n2 = a.n >> 1;
  const double2 *rp2 = reinterpret_cast<const double2 *>(v);
  for (int pass0 = 0; c + (int64_t)pass0 * (FT / 32) * G < m; pass0++) {
    const int i = c + (pass0 * (FT / 32) + warp) * G;
    const bool act = i < m;
    const double *row = a.J + (int64_t)(act ? i : 0) * a.ldj;
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
        for (int p = lane; p < len; p += 32 * CU) {
          double2 q[CU];
#pragma unroll
          for (int k = 0; k < CU; k++) { const int pp = p + k * 32; q[k] = (pp < len) ? ld_stream2(rb + 2 * pp) : make_double2(0.0, 0.0); }
#pragma unroll
          for (int k = 0; k < CU; k++) { const int pp = p + k * 32; if (pp < len) { const double2 w = cur[pp]; acc += q[k].x * w.x + q[k].y * w.y; } }
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
template <class F>
__device__ __forceinline__ void fz_cols(const FusedArgs &a, const double *us, double2 *red, int64_t p0, int64_t p1, F fin) {
  const int tid = threadIdx.x, m = a.m;
  for (int64_t pc = p0; pc < p1; pc += FT) {
    const int PW = (int)min((int64_t)FT, p1 - pc);
    const int RG = FT / PW;                       // row groups sharing one column pair
    const int g = tid / PW, pl = tid - g * PW;
    double a0 = 0.0, a1 = 0.0;
    if (g < RG) {
      const double *base = a.J + 2 * (pc + pl);
      int i = g;
      for (; i + (CU - 1) * RG < m; i += CU * RG) {
        double2 q[CU];
#pragma unroll
        for (int k = 0; k < CU; k++) q[k] = ld_stream2(base + (int64_t)(i + k * RG) * a.ldj);
#pragma unroll
        for (int k = 0; k < CU; k++) { const double w = us[i + k * RG]; a0 += q[k].x * w; a1 += q[k].y * w; }
      }
      for (; i < m; i += RG) { const double2 q = ld_stream2(base + (int64_t)i * a.ldj); const double w = us[i]; a0 += q.x * w; a1 += q.y * w; }
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
struct GridBar {
  unsigned *ctr; unsigned gen, nblk;
  __device__ __forceinline__ void sync() {
    __syncthreads();
    if (threadIdx.x == 0) {
      gen++;
      const unsigned target = gen * nblk;
      asm volatile("red.release.gpu.global.add.u32 [%0], %1;" ::"l"(ctr), "r"(1u) : "memory");
      unsigned v;
      do { asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(ctr) : "memory"); } while (v < target);
    }
    __syncthreads();
  }
};

__global__ void __launch_bounds__(FT, 1) fused_projcg_kernel(FusedArgs a) {
  GridBar grid{a.bar, 0u, gridDim.x};
  extern __shared__ __align__(16) double fsm[];            // [m] staged u | [FT] double2 scratch for the column phase
  __shared__ double sh[33];
  const int G = gridDim.x, c = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
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
  double dAd = 0.0, alpha = 0.0, beta = 0.0, rpgp = 0.0, gg = ctrl->gg, nr = ctrl->nr;
  const bool multi = a.world > 1;
  unsigned long long ep = multi ? *a.epoch : 0ULL;   // exchanges completed so far (every CTA counts the same sequence)
  __shared__ int s_timeout;
  if (tid == 0) s_timeout = 0;
  __syncthreads();
  grid.sync();                               // every CTA has read the control block before anyone may rewrite it
  // optional phase profile (LFPSQP_FUSED_PROF=1): CTA 0 / thread 0 accumulates globaltimer deltas per phase
  const bool prof = a.prof != nullptr && c == 0 && tid == 0;
  unsigned long long tph[8] = {0, 0, 0, 0, 0, 0, 0, 0}, tlast = 0;
  auto tick = [&](int ph) {
    if (prof) { unsigned long long now; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(now)); if (ph >= 0) tph[ph] += now - tlast; tlast = now; }
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
    grid.sync();
    tick(0);
    // ---- update1 (projcg.jl:74-93)
    dAd = cta_sum_fixed(pA, G, sh);
    if (multi) { double o; if (!fz_allreduce_scal(a, ++ep, 0, &dAd, 1, &o, red_d)) { status = 5; break; } dAd = o; }
    iter++;
    if (dAd <= 0.0) { status = 2; break; }
    if (rg <= 0.0) { status = 3; break; }
    alpha = rg / dAd;
    for (int64_t p = p0 + tid; p < p1; p += FT) {
      const double2 d2 = *reinterpret_cast<const double2 *>(a.dc + 2 * p);
      const double2 r2 = *reinterpret_cast<const double2 *>(a.r + 2 * p);
      const double2 A2 = *reinterpret_cast<const double2 *>(a.Ad + 2 * p);
      double2 x2 = *reinterpret_cast<double2 *>(a.xs + 2 * p);
      x2.x += alpha * d2.x; x2.y += alpha * d2.y;
      *reinterpret_cast<double2 *>(a.xs + 2 * p) = x2;
      *reinterpret_cast<double2 *>(a.rp + 2 * p) = make_double2(r2.x + alpha * A2.x, r2.y + alpha * A2.y);
    }
    grid.sync();
    tick(1);
    // ---- rows: t = J rp (fz_rows: one warp per row; column-sharded: partials pushed into every rank's mailboxes)
    fz_rows(a, a.rp, vch, multi, ep + 1);
    // t is complete behind a grid barrier; column-sharded, the remote partials are already on their way (no fence, no flag
    // round trip) and the solve phase checks the per-entry exchange numbers.  (Without this barrier the early CTAs'
    // polling competes with the CTAs still streaming J: measured slower.)
    grid.sync();
    if (multi) ++ep;
    tick(2);
    // ---- u = G^-1 t with the explicit symmetric inverse G^-1 = L^-T L^-1 (formed once per factorisation by a DMMA
    // GEMM): ONE grid phase instead of two dependent triangular ones.  The CTA owns the rows c, c + G, ... and works
    // on TR of them at once: every thread takes the same k-slices of all TR rows (TR x 128-bit loads in flight), one
    // CTA-wide reduction per sweep.
    {
      const int m2 = (m + 1) >> 1;
      for (int i0 = c; i0 < m; i0 += G * TR) {
        double acc[TR];
#pragma unroll
        for (int q = 0; q < TR; q++) acc[q] = 0.0;
        for (int k2 = tid; k2 < m2; k2 += FT) {
          const int k = 2 * k2;
          const bool has1 = k + 1 < m;
          double v0, v1;
          if (multi) {   // t = rank-ordered sum of the mailbox entries (spin until each carries this exchange)
            // first try: the entries of 4 ranks at a time with independent loads in flight (they have normally arrived
            // behind the barrier); a late entry is then spun on individually.  Odd tail (k + 1 == m): re-read entry k.
            v0 = 0.0; v1 = 0.0;
            const int k1 = has1 ? k + 1 : k;
            for (int r0 = 0; r0 < a.world; r0 += 4) {
              long long b0[4], b1[4]; unsigned long long f0[4], f1[4];
#pragma unroll
              for (int q = 0; q < 4; q++) {
                const int r = min(r0 + q, a.world - 1);
                const LLEntry *mb = ll_vec(a.peer[a.rank], r);
                asm volatile("ld.relaxed.sys.global.v2.b64 {%0, %1}, [%2];" : "=l"(b0[q]), "=l"(f0[q]) : "l"(mb + k) : "memory");
                asm volatile("ld.relaxed.sys.global.v2.b64 {%0, %1}, [%2];" : "=l"(b1[q]), "=l"(f1[q]) : "l"(mb + k1) : "memory");
              }
#pragma unroll
              for (int q = 0; q < 4; q++) {
                if (r0 + q < a.world) {
                  const LLEntry *mb = ll_vec(a.peer[a.rank], r0 + q);
                  double w0 = __longlong_as_double(b0[q]), w1 = __longlong_as_double(b1[q]);
                  if (f0[q] < ep && !ll_load(mb + k, ep, w0)) s_timeout = 1;
                  if (f1[q] < ep && !ll_load(mb + k1, ep, w1)) s_timeout = 1;
                  v0 += w0; v1 += has1 ? w1 : 0.0;
                }
              }
            }
          } else { v0 = a.tm[k]; v1 = has1 ? a.tm[k + 1] : 0.0; }
#pragma unroll
          for (int q = 0; q < TR; q++) {
            const int row = i0 + q * G;
            const bool inr = row < m;
            const double2 w = *reinterpret_cast<const double2 *>(a.Ginv + (inr ? (int64_t)row * a.ldm + k : 0));
            acc[q] += (inr ? w.x * v0 : 0.0) + ((inr && has1) ? w.y * v1 : 0.0);
          }
        }
        cta_sum_multi<TR>(acc, red_d);
        if (tid < TR && i0 + tid * G < m) a.tu[i0 + tid * G] = acc[0];
      }
      grid.sync();
      tick(3);
      if (multi && s_timeout) { status = 5; break; }
    }
    // ---- cols: gp = rp - J' u on the owned columns ; partials rp.gp, gp.gp
    {
      for (int i = tid; i < m; i += FT) fsm[i] = a.tu[i];
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
    grid.sync();
    tick(5);
    // ---- update3 (projcg.jl:98-111)
    rpgp = cta_sum_fixed(pB, G, sh);
    gg = cta_sum_fixed(pC, G, sh);
    if (multi) {
      double loc[2] = {rpgp, gg}, o[2];
      if (!fz_allreduce_scal(a, ++ep, 1, loc, 2, o, red_d)) { status = 5; break; }
      rpgp = o[0]; gg = o[1];
    }
    beta = rpgp / rg;
    for (int64_t p = p0 + tid; p < p1; p += FT) {
      const double2 g2 = *reinterpret_cast<const double2 *>(a.gp + 2 * p);
      double2 d2 = *reinterpret_cast<double2 *>(a.dc + 2 * p);
      d2.x = beta * d2.x - g2.x; d2.y = beta * d2.y - g2.y;
      *reinterpret_cast<double2 *>(a.dc + 2 * p) = d2;
      *reinterpret_cast<double2 *>(a.r + 2 * p) = g2;
    }
    nr = sqrt(gg);
    rg = gg;                                    // r == g after every projection (:100-101)
    if (nr < tol) status = 1; else if (iter >= lim) status = 4;
    tick(6);
    // no barrier: the next P1 touches only this CTA's own columns; pA is next written after every CTA has passed the
    // barrier that follows its last read of pB/pC
  }
  if (prof) for (int q = 0; q < 8; q++) a.prof[q] = (double)tph[q];
  if (c == 0 && tid == 0) {
    if (multi) *a.epoch = ep;
    if (status == 5) ctrl->rankflag = 99;
    ctrl->iter = iter; ctrl->status = status; ctrl->dAd = dAd; ctrl->alpha = alpha; ctrl->beta = beta;
    ctrl->rpgp = rpgp; ctrl->gg = gg; ctrl->rg = rg; ctrl->nr = nr;
  }
}


}  // namespace

// Returns 0 when the chunk was enqueued, 1 when this configuration is not eligible (the caller uses the unfused path).
int fused_projcg_chunk_single(LargeState &S, int iters, int first, double *xs, double *r, double *dc, double *Ad, double *rp, double *gp) {
  if (S.ineq || S.family != LFPSQP_FAM_DIAGQUAD || (S.n_loc & 1) || S.m < 1 || !S.fused_ok || !S.Ginv || S.world > 1) return 1;
  {
    static bool attr_set = false;   // opt in to the dynamic shared memory once (same size rule as large_fused.cu)
    const size_t smem0 = ((size_t)((S.m + 1) & ~1) + 2 * FT + 4 * RCH) * sizeof(double);
    if (!attr_set) { if (cudaFuncSetAttribute(fused_projcg_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 220 * 1024) != cudaSuccess) { cudaGetLastError(); return 1; } attr_set = true; }
    (void)smem0;
  }
  FusedArgs a;
  for (int r = 0; r < PC_RANKS; r++) a.peer[r] = (S.world > 1) ? S.comm->peer_map[r] : nullptr;
  a.rank = S.rank; a.world = S.world; a.epoch = (S.world > 1) ? reinterpret_cast<unsigned long long *>(S.comm->peer_local + FZ_FLAG + PC_RANKS) : nullptr;   // lives with the region
  a.n = S.n_loc; a.ldj = S.ldj; a.ldm = S.ldm; a.m = S.m;
  a.J = S.J; a.Ginv = S.Ginv; a.hd = S.hdiag;
  a.xs = xs; a.dc = dc; a.r = r; a.Ad = Ad; a.rp = rp; a.gp = gp; a.tm = S.tm; a.tu = S.tu;
  a.part = S.fused_part; a.lp_rg = S.lp + 3 * (size_t)MAXP; a.np_rg = S.np_loop; a.first = first; a.max_iters = iters;
  a.ctrl = S.ctrl;
  a.bar = reinterpret_cast<unsigned *>(S.fused_part + 3 * (size_t)S.fused_grid + 8);
  cudaMemsetAsync(a.bar, 0, sizeof(unsigned), S.stream);
  static const bool want_prof = getenv("LFPSQP_FUSED_PROF") != nullptr;
  a.prof = want_prof ? S.fused_part + 3 * (size_t)S.fused_grid : nullptr;
  const size_t smem = ((size_t)((S.m + 1) & ~1) + 2 * FT + 4 * RCH) * sizeof(double);
  void *args[] = {&a};
  cudaError_t e = cudaLaunchCooperativeKernel((void *)fused_projcg_kernel, dim3(S.fused_grid), dim3(FT), args, smem, S.stream);
  if (e != cudaSuccess) { cudaGetLastError(); S.fused_ok = false; return 1; }
  S.launches++;
  S.disp[LARGE_DISP_FUSED_SINGLE]++; S.disp[LARGE_DISP_SOLVE] |= large_ginv_form(S);
  if (want_prof) {
    double h[8];
    cudaMemcpyAsync(h, a.prof, sizeof(h), cudaMemcpyDeviceToHost, S.stream);
    cudaStreamSynchronize(S.stream);
    fprintf(stderr, "[fused projcg] %d iterations max; us per phase over the chunk: hess %.1f | update1 %.1f | rows %.1f | solve %.1f | (unused %.1f) | cols %.1f | update3 %.1f\n",
            iters, h[0] / 1e3, h[1] / 1e3, h[2] / 1e3, h[3] / 1e3, h[4] / 1e3, h[5] / 1e3, h[6] / 1e3);
  }
  return 0;
}

