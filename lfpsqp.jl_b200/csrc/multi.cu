// multi.cu -- multi-GPU context for the batched mode: the instances of one lfpsqp_solve_batched call are sharded into
// contiguous ranges over the ctx's devices (SURVEY.md 8e: independent units, no collective), one host thread and one
// child ctx (own streams, own device arena) per device, results landing in disjoint slices of the caller's arrays.
#include <algorithm>
#include <string>
#include <thread>
#include <vector>
#include "ctx.h"

extern "C" int lfpsqp_ctx_create_multi(const int *devices, int ndev, lfpsqp_ctx **out) {
  if (!out) return LFPSQP_ERR_ARG;
  *out = nullptr;
  if (!devices || ndev < 1 || ndev > 64) return LFPSQP_ERR_ARG;
  for (int i = 0; i < ndev; i++) for (int j = 0; j < i; j++) if (devices[i] == devices[j]) return LFPSQP_ERR_ARG;   // each device once
  lfpsqp_ctx *parent = nullptr;
  int rc = lfpsqp_ctx_create(devices[0], &parent);     // the parent itself serves every single-GPU entry point on devices[0]
  if (rc) return rc;
  for (int i = 0; i < ndev; i++) {
    lfpsqp_ctx *ch = nullptr;
    rc = lfpsqp_ctx_create(devices[i], &ch);
    if (rc) { lfpsqp_ctx_destroy(parent); return rc; }
    parent->children.push_back(ch);
  }
  *out = parent;
  return LFPSQP_OK;
}

extern "C" int lfpsqp_ctx_device_count(lfpsqp_ctx *c) { return c ? std::max<int>(1, (int)c->children.size()) : 0; }

int solve_batched_multi(lfpsqp_ctx *c, int family, int64_t n, int64_t m, int64_t p, int64_t B, const double *fam_params,
                        int64_t fam_stride, const double *x0, const double *xl, const double *xu, const lfpsqp_params *prm,
                        double *x_out, double *obj_hist, int64_t H, int64_t *obj_len, double *lambda, lfpsqp_term *term,
                        lfpsqp_stats *stats) {
  const int G = (int)c->children.size();
  if (B < 0 || n < 1 || H < 1) return c->fail(LFPSQP_ERR_ARG, "bad sizes");
  const int64_t ME = m + p;
  std::vector<int> rcs(G, 0);
  std::vector<std::thread> th;
  double ms_max = 0.0; int64_t launches = 0;
  auto work = [&](int g) {
    // contiguous, balanced range [lo, hi) of device g
    const int64_t base = B / G, rem = B % G;
    const int64_t lo = g * base + std::min<int64_t>(g, rem), nb = base + (g < rem ? 1 : 0);
    lfpsqp_ctx *ch = c->children[g];
    if (nb == 0) { rcs[g] = 0; ch->last_ms = 0; ch->last_launches = 0; return; }
    if (c->noise_host) { ch->noise_host = c->noise_host + lo * c->noise_T * c->noise_N; ch->noise_T = c->noise_T; ch->noise_N = c->noise_N; ch->noise_B = nb; }
    else { ch->noise_host = nullptr; ch->noise_T = ch->noise_N = ch->noise_B = 0; }
    const double *shard_params = fam_params ? fam_params + (fam_stride ? lo * fam_stride : 0) : nullptr;
    lfpsqp_qcqp qs;
    if (family == LFPSQP_FAM_QCQP && fam_params) {   // the descriptor is shared; each per-instance array moves to the shard's first instance
      qs = *(const lfpsqp_qcqp *)fam_params;
      struct Field { const double *ptr; int64_t stride; };
      static_assert(sizeof(lfpsqp_qcqp) == 9 * sizeof(Field), "lfpsqp_qcqp is nine {pointer, stride} pairs");
      Field *F = (Field *)&qs;
      for (int i = 0; i < 9; i++) if (F[i].ptr && F[i].stride > 0) F[i].ptr += lo * F[i].stride;
      shard_params = (const double *)&qs;
    }
    rcs[g] = lfpsqp_solve_batched(ch, family, n, m, p, nb, shard_params, fam_stride,
                                  x0 ? x0 + lo * n : nullptr, xl, xu, prm, x_out ? x_out + lo * n : nullptr, obj_hist ? obj_hist + lo * H : nullptr, H,
                                  obj_len ? obj_len + lo : nullptr, lambda ? lambda + lo * ME : nullptr, term ? term + lo : nullptr,
                                  stats ? stats + lo : nullptr);
  };
  for (int g = 1; g < G; g++) th.emplace_back(work, g);
  work(0);
  for (auto &t : th) t.join();
  int rc = 0;
  for (int g = 0; g < G; g++) {
    if (rcs[g] && !rc) { rc = rcs[g]; c->err = "device " + std::to_string(c->children[g]->device) + ": " + c->children[g]->err; }
    ms_max = std::max(ms_max, c->children[g]->last_ms);
    launches += c->children[g]->last_launches;
  }
  c->last_ms = ms_max; c->last_launches = launches;
  std::copy(c->children[0]->last_kernel, c->children[0]->last_kernel + 4, c->last_kernel);   // every device runs the same kernel
  return rc;
}
