// K10: per-user ranking-metric sums of full-catalog top-k lists, on the device (sm_100a).
//
// Replaces (reference, DRecPy/): Evaluation/Processes/recommendation_evaluation.py:164-192 -- the per-user metric
// calls on model.recommend's list -> Evaluation/Metrics/ranking.py:20-114 (DCG / NDCG with strong relevancy, and the hit
// counts behind HitRatio / Recall / Precision) -- for a block of users whose top-k lists are still on the device.
//
// Contract: with the lookup table of user u holding the distinct items of its evaluated set (gain = 2^rel - 1 and the
// sampled-positive flag) and its ideal table holding the same gains, dcg / idcg / hits are bit for bit what
// drb_eval_metrics (host_rng.cpp) computes for the same thresholded list, with those distinct items as both its test
// table and its candidate list.  That host loop adds (2^rel - 1) / log2(2 + i) in position order; here the gains and
// the log2 discounts come precomputed by the host's C library, and every step is an explicit IEEE operation
// (__ddiv_rn, __dadd_rn), so nothing is contracted or reassociated.  A zero gain adds +0.0, which changes no bits.
//
// Layout: one warp per user.  Ranked list: the lanes look up 32 positions at a time (binary search in the user's table
// sorted by internal item id), then every lane adds the 32 terms in position order (the sum is warp-uniform).  Ideal
// list: the gains in descending order without sorting them -- each pass finds the largest gain below the previous one
// and how many entries carry it (a warp max/count reduction over the table), then adds that many equal terms.  A pass
// costs |table| / 32 loads per lane, and there are at most (distinct gains among the top max(ks)) passes: ratings have
// a handful of distinct values, so training-set evaluation (tables of thousands of items) stays a few sweeps.
#include "kernels.h"

namespace {

constexpr int EV_THREADS = 256;   // 8 warps = 8 users per CTA

struct EvalTopkArgs {
  const int32_t* top_iid; const float* top_score; int ld; const int32_t* n_out;
  int use_threshold; float threshold;
  const int64_t* lut_off; const int32_t* lut_iid; const double* lut_gain; const uint8_t* lut_pos;
  const int64_t* ideal_off; const double* ideal_gain;
  const double* disc; const int32_t* ks; int n_ks; int k_max;
  double* dcg; double* idcg; int32_t* hits; int32_t* n_rec;
  int n;
};

__global__ void __launch_bounds__(EV_THREADS) k_eval_topk_metrics(EvalTopkArgs a) {
  const int lane = threadIdx.x & 31;
  const int u = blockIdx.x * (EV_THREADS / 32) + (threadIdx.x >> 5);
  if (u >= a.n) return;
  const int64_t ob = (int64_t)u * a.n_ks;
  const int32_t* iid = a.top_iid + (int64_t)u * a.ld;
  const float* score = a.top_score + (int64_t)u * a.ld;

  // valid prefix: the first min(n_out, k_max) entries, cut at the first score below the threshold (descending scores)
  const int nv = min(max(a.n_out[u], 0), a.k_max);
  int n_valid = nv;
  if (a.use_threshold) {
    for (int b = 0; b < nv; b += 32) {
      const int i = b + lane;
      const unsigned bad = __ballot_sync(0xffffffffu, i < nv && !(score[i] >= a.threshold));
      if (bad) { n_valid = b + __ffs(bad) - 1; break; }
    }
  }
  for (int j = lane; j < a.n_ks; j += 32) {
    a.dcg[ob + j] = 0.0; a.idcg[ob + j] = 0.0; a.hits[ob + j] = 0;
    a.n_rec[ob + j] = min(a.ks[j], n_valid);
  }

  // ranked list: running DCG and hit count, read off where a cut-off ends (cut-off j owned by lane j % 32)
  const int64_t lb = a.lut_off[u], le = a.lut_off[u + 1];
  double cur = 0.0;
  int nh = 0;
  for (int b = 0; b < n_valid; b += 32) {
    const int i = b + lane;
    double term = 0.0;
    bool pos = false;
    if (i < n_valid) {
      const int32_t key = iid[i];
      int64_t lo = lb, hi = le;
      while (lo < hi) {
        const int64_t mid = (lo + hi) >> 1;
        if (a.lut_iid[mid] < key) lo = mid + 1; else hi = mid;
      }
      double g = 0.0;
      if (lo < le && a.lut_iid[lo] == key) { g = a.lut_gain[lo]; pos = a.lut_pos[lo] != 0; }
      term = __ddiv_rn(g, a.disc[i]);
    }
    const unsigned pm = __ballot_sync(0xffffffffu, pos);
    const int cnt = min(32, n_valid - b);
    for (int t = 0; t < cnt; t++) {
      cur = __dadd_rn(cur, __shfl_sync(0xffffffffu, term, t));
      nh += (pm >> t) & 1u;
      for (int j = lane; j < a.n_ks; j += 32)
        if (min(a.ks[j], n_valid) == b + t + 1) { a.dcg[ob + j] = cur; a.hits[ob + j] = nh; }
    }
  }

  // ideal list: gains in descending order, one pass per distinct value (count = how many entries carry it)
  const int64_t gb = a.ideal_off[u], ge = a.ideal_off[u + 1];
  const int top = (int)(ge - gb < (int64_t)a.k_max ? ge - gb : (int64_t)a.k_max);
  double best = 0.0, prev = __longlong_as_double(0x7ff0000000000000ll);   // +inf
  int p = 0;
  while (p < top) {
    double m = __longlong_as_double(0xfff0000000000000ll);                // -inf
    int c = 0;
    for (int64_t q = gb + lane; q < ge; q += 32) {
      const double g = a.ideal_gain[q];
      if (g < prev) {
        if (g > m) { m = g; c = 1; } else if (g == m) { c++; }
      }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const double m2 = __shfl_xor_sync(0xffffffffu, m, o);
      const int c2 = __shfl_xor_sync(0xffffffffu, c, o);
      if (m2 > m) { m = m2; c = c2; } else if (m2 == m) { c += c2; }
    }
    if (c == 0) break;                 // nothing left below prev (only NaN gains remain)
    for (int t = 0; t < c && p < top; t++, p++) {
      best = __dadd_rn(best, __ddiv_rn(m, a.disc[p]));
      for (int j = lane; j < a.n_ks; j += 32)
        if (min(a.ks[j], top) == p + 1) a.idcg[ob + j] = best;
    }
    prev = m;
  }
}

}  // namespace

extern "C" {

int drb_eval_topk_metrics(drb_ctx* ctx, int32_t n, const int32_t* top_iid, const float* top_score, int32_t ld,
                          const int32_t* n_out, int32_t use_threshold, double threshold, const int64_t* lut_off,
                          const int32_t* lut_iid, const double* lut_gain, const uint8_t* lut_pos,
                          const int64_t* ideal_off, const double* ideal_gain, const double* disc, const int32_t* ks,
                          int32_t n_ks, int32_t k_max, double* dcg, double* idcg, int32_t* hits, int32_t* n_rec) {
  if (!ctx || n < 0 || ld < 1 || n_ks < 1 || k_max < 1 || k_max > ld)
    return drb_fail(DRB_E_INVALID, "drb_eval_topk_metrics: bad argument");
  if (n == 0) return DRB_OK;
  if (!top_iid || !top_score || !n_out || !lut_off || !lut_iid || !lut_gain || !lut_pos || !ideal_off || !ideal_gain ||
      !disc || !ks || !dcg || !idcg || !hits || !n_rec)
    return drb_fail(DRB_E_INVALID, "drb_eval_topk_metrics: NULL pointer");
  EvalTopkArgs a{top_iid, top_score, ld, n_out, use_threshold != 0, (float)threshold, lut_off, lut_iid, lut_gain,
                 lut_pos, ideal_off, ideal_gain, disc, ks, n_ks, k_max, dcg, idcg, hits, n_rec, n};
  const int per = EV_THREADS / 32;
  drb_prof_scope prof_(ctx, "k_eval_topk_metrics");
  k_eval_topk_metrics<<<(n + per - 1) / per, EV_THREADS, 0, ctx->stream>>>(a);
  DRB_LAUNCH_CHECK(ctx, "k_eval_topk_metrics");
  return DRB_OK;
}

}  // extern "C"
