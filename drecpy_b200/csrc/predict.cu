// K11: scores of (user, item) pairs, bit for bit what predict() returns for each pair (sm_100a).
//
// Replaces (reference, DRecPy/): Recommender/recommender_abc.py:354-383 (predict) -> cdae.py:84-88 / dmf.py:101-106
// (_predict), called once per pair by Evaluation/Processes/predictive_evaluation.py.  The pairs come grouped by user
// as a CSR (drb_cdae_predict_pairs / drb_dmf_predict_pairs in api.cu): the user side (CDAE hidden layer, DMF user
// tower) is computed once per distinct user, in blocks of max_batch users, by the same calls the full-row paths make,
// and the kernels below score each pair against one catalog row.
//
// CDAE: one thread per pair forms the score with the arithmetic of k_sgemm<LAYOUT_KK, EPI_BIAS_ACT> with splits = 1
// (gemm.cu), which drb_cdae_predict_all runs: one fmaf chain over k = 0 .. ld-1 from +0, then acc + b'[iid], then
// 1 / (1 + expf(-r)).  The GEMM continues its chain over zero-filled k up to the next multiple of 16; fmaf(0, 0, acc)
// leaves acc unchanged except that -0 becomes +0, and a zero logit's sign does not reach the sigmoid's result.
// A warp works on the pairs of one user; the user's h row is staged in shared memory and read as a broadcast, and
// each thread streams its pair's W'^T row (ld-padded, 16-byte aligned) with 128-bit loads.
//
// DMF: one warp per pair runs the forward part of k_dmf_head (dmf.cu) on the user tower's row and the item's row of
// the catalog cache: lane-strided fmaf chains, the xor butterfly, 1 / sqrtf(fmaxf(., 1e-12)), fmaxf(1e-6, c).
#include "kernels.h"

namespace {

constexpr int PR_THREADS = 128;               // 4 warps
constexpr int PR_WARPS = PR_THREADS / 32;
constexpr float L2N_EPS = 1e-12f;

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// bit 0: a user id, 1: pair_off (not 0 .. n, or decreasing), 2: an item id, 3: an output position out of range
__global__ void k_pair_args_check(PairArgs p, int n_users, int n_items, int* bad) {
  int flags = 0;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < (int64_t)p.n + p.n_u + 1;
       i += (int64_t)gridDim.x * blockDim.x) {
    if (i < p.n_u) {
      const int32_t u = p.users[i];
      if (u < 0 || u >= n_users) flags |= 1;
      if (p.pair_off[i] > p.pair_off[i + 1]) flags |= 2;
    }
    if (i == 0 && (p.pair_off[0] != 0 || p.pair_off[p.n_u] != p.n)) flags |= 2;
    if (i < p.n) {
      const int32_t it = p.pair_iid[i], d = p.pair_dst[i];
      if (it < 0 || it >= n_items) flags |= 4;
      if (d < 0 || d >= p.n) flags |= 8;
    }
  }
  if (flags) atomicOr(bad, flags);
}

// users [u0, u0 + c) of the CSR; h row j belongs to user u0 + j
__global__ void __launch_bounds__(PR_THREADS) k_cdae_pair_scores(PairArgs p, int u0, int c, const float* __restrict__ h,
                                                                 const float* __restrict__ w2t,
                                                                 const float* __restrict__ b2, int ld, float* out) {
  extern __shared__ __align__(16) float s_h[];         // [PR_WARPS][ld]
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int j = blockIdx.x * PR_WARPS + warp;
  if (j >= c) return;
  float* hs = s_h + warp * ld;
  for (int k = lane; k < ld; k += 32) hs[k] = h[(int64_t)j * ld + k];
  __syncwarp();
  const int64_t pb = p.pair_off[u0 + j], pe = p.pair_off[u0 + j + 1];
  for (int64_t q = pb + lane; q < pe; q += 32) {
    const int32_t iid = p.pair_iid[q];
    const float4* wr = reinterpret_cast<const float4*>(w2t + (int64_t)iid * ld);
    const float4* hr = reinterpret_cast<const float4*>(hs);
    float acc = 0.f;
    for (int k4 = 0; k4 < ld / 4; k4++) {
      const float4 w = __ldg(wr + k4), x = hr[k4];
      acc = fmaf(x.x, w.x, acc);
      acc = fmaf(x.y, w.y, acc);
      acc = fmaf(x.z, w.z, acc);
      acc = fmaf(x.w, w.w, acc);
    }
    const float r = acc + b2[iid];
    out[p.pair_dst[q]] = 1.0f / (1.0f + expf(-r));
  }
}

// users [u0, u0 + c); CTA j takes user u0 + j, its warps stride over the user's pairs
__global__ void __launch_bounds__(PR_THREADS) k_dmf_pair_head(PairArgs p, int u0, const float* __restrict__ urep,
                                                              int ld_u, const float* __restrict__ irep, int ld_i,
                                                              int width, float* out) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int j = blockIdx.x;
  const float* a = urep + (int64_t)j * ld_u;
  const int64_t pb = p.pair_off[u0 + j], pe = p.pair_off[u0 + j + 1];
  for (int64_t q = pb + warp; q < pe; q += PR_WARPS) {
    const float* e = irep + (int64_t)p.pair_iid[q] * ld_i;
    float ssa = 0.f, sse = 0.f, dot = 0.f;
    for (int k = lane; k < width; k += 32) {
      const float av = a[k], ev = e[k];
      ssa = fmaf(av, av, ssa);
      sse = fmaf(ev, ev, sse);
      dot = fmaf(av, ev, dot);
    }
    ssa = warp_sum(ssa); sse = warp_sum(sse); dot = warp_sum(dot);
    const float inva = 1.0f / sqrtf(fmaxf(ssa, L2N_EPS)), inve = 1.0f / sqrtf(fmaxf(sse, L2N_EPS));
    const float cs = dot * inva * inve;
    if (lane == 0) out[p.pair_dst[q]] = fmaxf(1e-6f, cs);
  }
}

}  // namespace

int launch_pair_args_check(drb_ctx* ctx, const PairArgs& p, int n_users, int n_items, int* bad_dev) {
  DRB_CUDA_TRY(ctx, cudaMemsetAsync(bad_dev, 0, sizeof(int), ctx->stream));
  const int64_t work = (int64_t)p.n + p.n_u + 1;
  const int blocks = (int)std::min<int64_t>((work + 255) / 256, 4096);
  drb_prof_scope prof_(ctx, "k_pair_args_check");
  k_pair_args_check<<<blocks, 256, 0, ctx->stream>>>(p, n_users, n_items, bad_dev);
  DRB_LAUNCH_CHECK(ctx, "k_pair_args_check");
  return DRB_OK;
}

int launch_cdae_pair_scores(drb_ctx* ctx, const PairArgs& p, int u0, int c, const float* h, const float* w2t,
                            const float* b2, int ld, float* out) {
  if (c <= 0) return DRB_OK;
  if (ld % 4) return drb_fail(DRB_E_INVALID, "cdae pair scores: ld %d is not a multiple of 4", ld);
  const size_t smem = (size_t)PR_WARPS * ld * sizeof(float);
  if (smem > 48 * 1024) return drb_fail(DRB_E_INVALID, "cdae pair scores: hidden width %d too large", ld);
  drb_prof_scope prof_(ctx, "k_cdae_pair_scores");
  k_cdae_pair_scores<<<(c + PR_WARPS - 1) / PR_WARPS, PR_THREADS, smem, ctx->stream>>>(p, u0, c, h, w2t, b2, ld, out);
  DRB_LAUNCH_CHECK(ctx, "k_cdae_pair_scores");
  return DRB_OK;
}

int launch_dmf_pair_head(drb_ctx* ctx, const PairArgs& p, int u0, int c, const float* urep, int ld_u,
                         const float* irep, int ld_i, int width, float* out) {
  if (c <= 0) return DRB_OK;
  drb_prof_scope prof_(ctx, "k_dmf_pair_head");
  k_dmf_pair_head<<<c, PR_THREADS, 0, ctx->stream>>>(p, u0, urep, ld_u, irep, ld_i, width, out);
  DRB_LAUNCH_CHECK(ctx, "k_dmf_pair_head");
  return DRB_OK;
}
