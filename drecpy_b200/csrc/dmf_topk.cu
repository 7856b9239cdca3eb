// K6c: full-catalog top-k for DMF (sm_100a): score = max(1e-6, cos(user tower(u), item tower(i))) for a block of users
// against the whole catalog on the CUDA cores, with the top-k kept in bounded per-user candidate lists.
//
// Replaces (reference, DRecPy/): Recommender/recommender_abc.py:413-419 (_recommend = _rank over range(n_items)) ->
// :454-461 (DMF: one _predict per candidate, dmf.py:101-106, then heapq.nlargest on (score, iid)), for many users.
//
// Contract: row u is bit for bit what drb_dmf_rank_candidates (score.cu, k_rank_candidates, mode 1) returns for user u
// with the whole catalog as candidates, truncated to k.  That kernel forms a score in one warp: lane L keeps the fmaf
// chain over k = L, L + 32, ..., the 32 partials are added by the xor butterfly (16, 8, 4, 2, 1), and
//   score = fmaxf(1e-6f, dot * (1 / sqrtf(fmaxf(|u|^2, 1e-12f))) * (1 / sqrtf(fmaxf(|t|^2, 1e-12f)))).
// Here one THREAD forms a whole score with the same arithmetic: the 32 lane partials in the same chains, added in the
// butterfly's pairing (float addition is commutative, so lane 0's sum is the one every lane of the warp holds), and the
// same inverse norms (computed per user and per item by the rank path's own code).  The build has no fast-math, and
// the tree uses __fadd_rn / __fmaf_rn so that nothing is contracted.  Vectors are zero-padded to a multiple of 32: an
// extra fmaf(0, 0, p) returns p (up to the sign of a zero, which only a zero dot can carry, and that scores 1e-6).
//
// Selection scheme (drb_dmf_topk in api.cu drives it; the select kernels are score.cu's, shared with drb_cdae_topk):
//   the catalog is swept from the highest item id down in item ranges growing geometrically.  The first range lists
//   every unseen item; after each range but the last the select keeps the keys >= tau = the k-th best score so far;
//   later ranges list only the scores whose orderable value is STRICTLY above tau.  An item that only ties tau has a
//   smaller id than every key already listed with that score, so it can never enter the answer -- this is what keeps
//   the lists bounded when thousands of items share one score (ReLU on the last layer of both towers: an all-zero
//   tower output puts every score of that user or item at the 1e-6 floor).  The last select emits the answer in the
//   reference's order (score desc, iid desc).  A list that overflows its capacity sends its user to the exact
//   fallback (k_dmf_fallback_scores + k_topk), so the result never depends on the list capacity.
#include <algorithm>

#include "topk_common.cuh"

namespace {

constexpr int DT_THREADS = 256;              // 8 warps
constexpr int DT_R = 4;                      // users per thread (one warp = 4 users)
constexpr int DT_UT = DT_R * (DT_THREADS / 32);   // users per CTA
constexpr int DT_QCAP = 128;                 // entries of a warp's key queue

// Inverse norm of every item's tower output (the rank path's arithmetic), and the output transposed to [W32][I_pad]
// (k-major, zero-padded to W32 = 32 NJ rows and I_pad columns) for the filter's shared-memory tiles.  One warp per item.
__global__ void __launch_bounds__(256) k_dmf_topk_prep(const float* irep, int ld_i, int width, int n_items, int i_pad,
                                                       int w32, float* irep_t, float* item_inv) {
  const int i = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (i >= i_pad) return;
  const float* tr = irep + (int64_t)i * ld_i;
  float tss = 0.f;
  for (int k = lane; k < w32; k += 32) {
    const float t = (i < n_items && k < width) ? tr[k] : 0.f;
    irep_t[(int64_t)k * i_pad + i] = t;
    if (k < width) tss = fmaf(t, t, tss);
  }
  tss = warp_sum(tss);
  if (lane == 0) item_inv[i] = i < n_items ? 1.0f / sqrtf(fmaxf(tss, 1e-12f)) : 0.f;
}

// Sum of the 32 lane partials in the xor butterfly's pairing, as lane 0 sees it: V(o, L) = V(2o, L) + V(2o, L ^ o),
// V(32, L) = lane L's fmaf chain over k = L, L + 32, ...  For R users x C items at once: us[k][DT_UT] and ts[k][IT]
// are the k-major shared-memory tiles, u0 / c0 the thread's first user / item column.
template <int O, int L, int NJ, int C, int IT>
__device__ __forceinline__ void tree_dot(const float* us, const float* ts, int u0, int c0, float (&v)[DT_R][C]) {
  if constexpr (O == 32) {
#pragma unroll
    for (int r = 0; r < DT_R; r++)
#pragma unroll
      for (int c = 0; c < C; c++) v[r][c] = 0.f;
#pragma unroll
    for (int j = 0; j < NJ; j++) {
      const int k = j * 32 + L;
      const float4 u = *reinterpret_cast<const float4*>(us + k * DT_UT + u0);     // broadcast
      float t[C];
      if constexpr (C == 4) {
        const float4 q = *reinterpret_cast<const float4*>(ts + k * IT + c0);
        t[0] = q.x; t[1] = q.y; t[2] = q.z; t[3] = q.w;
      } else if constexpr (C == 2) {
        const float2 q = *reinterpret_cast<const float2*>(ts + k * IT + c0);
        t[0] = q.x; t[1] = q.y;
      } else {
        t[0] = ts[k * IT + c0];
      }
      const float uu[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
      for (int r = 0; r < DT_R; r++)
#pragma unroll
        for (int c = 0; c < C; c++) v[r][c] = __fmaf_rn(uu[r], t[c], v[r][c]);
    }
  } else {
    float b[DT_R][C];
    tree_dot<O * 2, L, NJ, C, IT>(us, ts, u0, c0, v);
    tree_dot<O * 2, (L ^ O), NJ, C, IT>(us, ts, u0, c0, b);
#pragma unroll
    for (int r = 0; r < DT_R; r++)
#pragma unroll
      for (int c = 0; c < C; c++) v[r][c] = __fadd_rn(v[r][c], b[r][c]);
  }
}

__device__ __forceinline__ void cp_async16(void* smem, const void* gmem) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"((uint32_t)__cvta_generic_to_shared(smem)), "l"(gmem)
               : "memory");
}

// Scoring and filter pass over the item range [item_lo, item_hi) for a block of users.  A CTA holds DT_UT users'
// vectors (k-major) in shared memory and sweeps its share of the range in tiles of IT items, double-buffered through
// cp.async (the transposed item tower output is 32 NJ x I_pad floats and stays in L2).  Thread (warp w, lane l) owns the
// DT_R x C micro-tile of users 4w..4w+3 and items C l..C l+C-1 of the tile.  Keys that pass go through a per-warp queue
// in shared memory into the users' lists.
template <int NJ, int C>
__global__ void __launch_bounds__(DT_THREADS) k_dmf_topk_filter(DmfFilterArgs a) {
  constexpr int W32 = 32 * NJ, IT = 32 * C;
  extern __shared__ __align__(16) uint8_t dt_smem[];
  float* us = reinterpret_cast<float*>(dt_smem);                     // [W32][DT_UT]
  float* ts = us + W32 * DT_UT;                                       // [2][W32][IT]
  uint64_t* qk_all = reinterpret_cast<uint64_t*>(ts + 2 * W32 * IT);   // [8][DT_QCAP]
  unsigned short* qu_all = reinterpret_cast<unsigned short*>(qk_all + 8 * DT_QCAP);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int row0 = blockIdx.x * DT_UT;
  const int n_tiles = (a.item_hi - a.item_lo + IT - 1) / IT;

  auto load_tile = [&](int t, int buf) {
    const float* src = a.irep_t + a.item_lo + t * IT;
    float* dst = ts + buf * W32 * IT;
    for (int f = threadIdx.x; f < W32 * (IT / 4); f += DT_THREADS) {
      const int k = f / (IT / 4), q = f % (IT / 4);
      cp_async16(dst + k * IT + 4 * q, src + (int64_t)k * a.i_pad + 4 * q);
    }
    asm volatile("cp.async.commit_group;" ::: "memory");
  };
  int t = blockIdx.y;
  if (t < n_tiles) load_tile(t, 0);

  // the users' vectors, transposed and zero-padded; rows past the block never pass (tau = all ones)
  for (int f = threadIdx.x; f < W32 * DT_UT; f += DT_THREADS) {
    const int r = f % DT_UT, k = f / DT_UT;
    const int row = row0 + r;
    us[k * DT_UT + r] = (row < a.n_users && k < a.width) ? a.urep[(int64_t)row * a.ld_u + k] : 0.f;
  }
  // per user of the warp: inverse norm (the rank path's arithmetic: lane chains + warp_sum) and threshold
  float inv_u[DT_R];
  uint32_t tau[DT_R];
#pragma unroll
  for (int r = 0; r < DT_R; r++) {
    const int row = row0 + warp * DT_R + r;
    float uss = 0.f;
    if (row < a.n_users) {
      const float* ur = a.urep + (int64_t)row * a.ld_u;
      for (int k = lane; k < a.width; k += 32) uss = fmaf(ur[k], ur[k], uss);
    }
    uss = warp_sum(uss);
    inv_u[r] = 1.0f / sqrtf(fmaxf(uss, 1e-12f));
    tau[r] = row < a.n_users ? __ldg(a.tau_ord + row) : 0xffffffffu;
  }
  uint64_t* qk = qk_all + warp * DT_QCAP;
  unsigned short* qu = qu_all + warp * DT_QCAP;
  int qn = 0;
  const uint32_t lt_mask = (1u << lane) - 1u;

  for (int tl = 0; t < n_tiles; t += gridDim.y, tl++) {
    const int buf = tl & 1;
    if (t + (int)gridDim.y < n_tiles) {
      load_tile(t + gridDim.y, buf ^ 1);
      asm volatile("cp.async.wait_group 1;" ::: "memory");
    } else {
      asm volatile("cp.async.wait_group 0;" ::: "memory");
    }
    __syncthreads();
    const int item0 = a.item_lo + t * IT + C * lane;
    float inv_t[C];
#pragma unroll
    for (int c = 0; c < C; c++) inv_t[c] = __ldg(a.item_inv + item0 + c);
    float v[DT_R][C];
    tree_dot<1, 0, NJ, C, IT>(us, ts + buf * W32 * IT, warp * DT_R, C * lane, v);
#pragma unroll
    for (int r = 0; r < DT_R; r++) {
      const int row = warp * DT_R + r;                       // row of the block (the lists' index)
#pragma unroll
      for (int c = 0; c < C; c++) {
        const int item = item0 + c;
        const float s = fmaxf(1e-6f, __fmul_rn(__fmul_rn(v[r][c], inv_u[r]), inv_t[c]));
        const uint32_t ord = f2ord(s);
        bool pass = item < a.item_hi && ord > tau[r];
        uint32_t bal = __ballot_sync(0xffffffffu, pass);
        if (bal == 0u) continue;                               // warp-uniform
        if (a.seen_bits) {                                     // novelty: the user's stored items drop out
          if (pass) pass = !((__ldg(a.seen_bits + (int64_t)(row0 + row) * a.words_per_row + (item >> 5)) >> (item & 31)) & 1u);
          bal = __ballot_sync(0xffffffffu, pass);
          if (bal == 0u) continue;
        }
        const int n = __popc(bal);
        if (qn + n > DT_QCAP) {
          flush_key_queue<DT_QCAP>(qk, qu, qn, a.cnt + row0, a.lists + (int64_t)row0 * a.cap, a.cap);
          qn = 0;
        }
        if (pass) {
          const int e = qn + __popc(bal & lt_mask);
          qk[e] = ((uint64_t)ord << 32) | (uint32_t)item;
          qu[e] = (unsigned short)row;
        }
        qn += n;
      }
    }
    __syncthreads();                                          // the buffer is refilled two tiles on
  }
  if (qn > 0) flush_key_queue<DT_QCAP>(qk, qu, qn, a.cnt + row0, a.lists + (int64_t)row0 * a.cap, a.cap);
}

template <int NJ, int C>
int run_filter(drb_ctx* ctx, const DmfFilterArgs& a) {
  constexpr int W32 = 32 * NJ, IT = 32 * C;
  constexpr int SMEM = (W32 * DT_UT + 2 * W32 * IT) * 4 + 8 * DT_QCAP * (8 + 2);
  static_assert(SMEM <= 227 * 1024, "dmf top-k filter: shared memory");
  auto kern = k_dmf_topk_filter<NJ, C>;
  static bool attr_set = false;
  if (!attr_set) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM);
    if (e != cudaSuccess) return drb_fail(DRB_E_CUDA, "cudaFuncSetAttribute(k_dmf_topk_filter) failed: %s", cudaGetErrorString(e));
    attr_set = true;
  }
  const int ux = (a.n_users + DT_UT - 1) / DT_UT;
  const int n_tiles = (a.item_hi - a.item_lo + IT - 1) / IT;
  // enough CTAs for several waves over the SMs; each CTA keeps its users and walks every gridDim.y-th tile
  const int gy = std::max(1, std::min(n_tiles, (8 * ctx->sm_count + ux - 1) / ux));
  drb_prof_scope prof_(ctx, "k_dmf_topk_filter");
  kern<<<dim3(ux, gy), DT_THREADS, SMEM, ctx->stream>>>(a);
  DRB_LAUNCH_CHECK(ctx, "k_dmf_topk_filter");
  return DRB_OK;
}

// Exact fallback for users whose candidate list overflowed: fills the user's claimed scratch row with the scores over
// the whole catalog, computed exactly as k_rank_candidates computes them (one warp per item); k_topk (indirect form)
// then ranks the row.
__global__ void __launch_bounds__(256) k_dmf_fallback_scores(const float* urep, int ld_u, const float* irep, int ld_i,
                                                             int width, int n_items, float* rows, int ld_rows,
                                                             const int32_t* fb_users, const int32_t* fb_count, int fb_max) {
  const int slot = blockIdx.x;       // one CTA per claimed scratch row (k_select_lists claims them)
  if (slot >= min(*fb_count, fb_max)) return;
  const int u = fb_users[slot];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const float* ur = urep + (int64_t)u * ld_u;
  float* row = rows + (int64_t)slot * ld_rows;
  float uss = 0.f;
  for (int k = lane; k < width; k += 32) uss = fmaf(ur[k], ur[k], uss);
  uss = warp_sum(uss);
  for (int i = warp; i < n_items; i += 8) {
    const float* tr = irep + (int64_t)i * ld_i;
    float dot = 0.f, tss = 0.f;
    for (int k = lane; k < width; k += 32) {
      const float t = tr[k];
      dot = fmaf(ur[k], t, dot);
      tss = fmaf(t, t, tss);
    }
    dot = warp_sum(dot);
    tss = warp_sum(tss);
    const float c_ = dot * (1.0f / sqrtf(fmaxf(uss, 1e-12f))) * (1.0f / sqrtf(fmaxf(tss, 1e-12f)));
    if (lane == 0) row[i] = fmaxf(1e-6f, c_);
  }
}

}  // namespace

int dmf_topk_nj(int width) {
  int nj = 1;
  while (32 * nj < width) nj <<= 1;
  return nj;
}

int launch_dmf_topk_prep(drb_ctx* ctx, const float* irep, int ld_i, int width, int n_items, int i_pad, float* irep_t,
                         float* item_inv) {
  if (i_pad % 128 || i_pad < n_items) return drb_fail(DRB_E_INVALID, "dmf_topk_prep: bad item padding");
  drb_prof_scope prof_(ctx, "k_dmf_topk_prep");
  k_dmf_topk_prep<<<(i_pad + 7) / 8, 256, 0, ctx->stream>>>(irep, ld_i, width, n_items, i_pad, 32 * dmf_topk_nj(width),
                                                             irep_t, item_inv);
  DRB_LAUNCH_CHECK(ctx, "k_dmf_topk_prep");
  return DRB_OK;
}

int launch_dmf_topk_filter(drb_ctx* ctx, const DmfFilterArgs& a) {
  if (a.n_users <= 0 || a.item_lo >= a.item_hi) return DRB_OK;
  if (a.item_lo % 128 || a.item_hi > a.i_pad || a.n_users > 65536)
    return drb_fail(DRB_E_INVALID, "dmf_topk_filter: bad item range [%d, %d) or block of %d users", a.item_lo, a.item_hi,
                    a.n_users);
  switch (dmf_topk_nj(a.width)) {   // item tiles of 128, 64, 32 items as the vectors widen (shared memory)
    case 1: return run_filter<1, 4>(ctx, a);
    case 2: return run_filter<2, 4>(ctx, a);
    case 4: return run_filter<4, 2>(ctx, a);
    case 8: return run_filter<8, 1>(ctx, a);
    case 16: return run_filter<16, 1>(ctx, a);
  }
  return drb_fail(DRB_E_INVALID, "dmf_topk_filter: width %d above 512", a.width);
}

int launch_dmf_topk_fallback(drb_ctx* ctx, const TopkArgs& a, int n, const float* urep, int ld_u, const float* irep,
                             int ld_i, int width, float* rows, int32_t* fb_users, int32_t* fb_count, int fb_max) {
  if (n <= 0) return DRB_OK;
  {
    drb_prof_scope prof_(ctx, "k_dmf_fallback_scores");
    k_dmf_fallback_scores<<<fb_max, 256, 0, ctx->stream>>>(urep, ld_u, irep, ld_i, width, a.n_items, rows, a.ld, fb_users,
                                                           fb_count, fb_max);
    DRB_LAUNCH_CHECK(ctx, "k_dmf_fallback_scores");
  }
  TopkArgs t = a;
  t.scores = rows; t.fb_users = fb_users; t.fb_count = fb_count; t.fb_max = fb_max;
  return launch_topk(ctx, t, fb_max);
}
