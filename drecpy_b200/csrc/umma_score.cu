// Full-catalog scoring on the tensor cores with the top-k selection kept on chip: scores = sigmoid(h W'^T + b') for a
// block of users against a range of items (fp32-accurate split products on tcgen05.mma -- 3 x FP16, or 3 x TF32 --,
// TMA-fed, TMEM accumulators: the persistent CTA-pair skeleton of umma_loss.cu), and an epilogue that never writes a
// score to memory.  It appends to every user's candidate list the keys that can still belong to the user's top k.
//
// Replaces (reference, DRecPy/): Recommender/recommender_abc.py:413-419 (_recommend = _rank over range(n_items)) ->
// Recommender/cdae.py:84-103 (_predict over all items, drop the user's training items when novelty, heapq.nlargest on
// (score, iid)), as driven for every user by Evaluation/Processes/recommendation_evaluation.py:164.
//
// Selection scheme (drb_cdae_topk in api.cu drives it; DESIGN.md section 3):
//   stage 0   items [0, n_S): every unseen item of the slice lands in the list (FILTER = false); the select kernel
//             (score.cu) keeps the keys >= tau = the k-th best score and publishes tau and tau_z, a logit below which
//             no score can reach tau.  The k-th best of ANY subset is a lower bound of the final k-th best, so nothing
//             below tau can be in the answer;
//   stage s   item ranges growing geometrically (FILTER = true): one fma + one compare against tau_z per element and
//             one vote per four users decide for most elements; the exact test (fp32 sigmoid as an orderable integer
//             against tau, seen-bitmap knock-out) runs only where some lane passes; passing keys go to a per-warp queue
//             in shared memory and get their list slots when the queue is flushed.  After every stage but the last the
//             select tightens tau; the last select emits the answer in the reference's order (score desc, iid desc).
// Keys are 64-bit (orderable(score) << 32 | iid) as everywhere in score.cu.  The novelty filter is a per-user bitmap
// of the user's stored items (built by k_batch_prep from the `seen` CSR): one 32-bit word covers the 32 items a warp
// holds for one user.  A list that overflows its capacity is detected by the select kernel and that user is re-done by
// the exact fallback (score.cu), so the scheme is exact for any data.
//
// Orientation as in umma_loss.cu: MMA M = 128 items on the TMEM lanes, N = 256 users on the TMEM columns; an epilogue
// warp holds 32 consecutive items of one user across its lanes, so one ballot says which of them pass.
#include "umma_common.cuh"
#include "topk_common.cuh"

namespace {

constexpr int SC_EPI_WARPS = 16;
constexpr int SC_THREADS = 64 + 32 * SC_EPI_WARPS;
constexpr int SC_QCAP = 128;                 // entries of an epilogue warp's key queue (flushed when full and per tile)

template <int BN, int KB, int CL>
struct ScoreSmem {
  static constexpr int A_BYTES = BM * KB * 4;
  static constexpr int B_BYTES = (BN / CL) * KB * 4;
  static constexpr int STAGE_BYTES = 2 * A_BYTES + 2 * B_BYTES;
  static constexpr int BAR_BYTES = 256;
  // per epilogue warp and user of its column quarter: (exact threshold, seen word) + the conservative logit threshold
  // (FILTER: two buffers of (seen word, logit threshold) + exact threshold, filled by cp.async one tile ahead; first
  // slice: one buffer of (exact threshold, seen word))
  static constexpr int TAU_BYTES = SC_EPI_WARPS * (BN / 4) * 24;
  static constexpr int QUEUE_BYTES = SC_EPI_WARPS * SC_QCAP * 10; // per epilogue warp: (key, user) waiting for a list slot
  static constexpr int FIXED = 1024 + BAR_BYTES + TAU_BYTES + QUEUE_BYTES;
  static constexpr int FIT = (227 * 1024 - FIXED) / STAGE_BYTES;       // pipeline stages that fit next to the rest
  static constexpr int STAGES = FIT > 5 ? 5 : FIT;
  static constexpr int TOTAL = STAGES * STAGE_BYTES + FIXED;
  static_assert(STAGES >= 2, "score filter: the operand pipeline needs at least two stages");
};

struct ScoreParams {
  int M;                                   // users of this block
  int item_begin, item_end;                // item range of this pass (item_begin % 128 == 0, item_end <= n_items)
  int Kred;                                // hidden (padded to 4)
  const float* bias;                       // b' [n_items]
  const uint32_t* seen_bits; int words_per_row;   // NULL (no novelty filter) or [M][words_per_row]
  const uint32_t* tau_ord;                 // [M] orderable-score threshold per user (0 = take everything)
  const float* tau_z;                      // [M] logit below which no score can reach tau_ord (k_select_lists), or NULL:
                                           // no pre-filter (first slice: every unseen item is listed)
  int32_t* cnt;                            // [M] entries appended so far (may exceed cap: overflow)
  uint64_t* lists; int cap;                // [M][cap]
  int m_tiles, n_tiles;
  float out_scale; const float* out_scale_dev;   // H: accumulator -> logit (undoes the fp16 operand scaling)
  uint32_t wait_ns;                        // sleep between polls of the accumulator-full barrier (epilogue warps)
  int debug;   // DRB_SCORE_DEBUG bit mask (profiling experiments only, results are wrong): 1 = no appends, 2 = no seen
               // bitmap loads, 4 = no MMAs, 8 = nothing passes the logit pre-filter
};

__device__ __forceinline__ float sc_ex2(float x) { float y; asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
__device__ __forceinline__ float sc_rcp(float x) { float y; asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
__device__ __forceinline__ void sc_mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void sc_mbar_arrive_rank(uint32_t bar, uint32_t rank) {
  // relaxed: the arrival only reports completed tcgen05.ld reads (see umma_loss.cu); a cluster-scope release would
  // first drain the warp's outstanding list stores
  asm volatile("mbarrier.arrive.relaxed.cluster.shared::cluster.b64 _, [%0];" ::"r"(mapa_rank(bar, rank)) : "memory");
}

// FILTER = false: first slice, every unseen item is listed (one warp-aggregated atomicAdd per (warp, user) reserves the
// slots).  FILTER = true: later stages, a logit pre-filter and the exact test leave few keys; they go to a per-warp
// queue in shared memory and get their slots when the queue is flushed -- no global round trip inside the tile loop.
template <int BN, int KB, int CL, bool H, bool FILTER>
__global__ void __launch_bounds__(SC_THREADS, 1)
k_umma_score_filter(const __grid_constant__ CUtensorMap map_a_hi, const __grid_constant__ CUtensorMap map_a_lo,
                    const __grid_constant__ CUtensorMap map_b_hi, const __grid_constant__ CUtensorMap map_b_lo,
                    ScoreParams p) {
  using S = ScoreSmem<BN, KB, CL>;
  constexpr int BK = H ? 2 * KB : KB;            // elements of the hidden dimension per stage (KB: 4-byte units)
  constexpr int UK = H ? 16 : UMMA_K;            // elements one MMA consumes
  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw = smem_u32(smem_raw);
  const uint32_t base = (raw + 1023u) & ~1023u;
  const uint32_t bars = base + S::STAGES * S::STAGE_BYTES;
  auto full_bar = [&](int s) { return bars + 8u * s; };
  auto empty_bar = [&](int s) { return bars + 8u * (S::STAGES + s); };
  auto tfull_bar = [&](int a) { return bars + 8u * (2 * S::STAGES + a); };
  auto tempty_bar = [&](int a) { return bars + 8u * (2 * S::STAGES + 2 + a); };
  const uint32_t tmem_ptr_addr = bars + 8u * (2 * S::STAGES + 4);
  volatile uint32_t* tmem_ptr_generic = reinterpret_cast<volatile uint32_t*>(smem_raw + (tmem_ptr_addr - raw));
  uint2* tau_smem = reinterpret_cast<uint2*>(smem_raw + (bars + S::BAR_BYTES - raw));
  uint32_t* tord_smem = reinterpret_cast<uint32_t*>(tau_smem + 2 * SC_EPI_WARPS * (BN / 4));   // [warp][2][CW]
  uint64_t* q_smem = reinterpret_cast<uint64_t*>(tord_smem + 2 * SC_EPI_WARPS * (BN / 4));

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int nkb = (p.Kred + BK - 1) / BK;
  const uint32_t cta_rank = (CL > 1) ? cluster_ctarank() : 0u;
  const bool leader = cta_rank == 0;
  const int unit0 = blockIdx.x / CL, unit_stride = gridDim.x / CL;
  const int n_units = ((p.m_tiles + CL - 1) / CL) * p.n_tiles;
  auto unit_item0 = [&](int u) { return p.item_begin + ((u / p.n_tiles) * CL + (int)cta_rank) * BM; };
  auto unit_row0 = [&](int u) { return (u % p.n_tiles) * BN; };
  constexpr uint32_t TMEM_COLS = (2 * BN <= 64) ? 64 : (2 * BN <= 128) ? 128 : (2 * BN <= 256) ? 256 : 512;

  if (threadIdx.x == 0) {
    for (int s = 0; s < S::STAGES; s++) {
      mbar_init(full_bar(s), 1);
      mbar_init(empty_bar(s), 1);
    }
    for (int a = 0; a < 2; a++) {
      mbar_init(tfull_bar(a), 1);
      mbar_init(tempty_bar(a), CL * SC_EPI_WARPS);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {
    if (CL > 1) {
      asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tmem_ptr_addr), "r"(TMEM_COLS));
      asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;");
    } else {
      asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tmem_ptr_addr), "r"(TMEM_COLS));
      asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
    }
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  if (CL > 1) cluster_sync_all(); else __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem_base = *tmem_ptr_generic;

  if (warp == 0) {
    // ------------------------------------------------------------------ TMA producer (runs ahead across tiles)
    if (lane == 0) {
      int it = 0;
      for (int t = unit0; t < n_units; t += unit_stride) {
        const int i0 = unit_item0(t), r0 = unit_row0(t);
        for (int kb = 0; kb < nkb; kb++, it++) {
          const int s = it % S::STAGES;
          const uint32_t ph = (it / S::STAGES) & 1;
          mbar_wait(empty_bar(s), ph ^ 1);
          const uint32_t sa_hi = base + s * S::STAGE_BYTES, sa_lo = sa_hi + S::A_BYTES;
          const uint32_t sb_hi = sa_lo + S::A_BYTES, sb_lo = sb_hi + S::B_BYTES;
          if (CL > 1) {
            if (leader) mbar_expect_tx(full_bar(s), CL * S::STAGE_BYTES);
            const uint32_t fb = mapa_rank(full_bar(s), 0);
            const int rh = r0 + (int)cta_rank * (BN / CL);
            tma_load_2d_pair(sa_hi, &map_a_hi, fb, kb * BK, i0);
            tma_load_2d_pair(sa_lo, &map_a_lo, fb, kb * BK, i0);
            tma_load_2d_pair(sb_hi, &map_b_hi, fb, kb * BK, rh);
            tma_load_2d_pair(sb_lo, &map_b_lo, fb, kb * BK, rh);
          } else {
            mbar_expect_tx(full_bar(s), S::STAGE_BYTES);
            tma_load_2d(sa_hi, &map_a_hi, full_bar(s), kb * BK, i0);
            tma_load_2d(sa_lo, &map_a_lo, full_bar(s), kb * BK, i0);
            tma_load_2d(sb_hi, &map_b_hi, full_bar(s), kb * BK, r0);
            tma_load_2d(sb_lo, &map_b_lo, full_bar(s), kb * BK, r0);
          }
        }
      }
    }
  } else if (warp == 1) {
    // ------------------------------------------------------------------ MMA issuer
    if (lane == 0 && leader) {
      const uint32_t idesc = make_idesc<H>(BM * CL, BN);
      int it = 0, tl = 0;
      for (int t = unit0; t < n_units; t += unit_stride, tl++) {
        const int as = tl & 1;
        mbar_wait(tempty_bar(as), ((tl >> 1) & 1) ^ 1);
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        const uint32_t tacc = tmem_base + (uint32_t)(as * BN);
        for (int kb = 0; kb < nkb; kb++, it++) {
          const int s = it % S::STAGES;
          mbar_wait(full_bar(s), (it / S::STAGES) & 1);
          asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
          const uint32_t sa_hi = base + s * S::STAGE_BYTES, sa_lo = sa_hi + S::A_BYTES;
          const uint32_t sb_hi = sa_lo + S::A_BYTES, sb_lo = sb_hi + S::B_BYTES;
          // the last k-block holds fewer than BK real columns: the MMAs over the zero-filled rest are not issued
          const int kk_n = (p.debug & 4) ? 0 : min(BK / UK, (p.Kred - kb * BK + UK - 1) / UK);
#pragma unroll
          for (int kk = 0; kk < BK / UK; kk++) {
            if (kk >= kk_n) break;
            const uint64_t a_hi = make_desc_kmajor<KB>(sa_hi, kk), a_lo = make_desc_kmajor<KB>(sa_lo, kk);
            const uint64_t b_hi = make_desc_kmajor<KB>(sb_hi, kk), b_lo = make_desc_kmajor<KB>(sb_lo, kk);
            umma_split<H, CL>(tacc, a_lo, b_hi, idesc, (kb | kk) != 0);
            umma_split<H, CL>(tacc, a_hi, b_lo, idesc, 1u);
            umma_split<H, CL>(tacc, a_hi, b_hi, idesc, 1u);
          }
          if (CL > 1) umma_commit_pair(empty_bar(s));
          else umma_commit(empty_bar(s));
        }
        if (CL > 1) umma_commit_pair(tfull_bar(as));
        else umma_commit(tfull_bar(as));
      }
    }
  } else {
    // ------------------------------------------------------------------ epilogue warps 2..17
    // TMEM lane = item, column = user.  Warp w reads lanes 32*(w&3)..+31 (its sub-partition) = one 32-item block and the
    // column quarter (w-2)/4 of the tile: for one user the 32 lanes of a warp hold 32 consecutive items.
    const int q = warp & 3, cq = (warp - 2) >> 2;
    constexpr int CW = BN / 4;                    // users of this warp per tile
    // first slice: my_tau[c] = (exact threshold, seen word) of user c of the warp's column quarter, fetched in place.
    // FILTER: my_sz[buf][c] = (seen word, logit threshold); the next tile's values arrive by cp.async while this tile is
    // processed (no registers are held across the tile, nothing is waited for inside the loop); my_tord[buf][c] = the
    // exact threshold, used on the slow path only.
    uint2* my_tau = tau_smem + (warp - 2) * 2 * CW;
    uint32_t* my_tord = tord_smem + (warp - 2) * 2 * CW;
    uint64_t* my_q = q_smem + (warp - 2) * SC_QCAP;                 // queued keys ...
    unsigned short* my_qu = reinterpret_cast<unsigned short*>(q_smem + SC_EPI_WARPS * SC_QCAP) + (warp - 2) * SC_QCAP;  // ... and their users
    const uint32_t lt_mask = (1u << lane) - 1u;
    const float osc = H ? p.out_scale * (p.out_scale_dev ? __ldg(p.out_scale_dev) : 1.0f) : 1.0f;
    float nbias;
    auto fetch_users = [&](int t, int i, uint2* v) {   // first slice: user lane + 32 i of the warp's quarter in unit t
      const int row = unit_row0(t) + cq * CW + lane + 32 * i;
      const int ib = (unit_item0(t) >> 5) + q;     // 32-item block of this warp == word of the seen bitmap
      *v = make_uint2(0xffffffffu, 0u);
      if (t < n_units && row < p.M) {
        v->x = __ldg(p.tau_ord + row);
        if (p.seen_bits && !(p.debug & 2) && ib < p.words_per_row)
          v->y = __ldg(p.seen_bits + (int64_t)row * p.words_per_row + ib);
      }
    };
    auto prefetch_users = [&](int t, int buf) {        // FILTER: (seen word, logit threshold) of unit t into buffer buf
      const int ib = (unit_item0(t) >> 5) + q;
#pragma unroll
      for (int i = 0; i < CW / 32; i++) {
        const int c = lane + 32 * i, row = unit_row0(t) + cq * CW + c;
        uint2* dst = my_tau + buf * CW + c;
        const uint32_t d32 = smem_u32(dst);
        if (t < n_units && row < p.M && !(p.debug & 8)) {
          if (p.seen_bits && !(p.debug & 2) && ib < p.words_per_row)
            asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(d32), "l"(p.seen_bits + (int64_t)row * p.words_per_row + ib) : "memory");
          else
            dst->x = 0u;
          asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(d32 + 4u), "l"(p.tau_z + row) : "memory");
          asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(smem_u32(my_tord + buf * CW + c)), "l"(p.tau_ord + row) : "memory");
        } else {
          *dst = make_uint2(0u, 0x7f800000u);          // users beyond the block never pass
          my_tord[buf * CW + c] = 0xffffffffu;
        }
      }
      asm volatile("cp.async.commit_group;" ::: "memory");
    };
    auto fetch_consts = [&](int t) {
      const int item = unit_item0(t) + q * 32 + lane;
      nbias = (t < n_units && item < p.item_end) ? __ldg(p.bias + item) : 0.f;
    };
    fetch_consts(unit0);
    if (FILTER) prefetch_users(unit0, 0);
    int qn = 0;                                    // entries in the queue (warp-uniform); it lives across tiles and is
    auto flush_queue = [&]() {                     // flushed when the next row of keys would not fit, and at the end
      flush_key_queue<SC_QCAP>(my_q, my_qu, qn, p.cnt, p.lists, p.cap);
      qn = 0;
    };
    int tl = 0;
    for (int t = unit0; t < n_units; t += unit_stride, tl++) {
      const int i0 = unit_item0(t), r0 = unit_row0(t);
      const int as = tl & 1;
      const int item = i0 + q * 32 + lane;
      const bool item_ok = item < p.item_end;
      const float bias = nbias;
      __syncwarp();
      const uint2* cur_sz = my_tau + (tl & 1) * CW;      // FILTER: this tile's (seen word, logit threshold) ...
      const uint32_t* cur_tord = my_tord + (tl & 1) * CW;   // ... and exact thresholds
      if (FILTER) {
        asm volatile("cp.async.wait_group 0;" ::: "memory");
        __syncwarp();
        prefetch_users(t + unit_stride, (tl & 1) ^ 1);
      } else {                                     // the short first slice fetches in place
#pragma unroll
        for (int i = 0; i < CW / 32; i++) {
          uint2 v;
          fetch_users(t, i, &v);
          my_tau[lane + 32 * i] = v;
        }
        __syncwarp();
      }
      fetch_consts(t + unit_stride);
      mbar_wait_sleep(tfull_bar(as), (tl >> 1) & 1, p.wait_ns);
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
      const uint32_t tbase = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(as * BN + cq * CW);
      uint32_t rn[16];
      tmem_ld16_issue(tbase, rn);
#pragma unroll 1
      for (int cl = 0; cl < CW; cl += 16) {
        const int row = r0 + cq * CW + cl;        // first of this chunk's 16 users
        uint32_t r[16];
        tmem_ld16_wait(rn);
#pragma unroll
        for (int j = 0; j < 16; j++) r[j] = rn[j];
        if (cl + 16 < CW) tmem_ld16_issue(tbase + cl + 16, rn);
        if (FILTER) {
          // Pre-filter on the logit: one fma and one compare per element, one vote per four users.  The exact test --
          // the fp32 sigmoid value as an orderable integer against the user's threshold, the seen-bitmap knock-out --
          // runs only for groups of four (user, 32-item) rows in which some lane passes, the four sigmoid chains side
          // by side; the keys that really pass are queued.
#pragma unroll
          for (int j4 = 0; j4 < 16; j4 += 4) {
            const uint4 sz01 = *reinterpret_cast<const uint4*>(cur_sz + cl + j4);     // broadcast reads: (seen, tz) x 4
            const uint4 sz23 = *reinterpret_cast<const uint4*>(cur_sz + cl + j4 + 2);
            const float tz[4] = {__uint_as_float(sz01.y), __uint_as_float(sz01.w), __uint_as_float(sz23.y),
                                 __uint_as_float(sz23.w)};
            const uint32_t seen[4] = {sz01.x, sz01.z, sz23.x, sz23.z};
            float z[4];
            bool anyf = false;
#pragma unroll
            for (int jj = 0; jj < 4; jj++) {
              z[jj] = H ? fmaf(__uint_as_float(r[j4 + jj]), osc, bias) : __uint_as_float(r[j4 + jj]) + bias;
              anyf |= z[jj] >= tz[jj];
            }
            if (!__any_sync(0xffffffffu, anyf)) continue;
            uint32_t ord[4], bal[4];
#pragma unroll
            for (int jj = 0; jj < 4; jj++) {
              const float pr = sc_rcp(1.0f + sc_ex2(z[jj] * -1.4426950408889634f));   // sigmoid, > 0
              ord[jj] = __float_as_uint(pr) | 0x80000000u;                            // f2ord of a non-negative float
            }
#pragma unroll
            for (int jj = 0; jj < 4; jj++) {
              const uint32_t tau = cur_tord[cl + j4 + jj];                            // broadcast read
              const bool pass = item_ok && !((seen[jj] >> lane) & 1u) && (ord[jj] >= tau) && !(p.debug & 1);
              bal[jj] = __ballot_sync(0xffffffffu, pass);
            }
#pragma unroll
            for (int jj = 0; jj < 4; jj++) {
              if (bal[jj] != 0u) {                 // warp-uniform
                const int n = __popc(bal[jj]);
                if (qn + n > SC_QCAP) flush_queue();
                if ((bal[jj] >> lane) & 1u) {
                  const int e = qn + __popc(bal[jj] & lt_mask);
                  my_q[e] = ((uint64_t)ord[jj] << 32) | (uint32_t)item;
                  my_qu[e] = (unsigned short)(row + j4 + jj);
                }
                qn += n;
              }
            }
          }
          continue;
        }
        uint32_t bal[16];
        // 1. score, knock-out, threshold test: r[j] becomes the orderable score, bal[j] the lanes that pass for user j
#pragma unroll
        for (int j = 0; j < 16; j++) {
          const float z = H ? fmaf(__uint_as_float(r[j]), osc, bias) : __uint_as_float(r[j]) + bias;
          const float pr = sc_rcp(1.0f + sc_ex2(z * -1.4426950408889634f));         // sigmoid, > 0
          const uint32_t ord = __float_as_uint(pr) | 0x80000000u;                   // f2ord of a non-negative float
          const uint2 ts = my_tau[cl + j];                                          // broadcast read
          const bool pass = item_ok && (row + j < p.M) && !((ts.y >> lane) & 1u) && (ord >= ts.x);
          r[j] = ord;
          bal[j] = (p.debug & 1) ? 0u : __ballot_sync(0xffffffffu, pass);
        }
        // 2. one atomicAdd per (warp, user) reserves the slots of the passing lanes (all issued before any is consumed)
        int slot[16];
#pragma unroll
        for (int j = 0; j < 16; j++) {
          slot[j] = 0;
          if (bal[j] != 0u && lane == 0) slot[j] = atomicAdd(p.cnt + row + j, __popc(bal[j]));
        }
        // 3. append
#pragma unroll
        for (int j = 0; j < 16; j++) {
          if (bal[j] != 0u) {                      // warp-uniform
            const int b0 = __shfl_sync(0xffffffffu, slot[j], 0);
            if ((bal[j] >> lane) & 1u) {
              const int pos = b0 + __popc(bal[j] & lt_mask);
              if (pos < p.cap) p.lists[(int64_t)(row + j) * p.cap + pos] = ((uint64_t)r[j] << 32) | (uint32_t)item;
            }
          }
        }
      }
      asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
      __syncwarp();
      if (lane == 0) {
        if (CL > 1) sc_mbar_arrive_rank(tempty_bar(as), 0);
        else sc_mbar_arrive(tempty_bar(as));
      }
    }
    if (FILTER && qn > 0) flush_queue();
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  if (CL > 1) cluster_sync_all(); else __syncthreads();
  if (warp == 1) {
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    if (CL > 1) asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(TMEM_COLS));
    else asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(TMEM_COLS));
  }
}

template <int BN, int KB, int CL, bool H, bool FILTER>
int run_score(drb_ctx* ctx, const UmmaOperands& o, ScoreParams p, int n_items) {
  CUtensorMap ma_hi, ma_lo, mb_hi, mb_lo;
  int r;
  // A (M side, TMEM lanes) = W' rows = items; B (N side, TMEM columns) = h rows = users.  Rows past the end of either
  // matrix read as zeros (TMA out-of-bounds fill) and are masked in the epilogue.
  if ((r = make_operand_map<H>(&ma_hi, o.b_hi, p.Kred, n_items, o.ldb, KB, BM))) return r;
  if ((r = make_operand_map<H>(&ma_lo, o.b_lo, p.Kred, n_items, o.ldb, KB, BM))) return r;
  if ((r = make_operand_map<H>(&mb_hi, o.a_hi, p.Kred, p.M, o.lda, KB, BN / CL))) return r;
  if ((r = make_operand_map<H>(&mb_lo, o.a_lo, p.Kred, p.M, o.lda, KB, BN / CL))) return r;
  p.m_tiles = (p.item_end - p.item_begin + BM - 1) / BM;
  p.n_tiles = (p.M + BN - 1) / BN;
  auto kern = k_umma_score_filter<BN, KB, CL, H, FILTER>;
  constexpr int SMEM = ScoreSmem<BN, KB, CL>::TOTAL;
  static bool attr_set = false;
  static int max_clusters = 0;
  if (!attr_set) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM);
    if (e != cudaSuccess)
      return drb_fail(DRB_E_CUDA, "cudaFuncSetAttribute(smem=%d) failed: %s", SMEM, cudaGetErrorString(e));
    if (CL > 1) {
      cudaLaunchConfig_t qc{};
      cudaLaunchAttribute qa[1];
      qa[0].id = cudaLaunchAttributeClusterDimension;
      qa[0].val.clusterDim.x = CL; qa[0].val.clusterDim.y = 1; qa[0].val.clusterDim.z = 1;
      qc.gridDim = dim3(ctx->sm_count / CL * CL); qc.blockDim = dim3(SC_THREADS); qc.dynamicSmemBytes = SMEM;
      qc.attrs = qa; qc.numAttrs = 1;
      e = cudaOccupancyMaxActiveClusters(&max_clusters, kern, &qc);
      if (e != cudaSuccess || max_clusters < 1)
        return drb_fail(DRB_E_CUDA, "cudaOccupancyMaxActiveClusters failed: %s", cudaGetErrorString(e));
    }
    attr_set = true;
  }
  const int n_units = ((p.m_tiles + CL - 1) / CL) * p.n_tiles;
  if (n_units <= 0) return DRB_OK;
  const int grid = CL * std::min(n_units, CL > 1 ? max_clusters : ctx->sm_count);
  drb_prof_scope prof_(ctx, p.item_begin == 0 ? "k_umma_score_filter_slice" : "k_umma_score_filter_rest");
  if (CL > 1) {
    cudaLaunchConfig_t cfg{};
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = CL; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
    cfg.gridDim = dim3(grid); cfg.blockDim = dim3(SC_THREADS); cfg.dynamicSmemBytes = SMEM; cfg.stream = ctx->stream;
    cfg.attrs = at; cfg.numAttrs = 1;
    cudaError_t e = cudaLaunchKernelEx(&cfg, kern, ma_hi, ma_lo, mb_hi, mb_lo, p);
    if (e != cudaSuccess) return drb_fail(DRB_E_CUDA, "cluster launch of k_umma_score_filter failed: %s", cudaGetErrorString(e));
  } else {
    kern<<<grid, SC_THREADS, SMEM, ctx->stream>>>(ma_hi, ma_lo, mb_hi, mb_lo, p);
  }
  DRB_LAUNCH_CHECK(ctx, "k_umma_score_filter");
  return DRB_OK;
}

}  // namespace

int launch_umma_score_filter(drb_ctx* ctx, const UmmaOperands& o, int n_users, int n_items, int item_begin, int item_end,
                             int Kred, const float* bias, const uint32_t* seen_bits, int words_per_row,
                             const uint32_t* tau_ord, const float* tau_z, int32_t* cnt, uint64_t* lists, int cap) {
  if (item_begin % 128 != 0 || item_end > n_items || item_begin >= item_end)
    return drb_fail(DRB_E_INVALID, "score_filter: bad item range [%d, %d) of %d", item_begin, item_end, n_items);
  ScoreParams p{};
  p.M = n_users; p.item_begin = item_begin; p.item_end = item_end; p.Kred = Kred; p.bias = bias;
  p.seen_bits = seen_bits; p.words_per_row = words_per_row; p.tau_ord = tau_ord; p.tau_z = tau_z; p.cnt = cnt; p.lists = lists; p.cap = cap;
  p.debug = getenv("DRB_SCORE_DEBUG") ? atoi(getenv("DRB_SCORE_DEBUG")) : 0;
  p.wait_ns = getenv("DRB_WAIT_NS") ? (uint32_t)atoi(getenv("DRB_WAIT_NS")) : 100u;
  p.out_scale = o.out_scale; p.out_scale_dev = o.out_scale_dev;
  if (n_users > 65536) return drb_fail(DRB_E_INVALID, "score_filter: at most 65536 users per block");
  static const int kb_env = getenv("DRB_SCORE_KB") ? atoi(getenv("DRB_SCORE_KB")) : 32;
#define DRB_SCORE_CASE(F_)                                                             \
  {                                                                                    \
    if (o.half) {                                                                      \
      if (n_users > 128) {                                                             \
        /* DRB_SCORE_KB=16: five 32 KB stages instead of two 64 KB ones (measured slower) */ \
        if (kb_env == 16) return run_score<256, 16, 2, true, F_>(ctx, o, p, n_items);  \
        return run_score<256, 32, 2, true, F_>(ctx, o, p, n_items);                    \
      }                                                                                \
      return run_score<128, 32, 1, true, F_>(ctx, o, p, n_items);                      \
    }                                                                                  \
    if (n_users > 128) return run_score<256, 32, 2, false, F_>(ctx, o, p, n_items);    \
    return run_score<128, 32, 1, false, F_>(ctx, o, p, n_items);                       \
  }
  if (tau_z) DRB_SCORE_CASE(true)
  DRB_SCORE_CASE(false)
#undef DRB_SCORE_CASE
}
