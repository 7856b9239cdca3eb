// K6 scoring (sm_100a): candidate dot products + in-CTA ordering, and full-catalog top-k selection.
//
// Replaces (reference, DRecPy/): Recommender/cdae.py:90-103 (_rank: full forward, filter to the candidate set
// minus the user's training items when novelty, heapq.nlargest over (score, iid) tuples),
// Recommender/recommender_abc.py:454-461 (DMF: one _predict per candidate, then nlargest) and :413-419
// (_recommend = _rank over range(n_items)).
// Total order reproduced exactly: (score, iid) compared lexicographically, largest first, duplicates of the
// same candidate collapsed (the reference builds a set).  Scores are ordered through a monotone float->uint map
// packed with the item id into one 64-bit key, so ties on the score are broken by the larger item id.
#include "topk_common.cuh"

namespace {

__device__ __forceinline__ bool row_contains(const int32_t* lo, int n, int32_t x) {
  int a = 0, b = n;
  while (a < b) {
    const int mid = (a + b) >> 1;
    if (lo[mid] < x) a = mid + 1; else b = mid;
  }
  return a < n && lo[a] == x;
}

struct SelectState { uint32_t prefix; int need; int bucket_count; };

// descending bitonic sort of P (power of two) 64-bit keys in shared memory
__device__ void bitonic_desc(uint64_t* keys, int P) {
  for (int k = 2; k <= P; k <<= 1) {
    for (int j = k >> 1; j > 0; j >>= 1) {
      for (int i = threadIdx.x; i < P; i += blockDim.x) {
        const int ixj = i ^ j;
        if (ixj > i) {
          const uint64_t a = keys[i], b = keys[ixj];
          const bool desc = ((i & k) == 0);
          if (desc ? (a < b) : (a > b)) { keys[i] = b; keys[ixj] = a; }
        }
      }
      __syncthreads();
    }
  }
}

// write keys[0..P) (sorted descending; 0 = invalid) without duplicates; executed by warp 0
__device__ void emit_sorted(const uint64_t* keys, int P, int limit, int32_t* out_iid, float* out_score,
                            int32_t* n_out) {
  if (threadIdx.x >= 32) return;
  const int lane = threadIdx.x;
  int running = 0;
  for (int base = 0; base < P; base += 32) {
    const int i = base + lane;
    const uint64_t k = keys[i];
    const bool flag = (k != 0) && (i == 0 || keys[i - 1] != k);
    const uint32_t mask = __ballot_sync(0xffffffffu, flag);
    const int pos = running + __popc(mask & ((1u << lane) - 1u));
    if (flag && pos < limit) {
      out_iid[pos] = (int32_t)(uint32_t)(k & 0xffffffffu);
      out_score[pos] = ord2f((uint32_t)(k >> 32));
    }
    running += __popc(mask);
  }
  if (lane == 0) *n_out = min(running, limit);
}

// keys_global == NULL: the P keys of a user live in shared memory (P <= 4096, 128 threads); otherwise in the caller's
// scratch row keys_global[blockIdx.x * P ..) and the same bitonic network runs on global memory with 1024 threads
// (candidate lists as long as the catalog: recommend(n=None), recommender_abc.py:391-419)
__global__ void __launch_bounds__(1024) k_rank_candidates(CandScoreArgs a, int P, uint64_t* keys_global) {
  extern __shared__ uint64_t keys_smem[];  // [P] when keys_global == NULL
  uint64_t* keys = keys_global ? keys_global + (int64_t)blockIdx.x * P : keys_smem;
  const int nwarps = blockDim.x >> 5;
  const int u = blockIdx.x;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int uid = a.uids[u];
  const int cnt = min(a.cand_count[u], a.max_cand);
  const float* ur = a.urep + (int64_t)u * a.ld_u;
  const int32_t* seen = nullptr;
  int nseen = 0;
  if (a.novelty) {
    seen = a.seen_indices + a.seen_indptr[uid];
    nseen = (int)(a.seen_indptr[uid + 1] - a.seen_indptr[uid]);
  }
  for (int i = threadIdx.x; i < P; i += blockDim.x) keys[i] = 0;
  __syncthreads();
  float uss = 0.f;
  if (a.mode == 1) {
    for (int k = lane; k < a.width; k += 32) uss = fmaf(ur[k], ur[k], uss);
    uss = warp_sum(uss);
  }
  for (int c = warp; c < cnt; c += nwarps) {
    const int iid = a.cand[(int64_t)u * a.max_cand + c];
    if (iid < 0) continue;                                       // unknown raw item (skip_invalid_items)
    if (a.novelty && row_contains(seen, nseen, iid)) continue;   // warp-uniform
    const float* tr = a.table + (int64_t)iid * a.ld_t;
    float dot = 0.f, tss = 0.f;
    for (int k = lane; k < a.width; k += 32) {
      const float t = tr[k];
      dot = fmaf(ur[k], t, dot);
      tss = fmaf(t, t, tss);
    }
    dot = warp_sum(dot);
    float score;
    if (a.mode == 0) {
      score = 1.0f / (1.0f + expf(-(dot + (a.bias ? a.bias[iid] : 0.f))));
    } else {
      tss = warp_sum(tss);
      const float c_ = dot * (1.0f / sqrtf(fmaxf(uss, 1e-12f))) * (1.0f / sqrtf(fmaxf(tss, 1e-12f)));
      score = fmaxf(1e-6f, c_);
    }
    if (lane == 0) keys[c] = ((uint64_t)f2ord(score) << 32) | (uint32_t)iid;
  }
  __syncthreads();
  bitonic_desc(keys, P);
  emit_sorted(keys, P, a.max_cand, a.out_iid + (int64_t)u * a.max_cand, a.out_score + (int64_t)u * a.max_cand,
              a.n_out + u);
}

// ---------------------------------------------------------------- full-catalog top-k (radix select + sort)
constexpr int kTopkThreads = 256;


// one MSB-first 8-bit radix pass over `value(i)` for elements accepted by `live(i)`
template <typename KeyFn>
__device__ void radix_pass(int n, int shift, uint32_t prefix_mask, uint32_t prefix, KeyFn key, int* hist,
                           SelectState* st) {
  for (int i = threadIdx.x; i < 256; i += blockDim.x) hist[i] = 0;
  __syncthreads();
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    uint32_t k;
    if (key(i, &k) && (k & prefix_mask) == prefix) atomicAdd(&hist[(k >> shift) & 0xff], 1);
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    int need = st->need, d = 255;
    for (; d > 0; d--) {
      if (hist[d] >= need) break;
      need -= hist[d];
    }
    st->need = need;                       // rank wanted inside bucket d
    st->bucket_count = hist[d];
    st->prefix = prefix | ((uint32_t)d << shift);
  }
  __syncthreads();
}

__global__ void __launch_bounds__(kTopkThreads) k_topk(TopkArgs a, int P) {
  extern __shared__ uint64_t keys[];  // [P] selected keys
  __shared__ int hist[256];
  __shared__ SelectState st;
  __shared__ int n_sel;
  // direct: block b ranks score row b for user b.  Indirect (the exact fallback of the tensor-core path): block b ranks
  // score row b for user fb_users[b], for the first *fb_count rows only.
  int u = blockIdx.x;
  if (a.fb_users) {
    if (u >= min(*a.fb_count, a.fb_max)) return;
    u = a.fb_users[blockIdx.x];
  }
  const int uid = a.uids[u];
  // the score row is scratch: knock out the user's training items (cdae.py:93-98) in place
  float* row = const_cast<float*>(a.scores) + (int64_t)blockIdx.x * a.ld;
  if (a.novelty) {
    const int64_t lo = a.seen_indptr[uid], hi = a.seen_indptr[uid + 1];
    for (int64_t j = lo + threadIdx.x; j < hi; j += blockDim.x) row[a.seen_indices[j]] = -INFINITY;
  }
  for (int i = threadIdx.x; i < P; i += blockDim.x) keys[i] = 0;
  __syncthreads();
  const uint32_t dead = f2ord(-INFINITY);
  // number of live items
  if (threadIdx.x == 0) { st.need = 0; n_sel = 0; }
  __syncthreads();
  int live = 0;
  for (int i = threadIdx.x; i < a.n_items; i += blockDim.x) live += (f2ord(row[i]) != dead);
  atomicAdd(&st.need, live);
  __syncthreads();
  const int n_live = st.need;
  const int k = min(a.k, n_live);
  __syncthreads();
  if (k == 0) {
    if (threadIdx.x == 0) a.n_out[u] = 0;
    return;
  }
  auto score_key = [&](int i, uint32_t* out) { *out = f2ord(row[i]); return *out != dead; };
  uint32_t t32;
  int need_eq, count_eq;
  if (k == n_live) {           // everything live is selected
    t32 = 0; need_eq = 0; count_eq = 0;
  } else {
    if (threadIdx.x == 0) { st.need = k; st.prefix = 0; }
    __syncthreads();
    uint32_t pm = 0;
    for (int shift = 24; shift >= 0; shift -= 8) {
      radix_pass(a.n_items, shift, pm, st.prefix, score_key, hist, &st);
      pm |= 0xffu << shift;
    }
    t32 = st.prefix; need_eq = st.need; count_eq = st.bucket_count;
  }
  // ties on the threshold score: keep the need_eq largest item ids
  uint32_t tiid = 0;
  if (k != n_live && need_eq < count_eq) {
    __syncthreads();
    if (threadIdx.x == 0) { st.need = need_eq; st.prefix = 0; }
    __syncthreads();
    auto iid_key = [&](int i, uint32_t* out) { *out = (uint32_t)i; return f2ord(row[i]) == t32; };
    uint32_t pm = 0;
    for (int shift = 24; shift >= 0; shift -= 8) {
      radix_pass(a.n_items, shift, pm, st.prefix, iid_key, hist, &st);
      pm |= 0xffu << shift;
    }
    tiid = st.prefix;
  }
  __syncthreads();
  for (int i = threadIdx.x; i < a.n_items; i += blockDim.x) {
    const uint32_t o = f2ord(row[i]);
    if (o == dead) continue;
    const bool take = (k == n_live) || (o > t32) || (o == t32 && (uint32_t)i >= tiid);
    if (take) {
      const int pos = atomicAdd(&n_sel, 1);
      if (pos < P) keys[pos] = ((uint64_t)o << 32) | (uint32_t)i;
    }
  }
  __syncthreads();
  bitonic_desc(keys, P);
  emit_sorted(keys, P, a.k, a.out_iid + (int64_t)u * a.k, a.out_score + (int64_t)u * a.k, a.n_out + u);
}


// ---------------------------------------------------------------- candidate lists of the tensor-core top-k (umma_score.cu)
// Finds, among hist[0..256), the largest digit d with sum_{b >= d} hist[b] >= need (need >= 1, total >= need).
// Executed by warp 0; results through `st` (need = rank wanted inside bucket d, bucket_count = hist[d]).
__device__ __forceinline__ void pick_digit_warp(const int* hist, uint32_t prefix, int shift, SelectState* st) {
  const int lane = threadIdx.x & 31;
  int local = 0;
#pragma unroll
  for (int b = 0; b < 8; b++) local += hist[lane * 8 + b];
  int v = local;                                   // inclusive suffix sum over lanes >= lane
#pragma unroll
  for (int off = 1; off < 32; off <<= 1) {
    const int t = __shfl_down_sync(0xffffffffu, v, off);
    if (lane + off < 32) v += t;
  }
  const int need = st->need;
  const uint32_t ge = __ballot_sync(0xffffffffu, v >= need);
  const int L = 31 - __clz(ge);                    // v decreases with the lane: the last lane that still reaches `need`
  if (lane == L) {
    int rem = need - (v - local), d = lane * 8 + 7;
    for (; d > lane * 8; d--) {
      if (hist[d] >= rem) break;
      rem -= hist[d];
    }
    st->need = rem;
    st->bucket_count = hist[d];
    st->prefix = prefix | ((uint32_t)d << shift);
  }
}

// k-th largest (need = k) of the 32-bit values value(i), i < n, accepted by the functor: 4 MSB-first 8-bit passes over
// shared-memory keys.  On return st->prefix = that value, st->need = how many of the values equal to it belong to the
// top `need`, st->bucket_count = how many values equal it.  All threads of the CTA call it.
template <typename KeyFn>
__device__ void radix_select_u32(int n, int need, KeyFn key, int* hist, SelectState* st) {
  if (threadIdx.x == 0) { st->need = need; st->prefix = 0; }
  __syncthreads();
  uint32_t pm = 0;
  for (int shift = 24; shift >= 0; shift -= 8) {
    for (int i = threadIdx.x; i < 256; i += blockDim.x) hist[i] = 0;
    __syncthreads();
    const uint32_t prefix = st->prefix;
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
      uint32_t kx;
      if (key(i, &kx) && (kx & pm) == prefix) atomicAdd(&hist[(kx >> shift) & 0xff], 1);
    }
    __syncthreads();
    if (threadIdx.x < 32) pick_digit_warp(hist, prefix, shift, st);
    __syncthreads();
    pm |= 0xffu << shift;
  }
}

// The score filter (umma_score.cu) forms a score as rcp.approx(1 + ex2.approx(z * -log2 e)) and lists it when its
// orderable value reaches tau.  This returns a logit below which that cannot happen, so that the filter can discard
// most elements on the logit alone: the approximate sigmoid is within 2^-17 relative of the true one wherever it is
// not saturated (ex2.approx 2^-22, rcp.approx 2^-23, the rounded exponent argument |arg| * 2^-24 * ln 2 for |arg| up
// to 126), the bound takes 2^-16 and rounds the logit down.
__device__ __forceinline__ float logit_lower_bound(uint32_t tau_ord) {
  const float pt = __uint_as_float(tau_ord & 0x7fffffffu);      // scores are positive: ord = bits | 0x80000000
  if (!(pt > 0.f)) return __int_as_float(0xff800000);
  const double pp = (double)fminf(pt, 1.0f) * (1.0 - 1.0 / 65536.0);
  const float z = (float)log(pp / (1.0 - pp));
  return z - 1e-5f * fabsf(z) - 1e-6f;
}

// One CTA per user over the user's list of 64-bit keys (orderable score << 32 | iid), copied to shared memory once.
//   final == 0 (after a filter stage that is not the last): radix-selects tau = the k-th best score, keeps the keys
//               >= tau at the head of the list (unordered) and publishes tau and its logit bound (0 / -inf while fewer
//               than k exist: the next stage takes everything);
//   final != 0: radix-selects the k best keys -- score first, item id among equal scores, i.e. heapq.nlargest on
//               (score, iid) tuples (cdae.py:102-103) -- sorts those k and emits them.
// A list that overflowed its capacity marks the user (n_out = -1) for the exact fallback.
// Two launches share the code: lists are a few hundred keys long almost always, so the first launch runs 64 threads per
// user with shared memory for sm_cap = 1024 keys (32 users resident per SM instead of 7) and only records users with
// longer lists; the second is a small persistent grid of 256-thread CTAs with room for `cap` keys over those users.
struct SelectArgs {
  uint64_t* lists; int cap; int32_t* cnt; uint32_t* tau_ord; float* tau_z; int k; int final; int P;
  int32_t* out_iid; float* out_score; int32_t* n_out; int32_t* fb_users; int32_t* fb_count; int fb_max;
  int sm_cap; int32_t* big_users; int32_t* big_count; int big_pass;
};

__device__ void select_user(const SelectArgs& a, int u, int c, uint64_t* sm_keys, int* hist, SelectState* st, int* n_sel) {
  uint64_t* list = a.lists + (int64_t)u * a.cap;
  const int k = a.k;
  if (c > a.cap) {                  // overflow: the list is incomplete, this user goes through the exact fallback
    if (threadIdx.x == 0) {
      if (a.final) {                // claims a scratch row of the exact fallback (k_fallback_scores); beyond fb_max
        a.n_out[u] = -1;            // rows n_out stays -1 and the host re-runs the user
        const int slot = atomicAdd(a.fb_count, 1);
        if (slot < a.fb_max) a.fb_users[slot] = u;
      } else {                      // nothing more is appended for this user; cnt stays > cap
        a.tau_ord[u] = 0xffffffffu; a.tau_z[u] = __int_as_float(0x7f800000);
      }
    }
    return;
  }
  for (int i = threadIdx.x; i < c; i += blockDim.x) sm_keys[i] = list[i];
  if (threadIdx.x == 0) *n_sel = 0;
  __syncthreads();
  auto ord_key = [&](int i, uint32_t* out) { *out = (uint32_t)(sm_keys[i] >> 32); return true; };
  if (!a.final) {
    if (c < k) {                    // fewer than k so far: keep everything, no threshold yet
      if (threadIdx.x == 0) { a.tau_ord[u] = 0u; a.tau_z[u] = __int_as_float(0xff800000); }
      return;
    }
    radix_select_u32(c, k, ord_key, hist, st);
    const uint32_t t32 = st->prefix;
    for (int i = threadIdx.x; i < c; i += blockDim.x) {
      const uint64_t key = sm_keys[i];
      if ((uint32_t)(key >> 32) >= t32) list[atomicAdd(n_sel, 1)] = key;
    }
    __syncthreads();
    if (threadIdx.x == 0) { a.cnt[u] = *n_sel; a.tau_ord[u] = t32; a.tau_z[u] = logit_lower_bound(t32); }
    return;
  }
  const int P = a.P;
  uint64_t* sel = sm_keys + (a.big_pass ? a.cap : a.sm_cap);
  for (int i = threadIdx.x; i < P; i += blockDim.x) sel[i] = 0ull;
  const int kk = min(k, c);
  if (kk == 0) {
    if (threadIdx.x == 0) a.n_out[u] = 0;
    return;
  }
  uint32_t t32 = 0, tiid = 0;
  if (kk < c) {
    radix_select_u32(c, kk, ord_key, hist, st);
    t32 = st->prefix;
    const int need_eq = st->need, count_eq = st->bucket_count;
    __syncthreads();
    if (need_eq < count_eq) {       // ties on the threshold score: the need_eq largest item ids among them
      auto iid_key = [&](int i, uint32_t* out) {
        *out = (uint32_t)(sm_keys[i] & 0xffffffffu);
        return (uint32_t)(sm_keys[i] >> 32) == t32;
      };
      radix_select_u32(c, need_eq, iid_key, hist, st);
      tiid = st->prefix;
    }
  }
  __syncthreads();
  for (int i = threadIdx.x; i < c; i += blockDim.x) {
    const uint64_t key = sm_keys[i];
    const uint32_t o = (uint32_t)(key >> 32), id = (uint32_t)(key & 0xffffffffu);
    if (kk == c || o > t32 || (o == t32 && id >= tiid)) {
      const int pos = atomicAdd(n_sel, 1);
      if (pos < P) sel[pos] = key;
    }
  }
  __syncthreads();
  bitonic_desc(sel, P);
  emit_sorted(sel, P, k, a.out_iid + (int64_t)u * k, a.out_score + (int64_t)u * k, a.n_out + u);
}

__global__ void __launch_bounds__(256) k_select_lists(SelectArgs a, int n_users) {
  extern __shared__ uint64_t sm_keys[];            // [sm_cap | cap] the list, then [P] the selected keys (final)
  __shared__ int hist[256];
  __shared__ SelectState st;
  __shared__ int n_sel;
  if (!a.big_pass) {
    const int u = blockIdx.x;
    const int c = a.cnt[u];
    if (c <= a.cap && c > a.sm_cap) {              // too long for this launch's shared memory: the second launch's
      if (threadIdx.x == 0) a.big_users[atomicAdd(a.big_count, 1)] = u;
      return;
    }
    select_user(a, u, c, sm_keys, hist, &st, &n_sel);
    return;
  }
  const int n = min(*a.big_count, n_users);
  for (int w = blockIdx.x; w < n; w += gridDim.x) {
    const int u = a.big_users[w];
    select_user(a, u, a.cnt[u], sm_keys, hist, &st, &n_sel);
    __syncthreads();
  }
}

// Threshold select (final == 0) for lists of up to 1024 keys, one WARP per user and no shared memory: the 32-bit
// orderable scores sit in registers (SLOTS per lane), the k-th largest is found bit by bit from the top (count the
// keys that match the prefix so far and have the bit set; keep the bit when at least `need` do), then the list is
// re-read and compacted in place to the keys >= tau.  Same results as select_user (the k-th largest value is unique),
// about a third of its time: the CTA form spends its time in __syncthreads and shared-memory histograms.
template <int SLOTS>
__device__ __forceinline__ uint32_t warp_kth_largest(const uint64_t* list, int c, int k, int lane) {
  uint32_t v[SLOTS];
#pragma unroll
  for (int i = 0; i < SLOTS; i++) {
    const int idx = lane + 32 * i;
    v[i] = idx < c ? (uint32_t)(list[idx] >> 32) : 0u;        // valid scores have the top bit set: 0 never counts
  }
  uint32_t prefix = 0u;
  int need = k;
#pragma unroll 1
  for (int bit = 31; bit >= 0; bit--) {
    const uint32_t cand = prefix | (1u << bit), hi = ~((1u << bit) - 1u);
    int n1 = 0;
#pragma unroll
    for (int i = 0; i < SLOTS; i++) n1 += ((v[i] & hi) == cand);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) n1 += __shfl_xor_sync(0xffffffffu, n1, o);
    if (n1 >= need) prefix = cand; else need -= n1;
  }
  return prefix;
}

__global__ void __launch_bounds__(256) k_select_tau_warp(SelectArgs a, int n_users) {
  const int lane = threadIdx.x & 31;
  const int u = blockIdx.x * 8 + (threadIdx.x >> 5);
  if (u >= n_users) return;
  const int c = a.cnt[u];
  uint64_t* list = a.lists + (int64_t)u * a.cap;
  if (c > a.cap) {                  // overflow: nothing more is appended for this user; cnt stays > cap
    if (lane == 0) { a.tau_ord[u] = 0xffffffffu; a.tau_z[u] = __int_as_float(0x7f800000); }
    return;
  }
  if (c > 1024) {                   // too long for the registers: the CTA form (second launch) takes it
    if (lane == 0) a.big_users[atomicAdd(a.big_count, 1)] = u;
    return;
  }
  if (c < a.k) {                    // fewer than k so far: keep everything, no threshold yet
    if (lane == 0) { a.tau_ord[u] = 0u; a.tau_z[u] = __int_as_float(0xff800000); }
    return;
  }
  uint32_t t32;
  if (c <= 256) t32 = warp_kth_largest<8>(list, c, a.k, lane);
  else if (c <= 512) t32 = warp_kth_largest<16>(list, c, a.k, lane);
  else t32 = warp_kth_largest<32>(list, c, a.k, lane);
  // compaction in place: chunk i is read completely before anything is written, and what is kept lands at positions
  // below the chunk's end
  int n_sel = 0;
  for (int i0 = 0; i0 < c; i0 += 32) {
    const int idx = i0 + lane;
    const uint64_t key = idx < c ? list[idx] : 0ull;
    const bool keep = idx < c && (uint32_t)(key >> 32) >= t32;
    const uint32_t m = __ballot_sync(0xffffffffu, keep);
    __syncwarp();
    if (keep) list[n_sel + __popc(m & ((1u << lane) - 1u))] = key;
    n_sel += __popc(m);
    __syncwarp();
  }
  if (lane == 0) { a.cnt[u] = n_sel; a.tau_ord[u] = t32; a.tau_z[u] = logit_lower_bound(t32); }
}

// Exact fallback for users whose candidate list overflowed: fills the user's claimed scratch row with the scores
// sigmoid(h_u . W'_i + b'_i) over the whole catalog (one warp per item, fp32 FMA); k_topk (indirect) then ranks the row.
__global__ void __launch_bounds__(256) k_fallback_scores(const float* h, int ld_h, const float* table, int ld_t,
                                                         const float* bias, int width, int n_items, float* rows,
                                                         int ld_rows, const int32_t* fb_users, const int32_t* fb_count,
                                                         int fb_max) {
  const int slot = blockIdx.x;       // one CTA per claimed scratch row (k_select_lists claims them)
  if (slot >= min(*fb_count, fb_max)) return;
  const int u = fb_users[slot];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const float* ur = h + (int64_t)u * ld_h;
  float* row = rows + (int64_t)slot * ld_rows;
  for (int i = warp; i < n_items; i += 8) {
    const float* tr = table + (int64_t)i * ld_t;
    float dot = 0.f;
    for (int kx = lane; kx < width; kx += 32) dot = fmaf(ur[kx], tr[kx], dot);
    dot = warp_sum(dot);
    if (lane == 0) row[i] = 1.0f / (1.0f + expf(-(dot + bias[i])));
  }
}

int next_pow2(int x) {
  int p = 32;
  while (p < x) p <<= 1;
  return p;
}

}  // namespace

int64_t rank_scratch_rows(int64_t scratch_bytes, int max_cand) {
  return scratch_bytes / ((int64_t)next_pow2(max_cand) * (int64_t)sizeof(uint64_t));
}

int launch_rank_candidates(drb_ctx* ctx, const CandScoreArgs& a, int n, void* scratch, int64_t scratch_bytes) {
  if (n <= 0) return DRB_OK;
  if (a.max_cand < 1) return drb_fail(DRB_E_INVALID, "rank_candidates: max_cand must be >= 1");
  const int P = next_pow2(a.max_cand);
  drb_prof_scope prof_(ctx, "k_rank_candidates");
  if (a.max_cand <= 4096) {
    k_rank_candidates<<<n, 128, (size_t)P * sizeof(uint64_t), ctx->stream>>>(a, P, nullptr);
  } else {
    if (!scratch || rank_scratch_rows(scratch_bytes, a.max_cand) < n)
      return drb_fail(DRB_E_INVALID, "rank_candidates: %d lists of %d candidates need %lld bytes of key scratch", n,
                      a.max_cand, (long long)n * P * 8);
    k_rank_candidates<<<n, 1024, 0, ctx->stream>>>(a, P, static_cast<uint64_t*>(scratch));
  }
  DRB_LAUNCH_CHECK(ctx, "k_rank_candidates");
  return DRB_OK;
}

int launch_topk(drb_ctx* ctx, const TopkArgs& a, int n) {
  if (n <= 0) return DRB_OK;
  if (a.k < 1 || a.k > 2048) return drb_fail(DRB_E_INVALID, "topk: k must be in [1, 2048]");
  const int P = next_pow2(a.k);
  drb_prof_scope prof_(ctx, "k_topk");
  k_topk<<<n, kTopkThreads, (size_t)P * sizeof(uint64_t), ctx->stream>>>(a, P);
  DRB_LAUNCH_CHECK(ctx, "k_topk");
  return DRB_OK;
}

int launch_select_lists(drb_ctx* ctx, uint64_t* lists, int cap, int32_t* cnt, uint32_t* tau_ord, float* tau_z, int k,
                        bool final, int32_t* out_iid, float* out_score, int32_t* n_out, int32_t* fb_users, int32_t* fb_count,
                        int fb_max, int32_t* big_users, int32_t* big_count, int n) {
  if (n <= 0) return DRB_OK;
  if (cap < 32 || (cap & (cap - 1)) || cap > 8192) return drb_fail(DRB_E_INVALID, "select_lists: cap must be a power of two in [32, 8192]");
  if (k < 1 || k > 2048) return drb_fail(DRB_E_INVALID, "select_lists: k must be in [1, 2048]");
  static bool attr_set = false;
  if (!attr_set) {
    cudaError_t e = cudaFuncSetAttribute(k_select_lists, cudaFuncAttributeMaxDynamicSharedMemorySize, (8192 + 2048) * 8);
    if (e != cudaSuccess) return drb_fail(DRB_E_CUDA, "cudaFuncSetAttribute(k_select_lists) failed: %s", cudaGetErrorString(e));
    attr_set = true;
  }
  SelectArgs a{};
  a.lists = lists; a.cap = cap; a.cnt = cnt; a.tau_ord = tau_ord; a.tau_z = tau_z; a.k = k; a.final = final ? 1 : 0;
  a.P = next_pow2(k); a.out_iid = out_iid; a.out_score = out_score; a.n_out = n_out;
  a.fb_users = fb_users; a.fb_count = fb_count; a.fb_max = fb_max;
  a.sm_cap = std::min(cap, 1024); a.big_users = big_users; a.big_count = big_count;
  drb_prof_scope prof_(ctx, final ? "k_select_lists_final" : "k_select_lists_tau");
  static const bool warp_form = !(getenv("DRB_SELECT_WARP") && atoi(getenv("DRB_SELECT_WARP")) == 0);
  if (!final && warp_form && cap >= 1024) {
    k_select_tau_warp<<<(n + 7) / 8, 256, 0, ctx->stream>>>(a, n);
  } else {
    k_select_lists<<<n, 64, (size_t)(a.sm_cap + (final ? a.P : 0)) * sizeof(uint64_t), ctx->stream>>>(a, n);
  }
  DRB_LAUNCH_CHECK(ctx, "k_select_lists");
  if (cap > a.sm_cap) {             // users whose list is longer than 1024 keys (none, usually: the CTAs leave at once)
    a.big_pass = 1;
    k_select_lists<<<std::min(n, 7 * ctx->sm_count), 256, (size_t)(cap + (final ? a.P : 0)) * sizeof(uint64_t), ctx->stream>>>(a, n);
    DRB_LAUNCH_CHECK(ctx, "k_select_lists");
  }
  return DRB_OK;
}

int launch_topk_fallback(drb_ctx* ctx, const TopkArgs& a, int n, const float* h, int ld_h, const float* table, int ld_t,
                         const float* bias, int width, float* rows, int32_t* fb_users, int32_t* fb_count, int fb_max) {
  if (n <= 0) return DRB_OK;
  {
    drb_prof_scope prof_(ctx, "k_fallback_scores");
    k_fallback_scores<<<fb_max, 256, 0, ctx->stream>>>(h, ld_h, table, ld_t, bias, width, a.n_items, rows, a.ld, fb_users,
                                                       fb_count, fb_max);
    DRB_LAUNCH_CHECK(ctx, "k_fallback_scores");
  }
  TopkArgs t = a;
  t.scores = rows; t.fb_users = fb_users; t.fb_count = fb_count; t.fb_max = fb_max;
  return launch_topk(ctx, t, fb_max);
}
