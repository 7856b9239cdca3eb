// Device helpers shared by the full-catalog top-k kernels (score.cu, umma_score.cu, dmf_topk.cu): the orderable
// 32-bit form of a score, the warp sum whose pairing every exact score reproduces, and the flush of a per-warp queue of
// list keys.  Keys are 64-bit (orderable(score) << 32 | iid), compared as unsigned integers: score first, then item id.
#ifndef DRB_TOPK_COMMON_CUH
#define DRB_TOPK_COMMON_CUH

#include "kernels.h"

namespace {

__device__ __forceinline__ uint32_t f2ord(float f) {
  const uint32_t u = __float_as_uint(f);
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float ord2f(uint32_t o) {
  return __uint_as_float((o & 0x80000000u) ? (o & 0x7fffffffu) : ~o);
}
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// Gives the queued keys of one warp their list slots (one atomicAdd per key, all issued before any is consumed) and
// stores them.  A queue entry is the final 64-bit key plus the user's row in the block.  Not inlined: the filter loops
// have many call sites and must stay inside the instruction cache.
template <int QCAP>
__device__ __noinline__ void flush_key_queue(const uint64_t* qk, const unsigned short* qu, int qn, int32_t* cnt,
                                             uint64_t* lists, int cap) {
  const int lane = threadIdx.x & 31;
  __syncwarp();
  uint64_t ent[QCAP / 32];
  int row[QCAP / 32], pos[QCAP / 32];
#pragma unroll
  for (int bq = 0; bq < QCAP / 32; bq++) {
    const int e = bq * 32 + lane;
    pos[bq] = 0x7fffffff;
    if (e < qn) {
      ent[bq] = qk[e];
      row[bq] = qu[e];
      pos[bq] = atomicAdd(cnt + row[bq], 1);
    }
  }
#pragma unroll
  for (int bq = 0; bq < QCAP / 32; bq++)
    if (pos[bq] < cap) lists[(int64_t)row[bq] * cap + pos[bq]] = ent[bq];
  __syncwarp();
}

}  // namespace

#endif
