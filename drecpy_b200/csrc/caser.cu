// Caser (Tang & Wang, WSDM 2018) on sm_100a: the device batch sampler, the fused forward + backward pass of one
// training step and the user representation x = [z; P[u]] used for scoring.  The model is pinned by oracle/caser.py
// (float64); parity with DRecPy's TensorFlow Caser is unpinned (DESIGN.md section 8).
//
// k_caser_sample   one warp per window: a 64-bit philox draw modulo the window count, a binary search in the per-user
//                  window prefix sums, then T * neg_ratio negatives, each redrawn (attempt index in the counter, at
//                  most 32 attempts, the last kept) while it is one of the user's stored items.
// k_caser_step     persistent CTAs (one per SM): the conv / fc weights are staged in shared memory once, their
//                  gradients are accumulated there (every element owned by one thread: no shared atomics) and reach
//                  the gradient arena with one atomic per element and CTA.  Per window: embedding gather, vertical and
//                  horizontal convolutions (max-pooled, argmax kept), philox dropout, fc + relu, the T (1 + neg_ratio)
//                  scores, Keras BCE, and the backward pass.  The gradient rows of E, P, W2 and b2 go out with
//                  atomics (vector atomics for the 16-byte aligned rows of E and W2).
// k_caser_user_rep the same forward pass without dropout on the last L items of each user's sequence.
#include <algorithm>

#include "kernels.h"

namespace {

constexpr float KERAS_EPS = 1e-7f;
constexpr int kCsThreads = 256, kCsWarps = kCsThreads / 32;
constexpr uint32_t kSaltWindow = 0x9E3779B9u, kSaltNeg = 0x3C6EF372u, kSaltDrop = 0xDAA66D2Bu;

__device__ __forceinline__ uint32_t cs_philox(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0,
                                              uint32_t k1) {
#pragma unroll
  for (int r = 0; r < 10; r++) {
    const uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
    const uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
    const uint32_t n0 = hi1 ^ c1 ^ k0, n1 = lo1, n2 = hi0 ^ c3 ^ k1, n3 = lo0;
    c0 = n0; c1 = n1; c2 = n2; c3 = n3;
    k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
  }
  return c0;
}
__device__ __forceinline__ float cs_warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ bool cs_contains(const int32_t* lo, int n, int32_t x) {
  int a = 0, b = n;
  while (a < b) {
    const int mid = (a + b) >> 1;
    if (lo[mid] < x) a = mid + 1; else b = mid;
  }
  return a < n && lo[a] == x;
}
__device__ __forceinline__ uint64_t cs_step(const CaserArgs& a) {
  return a.step_dev ? (((uint64_t)a.step_dev[1] << 32) | a.step_dev[0]) : a.step;
}

__global__ void __launch_bounds__(256) k_caser_sample(CaserArgs a, int batch) {
  const int b = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (b >= batch) return;
  const uint64_t step = cs_step(a);
  const uint32_t slo = (uint32_t)step, shi = (uint32_t)(step >> 32);
  const uint32_t k0 = (uint32_t)a.seed, k1 = (uint32_t)(a.seed >> 32);
  int u = 0;
  int64_t start = 0;
  if (lane == 0) {
    const uint64_t v = ((uint64_t)cs_philox(0, b, slo, shi, k0 ^ kSaltWindow, k1) << 32) |
                       cs_philox(1, b, slo, shi, k0 ^ kSaltWindow, k1);
    const int64_t idx = (int64_t)(v % (uint64_t)a.n_windows);
    int lo = 0, hi = a.n_users;            // last u with win_off[u] <= idx
    while (hi - lo > 1) {
      const int mid = (lo + hi) >> 1;
      if (a.win_off[mid] <= idx) lo = mid; else hi = mid;
    }
    u = lo;
    start = idx - a.win_off[u];
  }
  u = __shfl_sync(0xffffffffu, u, 0);
  start = __shfl_sync(0xffffffffu, start, 0);
  const int row = a.L + a.n_tgt;
  int32_t* out = a.ex_items + (int64_t)b * row;
  if (lane == 0) a.ex_user[b] = u;
  const int32_t* s = a.seq + a.seq_off[u] + start;
  for (int q = lane; q < a.L + a.T; q += 32) out[q] = s[q];
  const int32_t* seen = a.seen_indices + a.seen_indptr[u];
  const int nseen = (int)(a.seen_indptr[u + 1] - a.seen_indptr[u]);
  for (int q = lane; q < a.n_tgt - a.T; q += 32) {
    int item = 0;
    for (int t = 0; t < 32; t++) {
      item = (int)(cs_philox((uint32_t)(q * 32 + t), b, slo, shi, k0 ^ kSaltNeg, k1) % (uint32_t)a.n_items);
      if (!cs_contains(seen, nseen, item)) break;
    }
    out[a.L + a.T + q] = item;
  }
}

// Shared-memory plan of k_caser_step / k_caser_user_rep (floats; caser_smem_bytes sizes it)
struct Smem {
  float *fv, *bv, *fh, *bh, *fc, *bfc;          // staged weights
  float *gfv, *gbv, *gfh, *gbh, *gfc, *gbfc;    // per-CTA gradient sums (training)
  float *eh, *deh, *conv, *cv, *dc, *keep, *x, *dxp, *red, *dz, *loss;
  int *items, *amax;
};

__device__ __forceinline__ Smem carve(const CaserArgs& a, float* base, bool train) {
  Smem s;
  float* p = base;
  auto take = [&](int64_t n) { float* r = p; p += (n + 3) & ~3ll; return r; };
  s.fv = take(a.L * a.n_v); s.bv = take(a.n_v); s.fh = take(a.n_fh); s.bh = take(a.L * a.n_h);
  s.fc = take((int64_t)a.F * a.d); s.bfc = take(a.d);
  if (train) {
    s.gfv = take(a.L * a.n_v); s.gbv = take(a.n_v); s.gfh = take(a.n_fh); s.gbh = take(a.L * a.n_h);
    s.gfc = take((int64_t)a.F * a.d); s.gbfc = take(a.d);
  }
  s.eh = take(a.L * a.lde); s.deh = take(a.L * a.lde); s.conv = take(a.n_conv); s.cv = take(a.F); s.dc = take(a.F);
  s.keep = take(a.F); s.x = take(a.ldx); s.dxp = take(kCsWarps * a.ldx); s.red = take(kCsThreads); s.dz = take(a.d);
  s.loss = take(kCsWarps);
  s.items = reinterpret_cast<int*>(take(a.L + a.n_tgt));
  s.amax = reinterpret_cast<int*>(take(a.L * a.n_h));
  return s;
}

// offset of the kernel of height h (1-based) inside the horizontal block: n_h d (h - 1) h / 2
__device__ __forceinline__ int fh_off(const CaserArgs& a, int h) { return a.n_h * a.d * (h - 1) * h / 2; }

// forward pass of one example up to x = [z; P[u]] (in s.x); items[0..L) hold the inputs (-1: zero row)
__device__ void caser_forward(const CaserArgs& a, const Smem& s, int user, int ex, bool train, uint64_t step) {
  const int tid = threadIdx.x, d = a.d, L = a.L, n_h = a.n_h, n_v = a.n_v;
  for (int e = tid; e < L * a.lde; e += kCsThreads) {
    const int l = e / a.lde, k = e % a.lde;
    const int it = s.items[l];
    s.eh[e] = (it >= 0 && k < d) ? a.params[a.off_e + (int64_t)it * a.lde + k] : 0.f;
  }
  __syncthreads();
  for (int e = tid; e < n_v * d; e += kCsThreads) {        // vertical: o~[c d + k]
    const int c = e / d, k = e % d;
    float v = s.bv[c];
    for (int l = 0; l < L; l++) v = fmaf(s.fv[l * n_v + c], s.eh[l * a.lde + k], v);
    s.cv[e] = v;
  }
  for (int e = tid; e < a.n_conv; e += kCsThreads) {       // horizontal, before pooling: (h, i, f)
    int h = 1, r = e;
    while (r >= (L - h + 1) * n_h) { r -= (L - h + 1) * n_h; h++; }
    const int i = r / n_h, f = r % n_h;
    const float* fh = s.fh + fh_off(a, h);
    float v = s.bh[(h - 1) * n_h + f];
    for (int q = 0; q < h; q++) {
      const float* er = s.eh + (i + q) * a.lde;
      const float* fr = fh + q * d * n_h + f;
      for (int k = 0; k < d; k++) v = fmaf(er[k], fr[k * n_h], v);
    }
    s.conv[e] = v;
  }
  __syncthreads();
  for (int e = tid; e < L * n_h; e += kCsThreads) {        // max over i of relu(.): first maximum, -1 when <= 0
    const int h = e / n_h + 1, f = e % n_h;
    int base = 0;
    for (int g = 1; g < h; g++) base += (L - g + 1) * n_h;
    float best = s.conv[base + f];
    int bi = 0;
    for (int i = 1; i <= L - h; i++) {
      const float v = s.conv[base + i * n_h + f];
      if (v > best) { best = v; bi = i; }
    }
    s.amax[e] = best > 0.f ? bi : -1;
    s.cv[n_v * d + e] = fmaxf(best, 0.f);
  }
  __syncthreads();
  if (train) {
    const uint32_t k0 = (uint32_t)a.seed ^ kSaltDrop, k1 = (uint32_t)(a.seed >> 32);
    for (int e = tid; e < a.F; e += kCsThreads) {
      float sc = 1.f;
      if (a.dropout > 0.f) {
        const uint32_t xr = cs_philox(e, ex, (uint32_t)step, (uint32_t)(step >> 32), k0, k1);
        const float u = (float)(xr >> 8) * (1.0f / 16777216.0f);
        sc = u >= a.dropout ? a.keep_scale : 0.f;
      }
      s.keep[e] = sc;
      s.cv[e] *= sc;
    }
    __syncthreads();
  }
  const int parts = max(1, kCsThreads / d);
  for (int t = tid; t < parts * d; t += kCsThreads) {     // fc: partial sums over a stride of the inputs
    const int o = t % d, p = t / d;
    float v = 0.f;
    for (int i = p; i < a.F; i += parts) v = fmaf(s.cv[i], s.fc[i * d + o], v);
    s.red[t] = v;
  }
  __syncthreads();
  for (int k = tid; k < a.ldx; k += kCsThreads) {
    float v = 0.f;
    if (k < d) {
      v = s.bfc[k];
      for (int p = 0; p < parts; p++) v += s.red[p * d + k];
      v = fmaxf(v, 0.f);
    } else if (k < 2 * d) {
      v = a.params[a.off_p + (int64_t)user * a.lde + (k - d)];
    }
    s.x[k] = v;
  }
  __syncthreads();
}

__global__ void __launch_bounds__(kCsThreads) k_caser_step(CaserArgs a, int batch) {
  extern __shared__ __align__(16) float smem[];
  const Smem s = carve(a, smem, true);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int d = a.d, L = a.L, n_h = a.n_h, n_v = a.n_v, F = a.F;
  const float* P = a.params;
  for (int e = tid; e < L * n_v; e += kCsThreads) { s.fv[e] = P[a.off_fv + e]; s.gfv[e] = 0.f; }
  for (int e = tid; e < n_v; e += kCsThreads) { s.bv[e] = P[a.off_bv + e]; s.gbv[e] = 0.f; }
  for (int e = tid; e < a.n_fh; e += kCsThreads) { s.fh[e] = P[a.off_fh + e]; s.gfh[e] = 0.f; }
  for (int e = tid; e < L * n_h; e += kCsThreads) { s.bh[e] = P[a.off_bh + e]; s.gbh[e] = 0.f; }
  for (int e = tid; e < F * d; e += kCsThreads) { s.fc[e] = P[a.off_fc + e]; s.gfc[e] = 0.f; }
  for (int e = tid; e < d; e += kCsThreads) { s.bfc[e] = P[a.off_bfc + e]; s.gbfc[e] = 0.f; }
  const uint64_t step = cs_step(a);
  float loss = 0.f;
  const int row = L + a.n_tgt;
  for (int b = blockIdx.x; b < batch; b += gridDim.x) {
    __syncthreads();                                   // the previous example is done with every buffer
    for (int q = tid; q < row; q += kCsThreads) s.items[q] = a.ex_items[(int64_t)b * row + q];
    for (int e = tid; e < kCsWarps * a.ldx; e += kCsThreads) s.dxp[e] = 0.f;
    const int user = a.ex_user[b];
    __syncthreads();
    caser_forward(a, s, user, b, true, step);
    // scores of the T targets (label 1) and the negatives (label 0), Keras BCE, dL/dy; dx partials per warp
    for (int q = warp; q < a.n_tgt; q += kCsWarps) {
      const int j = s.items[L + q];
      const float t = q < a.T ? 1.f : 0.f;
      const float* w = P + a.off_w2 + (int64_t)j * a.ldx;
      float dot = 0.f;
      for (int k = lane; k < a.ldx; k += 32) dot = fmaf(s.x[k], w[k], dot);
      dot = cs_warp_sum(dot);
      const float y = dot + P[a.off_b2 + j];
      const float p = 1.0f / (1.0f + expf(-y));
      const float one_m = 1.0f - KERAS_EPS;
      const float pc = fminf(fmaxf(p, KERAS_EPS), one_m);
      const float da = pc + KERAS_EPS, db = 1.0f - pc + KERAS_EPS;
      if (lane == 0) loss += -(t * logf(da) + (1.0f - t) * logf(db));
      const bool inside = (p >= KERAS_EPS) && (p <= one_m);
      const float gy = inside ? -(t / da - (1.0f - t) / db) * a.inv_count * (p * (1.0f - p)) : 0.f;
      for (int k = lane; k < a.ldx; k += 32) s.dxp[warp * a.ldx + k] = fmaf(gy, w[k], s.dxp[warp * a.ldx + k]);
      float4* gw = reinterpret_cast<float4*>(a.grads + a.off_w2 + (int64_t)j * a.ldx);
      const float4* x4 = reinterpret_cast<const float4*>(s.x);
      for (int k4 = lane; k4 < a.ldx / 4; k4 += 32) {
        const float4 xv = x4[k4];
        atomicAdd(gw + k4, make_float4(gy * xv.x, gy * xv.y, gy * xv.z, gy * xv.w));
      }
      if (lane == 0) atomicAdd(a.grads + a.off_b2 + j, gy);
    }
    __syncthreads();
    for (int k = tid; k < 2 * d; k += kCsThreads) {
      float dx = 0.f;
      for (int w = 0; w < kCsWarps; w++) dx += s.dxp[w * a.ldx + k];
      if (k < d) {
        const float dz = s.x[k] > 0.f ? dx : 0.f;
        s.dz[k] = dz;
        s.gbfc[k] += dz;
      } else {
        atomicAdd(a.grads + a.off_p + (int64_t)user * a.lde + (k - d), dx);
      }
    }
    __syncthreads();
    for (int i = tid; i < F; i += kCsThreads) {        // dc = (W_fc dz) * dropout scale
      float v = 0.f;
      for (int o = 0; o < d; o++) v = fmaf(s.fc[i * d + o], s.dz[o], v);
      s.dc[i] = v * s.keep[i];
    }
    for (int e = tid; e < F * d; e += kCsThreads) s.gfc[e] = fmaf(s.cv[e / d], s.dz[e % d], s.gfc[e]);
    __syncthreads();
    const float* dov = s.dc;                 // [n_v d] vertical, then [L n_h] pooled horizontal outputs
    const float* doh = s.dc + n_v * d;
    for (int e = tid; e < L * n_v; e += kCsThreads) {
      const int l = e / n_v, c = e % n_v;
      float v = 0.f;
      for (int k = 0; k < d; k++) v = fmaf(dov[c * d + k], s.eh[l * a.lde + k], v);
      s.gfv[e] += v;
    }
    for (int c = tid; c < n_v; c += kCsThreads) {
      float v = 0.f;
      for (int k = 0; k < d; k++) v += dov[c * d + k];
      s.gbv[c] += v;
    }
    for (int e = tid; e < L * n_h; e += kCsThreads)
      if (s.amax[e] >= 0) s.gbh[e] += doh[e];
    for (int e = tid; e < a.n_fh; e += kCsThreads) {   // (h, q, k, f) with q < h
      int h = 1, r = e;
      while (r >= h * d * n_h) { r -= h * d * n_h; h++; }
      const int q = r / (d * n_h), k = (r / n_h) % d, f = r % n_h;
      const int i0 = s.amax[(h - 1) * n_h + f];
      if (i0 >= 0) s.gfh[e] = fmaf(doh[(h - 1) * n_h + f], s.eh[(i0 + q) * a.lde + k], s.gfh[e]);
    }
    for (int e = tid; e < L * a.lde; e += kCsThreads) {   // dE^[l, k]
      const int l = e / a.lde, k = e % a.lde;
      float v = 0.f;
      if (k < d) {
        for (int c = 0; c < n_v; c++) v = fmaf(s.fv[l * n_v + c], dov[c * d + k], v);
        for (int h = 1; h <= L; h++) {
          const float* fh = s.fh + fh_off(a, h);
          for (int f = 0; f < n_h; f++) {
            const int i0 = s.amax[(h - 1) * n_h + f];
            if (i0 >= 0 && l >= i0 && l < i0 + h) v = fmaf(doh[(h - 1) * n_h + f], fh[((l - i0) * d + k) * n_h + f], v);
          }
        }
      }
      s.deh[e] = v;
    }
    __syncthreads();
    for (int e = tid; e < L * (a.lde / 4); e += kCsThreads) {   // rows of E: vector atomics
      const int l = e / (a.lde / 4), k4 = e % (a.lde / 4);
      const int it = s.items[l];
      const float4 v = reinterpret_cast<const float4*>(s.deh + l * a.lde)[k4];
      atomicAdd(reinterpret_cast<float4*>(a.grads + a.off_e + (int64_t)it * a.lde) + k4, v);
    }
  }
  if (lane == 0) s.loss[warp] = loss;
  __syncthreads();
  if (tid == 0) {
    float t = 0.f;
    for (int w = 0; w < kCsWarps; w++) t += s.loss[w];
    a.loss_part[blockIdx.x] = t;
  }
  float* G = a.grads;
  for (int e = tid; e < L * n_v; e += kCsThreads) atomicAdd(G + a.off_fv + e, s.gfv[e]);
  for (int e = tid; e < n_v; e += kCsThreads) atomicAdd(G + a.off_bv + e, s.gbv[e]);
  for (int e = tid; e < a.n_fh; e += kCsThreads) atomicAdd(G + a.off_fh + e, s.gfh[e]);
  for (int e = tid; e < L * n_h; e += kCsThreads) atomicAdd(G + a.off_bh + e, s.gbh[e]);
  for (int e = tid; e < F * d; e += kCsThreads) atomicAdd(G + a.off_fc + e, s.gfc[e]);
  for (int e = tid; e < d; e += kCsThreads) atomicAdd(G + a.off_bfc + e, s.gbfc[e]);
}

__global__ void __launch_bounds__(kCsThreads) k_caser_user_rep(CaserArgs a, const int32_t* uids, int n, float* out) {
  extern __shared__ __align__(16) float smem[];
  const Smem s = carve(a, smem, false);
  const int tid = threadIdx.x;
  const float* P = a.params;
  for (int e = tid; e < a.L * a.n_v; e += kCsThreads) s.fv[e] = P[a.off_fv + e];
  for (int e = tid; e < a.n_v; e += kCsThreads) s.bv[e] = P[a.off_bv + e];
  for (int e = tid; e < a.n_fh; e += kCsThreads) s.fh[e] = P[a.off_fh + e];
  for (int e = tid; e < a.L * a.n_h; e += kCsThreads) s.bh[e] = P[a.off_bh + e];
  for (int e = tid; e < a.F * a.d; e += kCsThreads) s.fc[e] = P[a.off_fc + e];
  for (int e = tid; e < a.d; e += kCsThreads) s.bfc[e] = P[a.off_bfc + e];
  for (int r = blockIdx.x; r < n; r += gridDim.x) {
    __syncthreads();
    const int u = uids[r];
    const int64_t lo = a.seq_off[u];
    const int len = (int)(a.seq_off[u + 1] - lo);
    for (int l = tid; l < a.L; l += kCsThreads) {      // the last L items, left-padded with zero rows
      const int idx = len - a.L + l;
      s.items[l] = idx >= 0 ? a.seq[lo + idx] : -1;
    }
    __syncthreads();
    caser_forward(a, s, u, r, false, 0);
    for (int k = tid; k < a.ldx; k += kCsThreads) out[(int64_t)r * a.ldx + k] = s.x[k];
  }
}

}  // namespace

int64_t caser_smem_bytes(const CaserArgs& a, bool train) {
  auto r4 = [](int64_t n) { return (n + 3) & ~3ll; };
  int64_t w = r4(a.L * a.n_v) + r4(a.n_v) + r4(a.n_fh) + r4(a.L * a.n_h) + r4((int64_t)a.F * a.d) + r4(a.d);
  int64_t f = w * (train ? 2 : 1) + 2 * r4(a.L * a.lde) + r4(a.n_conv) + 3 * r4(a.F) + r4(a.ldx) + r4(kCsWarps * a.ldx) +
              r4(kCsThreads) + r4(a.d) + r4(kCsWarps) + r4(a.L + a.n_tgt) + r4(a.L * a.n_h);
  return f * 4;
}

int launch_caser_sample(drb_ctx* ctx, const CaserArgs& a, int batch) {
  if (batch <= 0) return DRB_OK;
  drb_prof_scope prof_(ctx, "k_caser_sample");
  k_caser_sample<<<(batch * 32 + 255) / 256, 256, 0, ctx->stream>>>(a, batch);
  DRB_LAUNCH_CHECK(ctx, "k_caser_sample");
  return DRB_OK;
}

int launch_caser_step(drb_ctx* ctx, const CaserArgs& a, int batch, int* n_blocks_out) {
  const int64_t smem = caser_smem_bytes(a, true);
  if (smem > kCaserMaxSmem) return drb_fail(DRB_E_INVALID, "caser step: %lld bytes of shared memory needed", (long long)smem);
  const int grid = std::max(1, std::min(batch, ctx->sm_count));
  *n_blocks_out = grid;
  if (batch <= 0) return DRB_OK;
  cudaError_t e = cudaFuncSetAttribute(k_caser_step, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return drb_fail(DRB_E_CUDA, "cudaFuncSetAttribute(k_caser_step) failed: %s", cudaGetErrorString(e));
  drb_prof_scope prof_(ctx, "k_caser_step");
  k_caser_step<<<grid, kCsThreads, smem, ctx->stream>>>(a, batch);
  DRB_LAUNCH_CHECK(ctx, "k_caser_step");
  return DRB_OK;
}

int launch_caser_user_rep(drb_ctx* ctx, const CaserArgs& a, const int32_t* uids, int n, float* out) {
  if (n <= 0) return DRB_OK;
  const int64_t smem = caser_smem_bytes(a, false);
  if (smem > kCaserMaxSmem) return drb_fail(DRB_E_INVALID, "caser user rep: %lld bytes of shared memory needed", (long long)smem);
  cudaError_t e = cudaFuncSetAttribute(k_caser_user_rep, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return drb_fail(DRB_E_CUDA, "cudaFuncSetAttribute(k_caser_user_rep) failed: %s", cudaGetErrorString(e));
  drb_prof_scope prof_(ctx, "k_caser_user_rep");
  k_caser_user_rep<<<std::min(n, 2 * ctx->sm_count), kCsThreads, smem, ctx->stream>>>(a, uids, n, out);
  DRB_LAUNCH_CHECK(ctx, "k_caser_user_rep");
  return DRB_OK;
}
