// K2 on the tensor cores, persistent form: z2 = h W'^T (fp32-accurate split products on tcgen05.mma: 3 x FP16, or
// 3 x TF32; TMA-fed) with the fused
// b' + sigmoid + Keras BCE/MSE + dL/dz2 epilogue of the CDAE training step.
//
// Replaces (reference, DRecPy/): Recommender/cdae.py:76 (tf.matmul(hidden, W_) + b_ + sigmoid) and cdae.py:78-79
// (Keras loss on the (B,B,I) broadcast == batch-mean labels, SURVEY.md Q1) plus d(loss)/d(z2) of tape.gradient.
// p is never written to memory; the epilogue emits dL/dz2 already split into fp16 (or tf32) hi/lo for the backward
// GEMMs.
//
// The product is formed transposed, z2^T = W' h^T: MMA M = 128 items (TMEM lanes), N = up to 256 batch rows (TMEM
// columns).  An epilogue warp therefore holds 32 consecutive items of one batch row across its lanes, which is one
// 128-byte line of the dz layout below: every dz store instruction writes one full line.  (With batch rows on the
// lanes each store touched 32 lines, 16 bytes each, and the kernel was bound by the store path: 0.49 -> see DESIGN.md.)
//
// One CTA per SM loops over output tiles (batch tiles fastest, so co-running CTAs share the W' tile in L2).  The K
// extent is short (hidden <= 255 -> <= 8 k-blocks), so per-tile set-up and the exposed epilogue dominated the
// one-tile-per-CTA version; here the TMA producer runs ahead across tiles, the accumulator is double-buffered in TMEM
// (2 x BN columns) and the 16 epilogue warps drain tile t while the MMA warp fills tile t+1.
// dz is written in a tile-major layout (128 batch rows x 64 halfs, or x 32 floats, = 16 KB contiguous), and the two
// backward GEMMs later fetch whole tiles / sub-tiles with single TMA boxes (one copy: dh reads it K-major, dW'^T through
// the MN-major descriptor).
#include "umma_common.cuh"

namespace {

constexpr int DRB_LOSS_CLUSTER_DEFAULT = 2;              // 2 = CTA pairs, cta_group::2 MMAs (env DRB_LOSS_CLUSTER)
constexpr int LOSS_EPI_WARPS = 16;                      // four per TMEM sub-partition, each takes a quarter of the columns
constexpr int LOSS_THREADS = 64 + 32 * LOSS_EPI_WARPS;

// KB: floats of the hidden dimension per pipeline stage; CL = 2: CTA pair, each CTA stages half of the h rows (see
// umma.cu: Smem)
template <int BN, int KB, int CL>
struct LossSmem {
  static constexpr int A_BYTES = BM * KB * 4;
  static constexpr int B_BYTES = (BN / CL) * KB * 4;
  static constexpr int STAGES = 192 * 1024 / (2 * A_BYTES + 2 * B_BYTES);
  static constexpr int STAGE_BYTES = 2 * A_BYTES + 2 * B_BYTES;
  static constexpr int BAR_BYTES = 256;
  static constexpr int TOTAL = STAGES * STAGE_BYTES + 1024 + BAR_BYTES;
};

struct LossParams {
  int M, N, Kred;                          // batch, n_items, hidden (padded to 4)
  float* dz_hi; float* dz_lo; int nib;     // tile-major (kernels.h: drb_dz_nib), nib column blocks per row tile
  const float* bias;                       // b' [N]
  const float* label_count; const uint32_t* label_bits; int words_per_row;
  int loss_kind; float inv_count; int batch;
  float* loss_part;                        // [gridDim.x]
  float* colsum;                           // NULL, or [N]: db' += column sums of dz (hidden = 256: no room for the ones feature)
  int m_tiles, n_tiles, row_tiles;         // item tiles (128), batch tiles (BN), 128-row tiles of the dz layout
  DzHalf dzh;                              // H: fp16 dz copies (kernels.h), values scaled by DRB_DZ_F16_SCALE / inv_count
  float out_scale; const float* out_scale_dev;   // H: accumulator -> logit (undoes the operand scaling)
  float* z_dbg; int ldz;                   // tests only (drb_debug_cdae_capture_logits): z2 = h W'^T + b' as this kernel
                                           // formed it, row-major [M][ldz]; NULL in production
  uint32_t wait_ns;                        // sleep between polls of the accumulator-full barrier (epilogue warps)
  int debug;   // DRB_LOSS_DEBUG bit mask (profiling experiments only, results are wrong): 2 = skip TMA + MMA, 4 = skip the dz stores, 8 = skip the B_lo loads, 16 = skip the MMAs,
               // 32 = no lg2 in the fast epilogue form
};

__device__ __forceinline__ float fast_ex2(float x) { float y; asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
__device__ __forceinline__ float fast_lg2(float x) { float y; asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
__device__ __forceinline__ float fast_rcp(float x) { float y; asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }

__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}

// same barrier offset in CTA `rank`.  Relaxed: the arrival only says "this warp's tcgen05.ld of the accumulator have
// completed" (tcgen05.wait::ld precedes it); a release at cluster scope is a MEMBAR that first drains the warp's ~150
// outstanding dz stores (ncu: stall_membar + ERRBAR were 12 % of the kernel's samples)
__device__ __forceinline__ void mbar_arrive_rank(uint32_t bar, uint32_t rank) {
  asm volatile("mbarrier.arrive.relaxed.cluster.shared::cluster.b64 _, [%0];" ::"r"(mapa_rank(bar, rank)) : "memory");
}

// CL = 2: the two CTAs of a cluster (one TPC) work on two item tiles of the same batch tile as a CTA pair: the even
// CTA issues cta_group::2 MMAs (M = 256) that read each CTA's own W' tile and each CTA's half of the shared h tile and
// write each CTA's own accumulator, so the h tile is staged once per pair and the MMAs read a third less shared memory.
// (TMA multicast of the h tile with one-CTA MMAs was measured first: no gain, 0.299 vs 0.302 ms.)
// ZDBG: the test-only logit capture (drb_debug_cdae_capture_logits) is its own instantiation, so that the production
// epilogue stays branch free (a per-element `if (z_dbg)` cost 6 % of the kernel)
template <int BN, int LOSS, bool PER_USER, int KB, int CL, bool H, bool ZDBG>
__global__ void __launch_bounds__(LOSS_THREADS, 1)
k_umma_cdae_loss(const __grid_constant__ CUtensorMap map_a_hi, const __grid_constant__ CUtensorMap map_a_lo,
                 const __grid_constant__ CUtensorMap map_b_hi, const __grid_constant__ CUtensorMap map_b_lo,
                 LossParams p) {
  using S = LossSmem<BN, KB, CL>;
  constexpr int BK = H ? 2 * KB : KB;            // elements of the hidden dimension per stage (KB is in 4-byte units)
  constexpr int UK = H ? 16 : UMMA_K;            // elements one MMA consumes (32 bytes either way)
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
  volatile float* lred = reinterpret_cast<volatile float*>(smem_raw + (bars + 8u * (2 * S::STAGES + 5) - raw));

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int nkb = (p.debug & 2) ? 0 : (p.Kred + BK - 1) / BK;
  // work units: CL = 1 -> one tile per CTA per iteration; CL = 2 -> one pair of item tiles per cluster per iteration.
  // Batch tiles run fastest, so co-running CTAs share W' tiles in L2.
  const uint32_t cta_rank = (CL > 1) ? cluster_ctarank() : 0u;
  const bool leader = cta_rank == 0;
  const int unit0 = blockIdx.x / CL, unit_stride = gridDim.x / CL;
  const int n_units = ((p.m_tiles + CL - 1) / CL) * p.n_tiles;
  auto unit_item0 = [&](int u) { return ((u / p.n_tiles) * CL + (int)cta_rank) * BM; };
  auto unit_row0 = [&](int u) { return (u % p.n_tiles) * BN; };
  constexpr uint32_t TMEM_COLS = (2 * BN <= 64) ? 64 : (2 * BN <= 128) ? 128 : (2 * BN <= 256) ? 256 : 512;

  if (threadIdx.x == 0) {
    for (int s = 0; s < S::STAGES; s++) {
      mbar_init(full_bar(s), 1);
      mbar_init(empty_bar(s), 1);
    }
    for (int a = 0; a < 2; a++) {
      mbar_init(tfull_bar(a), 1);
      mbar_init(tempty_bar(a), CL * LOSS_EPI_WARPS);   // one arrival per epilogue warp of the pair (even CTA's is used)
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {
    if (CL > 1) {   // collective: the same warp of both CTAs
      asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tmem_ptr_addr), "r"(TMEM_COLS));
      asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;");
    } else {
      asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tmem_ptr_addr), "r"(TMEM_COLS));
      asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
    }
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  if (CL > 1) cluster_sync_all(); else __syncthreads();   // peers' barriers are initialised before anything is sent
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
          if (CL > 1) {   // both CTAs' loads report to the even CTA's barrier; this CTA stages its half of the h rows
            if (leader) mbar_expect_tx(full_bar(s), CL * S::STAGE_BYTES);
            const uint32_t fb = mapa_rank(full_bar(s), 0);
            const int rh = r0 + (int)cta_rank * (BN / CL);
            tma_load_2d_pair(sa_hi, &map_a_hi, fb, kb * BK, i0);
            tma_load_2d_pair(sa_lo, &map_a_lo, fb, kb * BK, i0);
            tma_load_2d_pair(sb_hi, &map_b_hi, fb, kb * BK, rh);
            tma_load_2d_pair(sb_lo, &map_b_lo, fb, kb * BK, rh);
          } else {
            mbar_expect_tx(full_bar(s), S::STAGE_BYTES - ((p.debug & 8) ? S::B_BYTES : 0));
            tma_load_2d(sa_hi, &map_a_hi, full_bar(s), kb * BK, i0);
            tma_load_2d(sa_lo, &map_a_lo, full_bar(s), kb * BK, i0);
            tma_load_2d(sb_hi, &map_b_hi, full_bar(s), kb * BK, r0);
            if (!(p.debug & 8)) tma_load_2d(sb_lo, &map_b_lo, full_bar(s), kb * BK, r0);
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
        mbar_wait(tempty_bar(as), ((tl >> 1) & 1) ^ 1);     // epilogue has drained this accumulator
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        const uint32_t tacc = tmem_base + (uint32_t)(as * BN);
        for (int kb = 0; kb < nkb; kb++, it++) {
          const int s = it % S::STAGES;
          mbar_wait(full_bar(s), (it / S::STAGES) & 1);
          asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
          const uint32_t sa_hi = base + s * S::STAGE_BYTES, sa_lo = sa_hi + S::A_BYTES;
          const uint32_t sb_hi = sa_lo + S::A_BYTES, sb_lo = sb_hi + S::B_BYTES;
          // the last k-block holds fewer than BK real columns (K = 200: 6 full blocks + 8 columns): TMA zero-fills the
          // rest of the box, the MMAs over those zeros are simply not issued
          const int kk_n = (p.debug & 16) ? 0 : min(BK / UK, (p.Kred - kb * BK + UK - 1) / UK);
#pragma unroll
          for (int kk = 0; kk < BK / UK; kk++) {
            if (kk >= kk_n) break;
            const uint64_t a_hi = make_desc_kmajor<KB>(sa_hi, kk), a_lo = make_desc_kmajor<KB>(sa_lo, kk);
            const uint64_t b_hi = make_desc_kmajor<KB>(sb_hi, kk), b_lo = make_desc_kmajor<KB>(sb_lo, kk);
            umma_split<H, CL>(tacc, a_lo, b_hi, idesc, (kb | kk) != 0);
            umma_split<H, CL>(tacc, a_hi, b_lo, idesc, 1u);
            umma_split<H, CL>(tacc, a_hi, b_hi, idesc, 1u);
          }
          if (CL > 1) umma_commit_pair(empty_bar(s));   // frees the stage in both CTAs' producers
          else umma_commit(empty_bar(s));
        }
        if (CL > 1) umma_commit_pair(tfull_bar(as));
        else umma_commit(tfull_bar(as));
      }
    }
  } else {
    // ------------------------------------------------------------------ epilogue warps 2..17
    // The accumulator holds z2^T: TMEM lane = item, column = batch row.  Warp w reads lanes 32*(w&3)..+31 (hardware
    // sub-partition rule) = one 32-item block of the dz layout, and the column quarter (w-2)/4 of the tile.  For one
    // batch row the 32 lanes of a warp then own 128 contiguous bytes of a dz tile: every store is one full line.
    const int q = warp & 3, cq = (warp - 2) >> 2;
    const int ew = warp - 2;
    float loss_local = 0.f;
    const float one_m = 1.0f - KERAS_EPS;
    constexpr int CW = BN / 4;                    // batch rows of this warp per tile
    const float fbatch = (float)p.batch;
    // H: the operands were scaled into the fp16 range by powers of two; one multiply brings the accumulator back
    const float osc = H ? p.out_scale * (p.out_scale_dev ? __ldg(p.out_scale_dev) : 1.0f) : 1.0f;
    // H: dz leaves as fp16 hi/lo of (dL/dz2 / inv_count) * 2^14, a value in [-2^14, 2^14]; the backward GEMMs undo it
    const float gsc = H ? DRB_DZ_F16_SCALE : p.inv_count;
    // per-item constants (b', batch-mean label) live in registers and are fetched one tile ahead
    float nbias, ncount;
    auto fetch_consts = [&](int t) {
      const int item = unit_item0(t) + q * 32 + lane;
      const bool in = (t < n_units) && (item < p.N);
      nbias = in ? __ldg(p.bias + item) : 0.f;
      ncount = (!PER_USER && in) ? __ldg(p.label_count + item) : 0.f;
    };
    fetch_consts(unit0);
    int tl = 0;
    for (int t = unit0; t < n_units; t += unit_stride, tl++) {
      const int i0 = unit_item0(t), r0 = unit_row0(t);
      const int as = tl & 1;
      const int item = i0 + q * 32 + lane;
      const bool item_ok = item < p.N;
      const int ib = (i0 >> 5) + q;               // 32-item block of this warp
      const float bias = nbias, tgt_c = ncount / fbatch;
      const float osc2 = osc * -1.4426950408889634f, nb2 = bias * -1.4426950408889634f;   // exp2 argument = fma(acc, osc2, nb2)
      float sum_la = 0.f, sum_lb = 0.f;           // fast chunks: sums of lg2(p + eps), lg2(1 - p + eps) of this lane's item
      fetch_consts(t + unit_stride);
      mbar_wait_sleep(tfull_bar(as), (tl >> 1) & 1, p.wait_ns);
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
      const uint32_t tbase = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(as * BN + cq * CW);
      float csum = 0.f;                           // this lane's item: sum of dL/dz2 over the warp's batch rows
      // one chunk = 16 batch rows of this warp's 32 items; r[] holds the accumulator values on entry
      auto process_chunk = [&](uint32_t (&r)[16], const int cl) {
        const int row = r0 + cq * CW + cl;        // first of this chunk's 16 batch rows (same 128-row tile: 16 | 128)
        float lo[16];
        // branch-free element math: 16 independent dependency chains the scheduler can interleave.  MUFU ops are
        // issued directly (ex2 / rcp / lg2 .approx.ftz: no denormal fix-up sequences), 5 per element.
        //   p = 1 / (1 + 2^(-z log2 e));  pc = clip(p, eps, 1-eps);  da = pc + eps;  db = 1 - pc + eps
        //   bce term   = -(t ln da + (1-t) ln db) = -ln2 (lg2 db + t (lg2 da - lg2 db))
        //   dL/dp      = ((1-t) da - t db) / (da db) / (B I) = (da - t (da + db)) / (da db) / (B I)   [p inside the clip]
        //   dL/dz      = dL/dp * p (1-p)
        // Fast form of the same math for the common chunk (fp16 path, BCE, batch-mean labels): every (row, item) of the
        // chunk exists and no logit is extreme (|z| < 15.2, so p stays strictly inside Keras' clip and the clip, the
        // `inside` test and the row / item masks are the identity).  The logit is never formed: the exp2 argument is one
        // fma; log terms are summed as two plain sums (the label is constant per lane); da + db = 1 + 2 eps.  One
        // max-|arg| per element and one vote per chunk decide; the general form below handles everything else.
        bool fast = false;
        if (H && !ZDBG && LOSS == DRB_LOSS_BCE && !PER_USER) {
          fast = item_ok && (row + 16 <= p.M);
          float amax = 0.f;
#pragma unroll
          for (int j = 0; j < 16; j++) amax = fmaxf(amax, fabsf(fmaf(__uint_as_float(r[j]), osc2, nb2)));
          fast = !__any_sync(0xffffffffu, !fast || amax > 22.0f);
        }
        if (fast) {
          // One reciprocal per element: with s = 1 + e, t1 = 1 + eps s, t2 = e + eps s and R = 1 / (s t1 t2):
          //   p = 1/s = R t1 t2,  da = p + eps = t1/s,  db = 1 - p + eps = t2/s,  p (1-p) / (da db) = e / (t1 t2) = e s R.
          // The log terms of four elements are one lg2 of their product (da, db >= 3.4e-7 here: no underflow).
          float pa = 1.0f, pb = 1.0f;
#pragma unroll
          for (int j = 0; j < 16; j++) {
            const float e = fast_ex2(fmaf(__uint_as_float(r[j]), osc2, nb2));
            const float s1 = 1.0f + e;
            const float t12 = fmaf(KERAS_EPS, s1, 1.0f) * fmaf(KERAS_EPS, s1, e);
            const float R = fast_rcp(s1 * t12);
            const float pr = R * t12;
            const float da = pr + KERAS_EPS, db = (1.0f + KERAS_EPS) - pr;
            pa *= da; pb *= db;
            if ((j & 3) == 3) {
              sum_la += (p.debug & 32) ? pa : fast_lg2(pa); sum_lb += (p.debug & 32) ? pb : fast_lg2(pb);
              pa = 1.0f; pb = 1.0f;
            }
            const float num = fmaf(tgt_c, -(1.0f + 2.0f * KERAS_EPS), da);
            lo[j] = (num * e) * (R * (s1 * gsc));
          }
        } else
#pragma unroll
        for (int j = 0; j < 16; j++) {
          const bool ok = item_ok && (row + j < p.M);
          const float z = H ? fmaf(__uint_as_float(r[j]), osc, bias) : __uint_as_float(r[j]) + bias;
          if (ZDBG && ok) p.z_dbg[(int64_t)(row + j) * p.ldz + item] = z;
          const float pr = fast_rcp(1.0f + fast_ex2(z * -1.4426950408889634f));
          float tgt = tgt_c;
          if (PER_USER) {   // one broadcast word per batch row: bit `lane` of word ib
            const uint32_t w = (row + j < p.M && ib < p.words_per_row)
                                   ? __ldg(p.label_bits + (int64_t)(row + j) * p.words_per_row + ib) : 0u;
            tgt = (float)((w >> lane) & 1u);
          }
          float gz, lt;
          if (LOSS == DRB_LOSS_BCE) {
            const float pc = fminf(fmaxf(pr, KERAS_EPS), one_m);
            const float da = pc + KERAS_EPS, db = 1.0f - pc + KERAS_EPS;
            const float la = fast_lg2(da), lb = fast_lg2(db);
            lt = -0.6931471805599453f * fmaf(tgt, la - lb, lb);
            const bool inside = (pr >= KERAS_EPS) && (pr <= one_m);
            const float num = fmaf(-tgt, da + db, da);
            gz = inside ? num * (pr * (1.0f - pr)) * (fast_rcp(da * db) * gsc) : 0.f;
          } else {
            lt = PER_USER ? (pr - tgt) * (pr - tgt) : fmaf(pr, pr - 2.0f * tgt, tgt);
            gz = 2.0f * (pr - tgt) * gsc * (pr * (1.0f - pr));
          }
          loss_local += ok ? lt : 0.f;
          const float g = ok ? gz : 0.f;
          if (H) {
            lo[j] = g;                             // split below, two users at a time
          } else {
            float h;
            split_tf32(g, h, lo[j]);
            r[j] = __float_as_uint(h);
          }
        }
        if (H) {
          // fp16 hi/lo split of 16 values, two users at a time: hi = rn_f16(g) (one packed conversion for two values),
          // converted back exactly, lo = rn_f16(g - hi) -- the residual of the value actually stored as hi.
          // hp[i] / lp[i] = users (2i, 2i + 1) packed low | high.
          uint32_t hp[8], lp[8];
#pragma unroll
          for (int j = 0; j < 16; j += 2) {
            asm("cvt.rn.f16x2.f32 %0, %1, %2;" : "=r"(hp[j >> 1]) : "f"(lo[j + 1]), "f"(lo[j]));
            const float2 hf = __half22float2(*reinterpret_cast<const __half2*>(&hp[j >> 1]));
            asm("cvt.rn.f16x2.f32 %0, %1, %2;" : "=r"(lp[j >> 1]) : "f"(lo[j + 1] - hf.y), "f"(lo[j] - hf.x));
          }
          if (p.colsum) {                         // lo[] still holds the unsplit values
#pragma unroll
            for (int j = 0; j < 16; j++) csum += lo[j];
          }
          // two tile-major fp16 copies (tiles of 128 rows x 64 halfs).  U = [user tile][item block]: for one user the
          // lanes of the warp are 32 consecutive items = 64 contiguous bytes.  I = [item tile][user block]: this
          // thread's item row takes its 16 users = 32 contiguous bytes = hp[0..7] as they are.  Every element of an
          // existing tile is written (zeros outside the matrix): the backward GEMMs read whole tiles.
          const int rt = row >> 7, cbu = (i0 >> 6) + (q >> 1);
          if (rt < p.dzh.row_tiles && cbu < p.dzh.nib64 && !(p.debug & 4)) {
            const int64_t off = ((int64_t)(rt * p.dzh.nib64 + cbu) * 128 + (row & 127)) * 64 + (q & 1) * 32 + lane;
            unsigned short* uh = reinterpret_cast<unsigned short*>(p.dzh.u_hi) + off;
            unsigned short* ul = reinterpret_cast<unsigned short*>(p.dzh.u_lo) + off;
#pragma unroll
            for (int i = 0; i < 8; i++) {
              uh[(2 * i) * 64] = (unsigned short)hp[i];
              uh[(2 * i + 1) * 64] = (unsigned short)(hp[i] >> 16);
              ul[(2 * i) * 64] = (unsigned short)lp[i];
              ul[(2 * i + 1) * 64] = (unsigned short)(lp[i] >> 16);
            }
          }
          const int itile = i0 >> 7, ub = row >> 6;
          if (p.dzh.i_hi && itile < p.dzh.item_tiles && ub < p.dzh.nub && !(p.debug & 4)) {
            const int64_t off = ((int64_t)(itile * p.dzh.nub + ub) * 128 + q * 32 + lane) * 64 + (row & 63);
            uint4* dh4 = reinterpret_cast<uint4*>(reinterpret_cast<unsigned short*>(p.dzh.i_hi) + off);
            uint4* dl4 = reinterpret_cast<uint4*>(reinterpret_cast<unsigned short*>(p.dzh.i_lo) + off);
            dh4[0] = make_uint4(hp[0], hp[1], hp[2], hp[3]);
            dh4[1] = make_uint4(hp[4], hp[5], hp[6], hp[7]);
            dl4[0] = make_uint4(lp[0], lp[1], lp[2], lp[3]);
            dl4[1] = make_uint4(lp[4], lp[5], lp[6], lp[7]);
          }
        } else {
        if (p.colsum) {
#pragma unroll
          for (int j = 0; j < 16; j++) csum += __uint_as_float(r[j]) + lo[j];
        }
        // tile-major store: row j of this chunk is the 128-byte line ((row tile, item block), row in tile) and the
        // lanes are its 32 floats.  Every row and column of an existing tile is written (zeros outside the matrix)
        // because the backward GEMMs read whole tiles.
        const int rt = row >> 7;
        if (rt < p.row_tiles && ib < p.nib && !(p.debug & 4)) {   // wide tiles can overhang the last 128-row tile
          const int64_t off = ((int64_t)(rt * p.nib + ib) * 128 + (row & 127)) * 32 + lane;
#pragma unroll
          for (int j = 0; j < 16; j++) {
            p.dz_hi[off + j * 32] = __uint_as_float(r[j]);
            p.dz_lo[off + j * 32] = lo[j];
          }
        }
        }
      };
      // two register sets in turn: the tcgen05.ld of the next chunk runs behind the math of this one and no value is
      // ever copied between registers (CW is 32 or 64: an even number of chunks)
      uint32_t ra[16], rb[16];
      tmem_ld16_issue(tbase, ra);
#pragma unroll 1
      for (int cl = 0; cl < CW; cl += 32) {
        tmem_ld16_wait(ra);
        tmem_ld16_issue(tbase + cl + 16, rb);
        process_chunk(ra, cl);
        tmem_ld16_wait(rb);
        if (cl + 32 < CW) tmem_ld16_issue(tbase + cl + 32, ra);
        process_chunk(rb, cl + 16);
      }
      loss_local += -0.6931471805599453f * fmaf(tgt_c, sum_la - sum_lb, sum_lb);   // bce terms of the fast chunks
      if (p.colsum && item_ok) atomicAdd(p.colsum + item, H ? csum * (p.inv_count / DRB_DZ_F16_SCALE) : csum);
      // this warp has finished reading accumulator `as`
      asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
      __syncwarp();
      if (lane == 0) {
        if (CL > 1) mbar_arrive_rank(tempty_bar(as), 0);
        else mbar_arrive(tempty_bar(as));
      }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) loss_local += __shfl_xor_sync(0xffffffffu, loss_local, o);
    if (lane == 0) lred[ew] = loss_local;
    asm volatile("bar.sync 1, %0;" ::"n"(32 * LOSS_EPI_WARPS) : "memory");
    if (warp == 2 && lane == 0) {
      float tot = 0.f;
#pragma unroll
      for (int i = 0; i < LOSS_EPI_WARPS; i++) tot += lred[i];
      p.loss_part[blockIdx.x] = tot;
    }
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  if (CL > 1) cluster_sync_all(); else __syncthreads();   // no CTA leaves while its peer can still write to it
  if (warp == 1) {
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    if (CL > 1) asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(TMEM_COLS));
    else asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(TMEM_COLS));
  }
}

template <int BN, int LOSS, bool PER_USER, int KB, int CL, bool H, bool ZDBG>
int run_loss(drb_ctx* ctx, const UmmaOperands& o, LossParams p, int* n_blocks_out) {
  CUtensorMap ma_hi, ma_lo, mb_hi, mb_lo;
  int r;
  // MMA roles are swapped with respect to the caller's z = h W'^T: A (M side, 128 TMEM lanes) = W' rows = items,
  // B (N side, BN TMEM columns) = h rows = batch rows
  if ((r = make_operand_map<H>(&ma_hi, o.b_hi, p.Kred, o.b_rows, o.ldb, KB, BM))) return r;
  if ((r = make_operand_map<H>(&ma_lo, o.b_lo, p.Kred, o.b_rows, o.ldb, KB, BM))) return r;
  if ((r = make_operand_map<H>(&mb_hi, o.a_hi, p.Kred, p.M, o.lda, KB, BN / CL))) return r;
  if ((r = make_operand_map<H>(&mb_lo, o.a_lo, p.Kred, p.M, o.lda, KB, BN / CL))) return r;
  p.m_tiles = (p.N + BM - 1) / BM;      // item tiles
  p.n_tiles = (p.M + BN - 1) / BN;      // batch tiles
  p.row_tiles = (p.M + 127) / 128;
  auto kern = k_umma_cdae_loss<BN, LOSS, PER_USER, KB, CL, H, ZDBG>;
  constexpr int SMEM = LossSmem<BN, KB, CL>::TOTAL;
  static bool attr_set = false;       // per template instantiation
  static int max_clusters = 0;
  if (!attr_set) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM);
    if (e != cudaSuccess)
      return drb_fail(DRB_E_CUDA, "cudaFuncSetAttribute(smem=%d) failed: %s", SMEM, cudaGetErrorString(e));
    if (CL > 1) {   // clusters are placed inside a GPC: ask how many fit at once, the kernel is persistent
      cudaLaunchConfig_t qc{};
      cudaLaunchAttribute qa[1];
      qa[0].id = cudaLaunchAttributeClusterDimension;
      qa[0].val.clusterDim.x = CL; qa[0].val.clusterDim.y = 1; qa[0].val.clusterDim.z = 1;
      qc.gridDim = dim3(ctx->sm_count / CL * CL); qc.blockDim = dim3(LOSS_THREADS); qc.dynamicSmemBytes = SMEM;
      qc.attrs = qa; qc.numAttrs = 1;
      e = cudaOccupancyMaxActiveClusters(&max_clusters, kern, &qc);
      if (e != cudaSuccess || max_clusters < 1)
        return drb_fail(DRB_E_CUDA, "cudaOccupancyMaxActiveClusters failed: %s", cudaGetErrorString(e));
    }
    attr_set = true;
  }
  const int n_units = ((p.m_tiles + CL - 1) / CL) * p.n_tiles;
  const int grid = CL * std::min(n_units, CL > 1 ? max_clusters : ctx->sm_count);
  *n_blocks_out = grid;
  drb_prof_scope prof_(ctx, "k_umma_cdae_loss");
  if (CL > 1) {
    cudaLaunchConfig_t cfg{};
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = CL; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
    cfg.gridDim = dim3(grid); cfg.blockDim = dim3(LOSS_THREADS); cfg.dynamicSmemBytes = SMEM; cfg.stream = ctx->stream;
    cfg.attrs = at; cfg.numAttrs = 1;
    cudaError_t e = cudaLaunchKernelEx(&cfg, kern, ma_hi, ma_lo, mb_hi, mb_lo, p);
    if (e != cudaSuccess) return drb_fail(DRB_E_CUDA, "cluster launch of k_umma_cdae_loss failed: %s", cudaGetErrorString(e));
  } else {
    kern<<<grid, LOSS_THREADS, SMEM, ctx->stream>>>(ma_hi, ma_lo, mb_hi, mb_lo, p);
  }
  DRB_LAUNCH_CHECK(ctx, "k_umma_cdae_loss");
  return DRB_OK;
}

}  // namespace

int launch_umma_cdae_loss(drb_ctx* ctx, const UmmaOperands& o, int M, int N, int Kred, float* dz_hi, float* dz_lo,
                          int ldc, const float* bias, const float* label_count, const uint32_t* label_bits,
                          int words_per_row, int loss_kind, float inv_count, int batch, float* loss_part,
                          float* dz_colsum, int* n_blocks_out, float* z_dbg, int ldz, const DzHalf* dzh) {
  LossParams p{};
  p.z_dbg = z_dbg; p.ldz = ldz;
  if (o.half) {
    if (!dzh) return drb_fail(DRB_E_INVALID, "loss kernel: fp16 operands need the fp16 dz buffers");
    p.dzh = *dzh; p.out_scale = o.out_scale; p.out_scale_dev = o.out_scale_dev;
  }
  p.M = M; p.N = N; p.Kred = Kred; p.nib = drb_dz_nib(N); p.dz_hi = dz_hi; p.dz_lo = dz_lo; p.bias = bias;
  (void)ldc;
  p.label_count = label_count; p.label_bits = label_bits; p.words_per_row = words_per_row; p.loss_kind = loss_kind;
  p.inv_count = inv_count; p.batch = batch; p.loss_part = loss_part; p.colsum = dz_colsum;
  static const int dbg_env = getenv("DRB_LOSS_DEBUG") ? atoi(getenv("DRB_LOSS_DEBUG")) : 0;
  p.debug = dbg_env;
  static const int wait_env = getenv("DRB_WAIT_NS") ? atoi(getenv("DRB_WAIT_NS")) : 100;
  p.wait_ns = (uint32_t)wait_env;
  const bool per_user = label_count == nullptr;
  static const int bn_env = getenv("DRB_LOSS_BN") ? atoi(getenv("DRB_LOSS_BN")) : 0;
  // 256 batch rows per tile halve the re-reads of the W' tile (the main loop is L2->SM bandwidth bound)
  const bool wide = bn_env ? (bn_env == 256) : (M > 128);
  static const int cl_env = getenv("DRB_LOSS_CLUSTER") ? atoi(getenv("DRB_LOSS_CLUSTER")) : 0;   // override: 1 | 2
#define DRB_LOSS_CASE_Z(BN_, KB_, CL_, H_, Z_)                                                         \
  {                                                                                                    \
    if (loss_kind == DRB_LOSS_BCE)                                                                     \
      return per_user ? run_loss<BN_, DRB_LOSS_BCE, true, KB_, CL_, H_, Z_>(ctx, o, p, n_blocks_out)   \
                      : run_loss<BN_, DRB_LOSS_BCE, false, KB_, CL_, H_, Z_>(ctx, o, p, n_blocks_out); \
    return per_user ? run_loss<BN_, DRB_LOSS_MSE, true, KB_, CL_, H_, Z_>(ctx, o, p, n_blocks_out)     \
                    : run_loss<BN_, DRB_LOSS_MSE, false, KB_, CL_, H_, Z_>(ctx, o, p, n_blocks_out);   \
  }
#define DRB_LOSS_CASE(BN_, KB_, CL_)                                                                   \
  {                                                                                                    \
    if (o.half) {                                                                                      \
      if (p.z_dbg) DRB_LOSS_CASE_Z(BN_, KB_, CL_, true, true)                                          \
      DRB_LOSS_CASE_Z(BN_, KB_, CL_, true, false)                                                      \
    }                                                                                                  \
    if (p.z_dbg) DRB_LOSS_CASE_Z(BN_, KB_, CL_, false, true)                                           \
    DRB_LOSS_CASE_Z(BN_, KB_, CL_, false, false)                                                       \
  }
  // 128-byte stages only: the persistent loop keeps TMA ahead across tiles (64-byte stages measured 0.31 vs 0.30 ms)
  if (wide) {
    if ((cl_env ? cl_env : DRB_LOSS_CLUSTER_DEFAULT) == 2) DRB_LOSS_CASE(256, 32, 2)
    DRB_LOSS_CASE(256, 32, 1)
  }
  DRB_LOSS_CASE(128, 32, 1)
#undef DRB_LOSS_CASE
#undef DRB_LOSS_CASE_Z
}
