// C-ABI entry points of libdrb.so: context, CDAE and DMF step / scoring orchestration (see include/drb.h).
// The step functions only enqueue kernels on the context's stream; nothing here allocates device memory.
#include <algorithm>
#include <cstring>
#include <vector>

#include "kernels.h"

// ------------------------------------------------------------------------------------------ errors
static thread_local char g_err[512] = "";

int drb_fail(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  return code;
}

namespace {

struct Carver {  // bump allocator over the caller-provided workspace (256-byte aligned pieces)
  char* base; int64_t off = 0;
  explicit Carver(void* p) : base(static_cast<char*>(p)) {}
  template <typename T>
  T* take(int64_t count) {
    T* r = base ? reinterpret_cast<T*>(base + off) : nullptr;
    off += drb_round_up(count * (int64_t)sizeof(T), 256);
    return r;
  }
};

// upper bound on the row blocks k_dz1 / k_colpart use for any batch <= max_batch (8 rows per block, 4 below 2048 rows)
int colpart_blocks(int max_batch) { return std::max((max_batch + 7) / 8, (std::min(max_batch, 2047) + 3) / 4); }

// Argument checks of a pair-scoring call (drb_cdae_predict_pairs / drb_dmf_predict_pairs): host-side ones, then the
// device arrays are checked by one kernel whose verdict (one int in `flag_dev`, a scratch word) is read back here.
int pair_args_check(drb_ctx* ctx, const char* fn, const PairArgs& p, int n_users, int n_items, int* flag_dev) {
  if (p.n_u < 0 || p.n < 0) return drb_fail(DRB_E_INVALID, "%s: n_users %d, n %d", fn, p.n_u, p.n);
  if (!p.users || !p.pair_off || (p.n > 0 && (!p.pair_iid || !p.pair_dst)))
    return drb_fail(DRB_E_INVALID, "%s: NULL argument", fn);
  int r = launch_pair_args_check(ctx, p, n_users, n_items, flag_dev);
  if (r) return r;
  int bad = 0;
  DRB_CUDA_TRY(ctx, cudaMemcpyAsync(&bad, flag_dev, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
  DRB_CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
  if (bad & 1) return drb_fail(DRB_E_INVALID, "%s: a user id is outside [0, %d)", fn, n_users);
  if (bad & 2) return drb_fail(DRB_E_INVALID, "%s: pair_off must rise from 0 to n = %d", fn, p.n);
  if (bad & 4) return drb_fail(DRB_E_INVALID, "%s: an item id is outside [0, %d)", fn, n_items);
  if (bad & 8) return drb_fail(DRB_E_INVALID, "%s: an output position is outside [0, %d)", fn, p.n);
  return DRB_OK;
}

int gemm_splits(const drb_ctx* ctx, int M, int N, int Kred) {
  const int tiles = ((M + 127) / 128) * ((N + 127) / 128);
  int s = (2 * ctx->sm_count + tiles - 1) / tiles;
  s = std::min(s, std::max(1, Kred / 512));
  return std::max(1, std::min(s, 32));
}

}  // namespace

extern "C" {

int drb_version(void) { return DRB_VERSION; }
const char* drb_last_error(void) { return g_err; }

int drb_ctx_create(int device, drb_ctx** out) {
  if (!out) return drb_fail(DRB_E_INVALID, "drb_ctx_create: out is NULL");
  int count = 0;
  if (cudaGetDeviceCount(&count) != cudaSuccess || count == 0) {
    cudaGetLastError();
    return drb_fail(DRB_E_NODEVICE, "no CUDA device available (libdrb has no CPU fallback)");
  }
  if (device < 0 || device >= count) return drb_fail(DRB_E_INVALID, "device ordinal %d out of range", device);
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, device) != cudaSuccess)
    return drb_fail(DRB_E_CUDA, "cudaGetDeviceProperties failed");
  if (prop.major != 10)
    return drb_fail(DRB_E_NODEVICE, "device %d is sm_%d%d; libdrb is built for sm_100a only", device, prop.major,
                    prop.minor);
  drb_ctx* c = new (std::nothrow) drb_ctx;
  if (!c) return drb_fail(DRB_E_NOMEM, "out of memory");
  c->device = device;
  c->sm_count = prop.multiProcessorCount;
  c->stream = nullptr;
  c->launches = 0;
  c->sticky = 0;
  c->profile = 0;
  if (cudaSetDevice(device) != cudaSuccess) {
    delete c;
    return drb_fail(DRB_E_CUDA, "cudaSetDevice(%d) failed", device);
  }
  *out = c;
  return DRB_OK;
}
int drb_ctx_destroy(drb_ctx* ctx) { delete ctx; return DRB_OK; }
int drb_ctx_set_stream(drb_ctx* ctx, void* stream) {
  if (!ctx) return drb_fail(DRB_E_INVALID, "ctx is NULL");
  ctx->stream = static_cast<cudaStream_t>(stream);
  return DRB_OK;
}
int drb_ctx_synchronize(drb_ctx* ctx) {
  if (!ctx) return drb_fail(DRB_E_INVALID, "ctx is NULL");
  DRB_CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
  return DRB_OK;
}
int64_t drb_ctx_launch_count(const drb_ctx* ctx) { return ctx ? ctx->launches : 0; }

int drb_ctx_profile_enable(drb_ctx* ctx, int on) {
  if (!ctx) return drb_fail(DRB_E_INVALID, "ctx is NULL");
  ctx->profile = on ? 1 : 0;
  return DRB_OK;
}

int drb_ctx_profile_read(drb_ctx* ctx, char* names, int64_t names_cap, double* total_ms, int64_t* counts,
                         int32_t max_entries, int32_t* n_entries) {
  if (!ctx || !names || !total_ms || !counts || !n_entries || names_cap < 1)
    return drb_fail(DRB_E_INVALID, "drb_ctx_profile_read: bad argument");
  DRB_CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
  std::vector<const char*> keys;
  std::vector<double> ms;
  std::vector<int64_t> cnt;
  for (auto& r : ctx->recs) {
    float t = 0.f;
    cudaEventElapsedTime(&t, r.beg, r.end);
    cudaEventDestroy(r.beg);
    cudaEventDestroy(r.end);
    size_t k = 0;
    for (; k < keys.size(); k++) if (!std::strcmp(keys[k], r.name)) break;
    if (k == keys.size()) { keys.push_back(r.name); ms.push_back(0.0); cnt.push_back(0); }
    ms[k] += t; cnt[k] += 1;
  }
  ctx->recs.clear();
  names[0] = 0;
  int n = 0;
  int64_t used = 0;
  for (size_t k = 0; k < keys.size() && n < max_entries; k++) {
    const int64_t len = (int64_t)std::strlen(keys[k]);
    if (used + len + 2 > names_cap) break;
    std::memcpy(names + used, keys[k], len);
    names[used + len] = '\n';
    used += len + 1;
    names[used] = 0;
    total_ms[n] = ms[k]; counts[n] = cnt[k];
    n++;
  }
  *n_entries = n;
  return DRB_OK;
}

int drb_debug_split_tf32(drb_ctx* ctx, const float* src, int32_t rows, int32_t cols, int32_t ld, float* hi, float* lo,
                         float* t_hi, float* t_lo, int32_t ldt, int32_t ones_row) {
  if (!ctx || !src) return drb_fail(DRB_E_INVALID, "drb_debug_split_tf32: NULL argument");
  return launch_split_tf32(ctx, src, rows, cols, ld, hi, lo, t_hi, t_lo, ldt, ones_row);
}

int drb_debug_umma_gemm(drb_ctx* ctx, const float* a_hi, const float* a_lo, int32_t lda, const float* b_hi,
                        const float* b_lo, int32_t ldb, int32_t b_rows, int32_t a_mn_major, int32_t M, int32_t N,
                        int32_t Kred, int32_t splits, float* C, int32_t ldc, int32_t n_store, float* extra_col,
                        int32_t extra_col_index) {
  if (!ctx || !a_hi || !a_lo || !b_hi || !b_lo || !C) return drb_fail(DRB_E_INVALID, "drb_debug_umma_gemm: NULL argument");
  if (!umma_available()) return drb_fail(DRB_E_NODEVICE, "tcgen05/TMA path unavailable");
  UmmaOperands o{a_hi, a_lo, lda, b_hi, b_lo, ldb, b_rows};
  return launch_umma_store(ctx, o, a_mn_major != 0, M, N, Kred, splits, C, ldc, n_store, n_store, extra_col,
                           extra_col_index);
}

int drb_mt_keep_device(drb_ctx* ctx, const uint32_t* window_in, uint32_t* window_out, const uint64_t* polys,
                       const uint64_t* poly_total, const int32_t* uids, const int32_t* keep_off, const int64_t* csr_indptr,
                       const int32_t* csr_indices, uint8_t* keep, int32_t batch, int32_t n_items, int32_t users_per_cta,
                       uint64_t threshold) {
  if (!ctx || !window_in || !window_out || !poly_total || !uids || !keep_off || !csr_indptr || !csr_indices || !keep)
    return drb_fail(DRB_E_INVALID, "drb_mt_keep_device: NULL argument");
  if (batch <= 0 || n_items <= 0 || users_per_cta < 1) return drb_fail(DRB_E_INVALID, "drb_mt_keep_device: bad sizes");
  MtKeepArgs a{};
  a.window_in = window_in; a.window_out = window_out; a.polys = polys; a.poly_total = poly_total;
  a.uids = uids; a.keep_off = keep_off; a.indptr = csr_indptr; a.indices = csr_indices; a.keep = keep;
  a.batch = batch; a.n_items = n_items; a.ups = users_per_cta; a.n_cta = (batch + users_per_cta - 1) / users_per_cta;
  a.threshold = threshold;
  if (a.n_cta > 1 && !polys) return drb_fail(DRB_E_INVALID, "drb_mt_keep_device: jump polynomials missing");
  return launch_mt_keep(ctx, a);
}

int drb_debug_split_f16(drb_ctx* ctx, const float* src, int32_t rows, int32_t cols, int32_t ld, float alpha, void* hi,
                        void* lo, int32_t ldh, void* t_hi, void* t_lo, int32_t ldt, int32_t ones_row) {
  if (!ctx || !src) return drb_fail(DRB_E_INVALID, "drb_debug_split_f16: NULL argument");
  return launch_split_f16(ctx, src, rows, cols, ld, alpha, nullptr, hi, lo, ldh, t_hi, t_lo, ldt, ones_row);
}

int drb_debug_umma_gemm_f16(drb_ctx* ctx, const void* a_hi, const void* a_lo, int32_t lda, const void* b_hi,
                            const void* b_lo, int32_t ldb, int32_t b_rows, int32_t a_mn_major, int32_t M, int32_t N, int32_t Kred,
                            int32_t splits, float out_scale, float* C, int32_t ldc, int32_t n_store, float* extra_col,
                            int32_t extra_col_index) {
  if (!ctx || !a_hi || !a_lo || !b_hi || !b_lo || !C) return drb_fail(DRB_E_INVALID, "drb_debug_umma_gemm_f16: NULL argument");
  if (!umma_available()) return drb_fail(DRB_E_NODEVICE, "tcgen05/TMA path unavailable");
  UmmaOperands o{a_hi, a_lo, lda, b_hi, b_lo, ldb, b_rows};
  o.half = true; o.out_scale = out_scale;
  return launch_umma_store(ctx, o, a_mn_major != 0, M, N, Kred, splits, C, ldc, n_store, n_store, extra_col, extra_col_index);
}

}  // extern "C"

// ========================================================================================== step graphs
// CUDA-graph replay of a training step for the launch-bound shapes (a few microseconds per kernel).  One instantiated
// graph per argument set: the captured step reads its batch from the model's own buffers and its per-step scalars
// from device memory, which a one-thread kernel (k_set_scalars) refreshes before every replay.
struct StepGraphKey {   // a model fills the fields its step depends on and leaves the others zero
  const void* loss_out; int32_t batch, phases, global_batch, has_keep;
  float beta1, beta2, eps, reg; uint64_t philox_seed;
  bool operator==(const StepGraphKey& o) const {   // field by field: a NaN hyper-parameter never matches
    return loss_out == o.loss_out && batch == o.batch && phases == o.phases && global_batch == o.global_batch &&
           has_keep == o.has_keep && beta1 == o.beta1 && beta2 == o.beta2 && eps == o.eps && reg == o.reg &&
           philox_seed == o.philox_seed;
  }
};

struct StepGraphs {
  struct Entry { StepGraphKey key; cudaGraphExec_t exec; int64_t launches; };
  static constexpr int kSlots = 8;          // live graphs; beyond that a capture replaces one, round robin
  static constexpr int kMaxCaptures = 32;   // a caller that keeps changing the argument set would pay a capture per step
  Entry slots[kSlots];                      // [0, n_live) hold live execs
  int n_live = 0, next = 0, n_captures = 0;
  bool off;                                 // direct launches: DRB_GRAPH=0, or graphs were given up
  cudaStream_t stream = nullptr;            // capture happens here (the caller's stream may be the legacy default stream)

  StepGraphs() { const char* ge = getenv("DRB_GRAPH"); off = ge && atoi(ge) == 0; }
  StepGraphs(const StepGraphs&) = delete;   // owns the execs and the stream
  StepGraphs& operator=(const StepGraphs&) = delete;
  ~StepGraphs() {
    clear();
    if (stream) cudaStreamDestroy(stream);
  }

  // The entry for `key`.  On a miss `body()` (the step, enqueued on ctx->stream) is captured: nothing executes and its
  // launches are not counted.  nullptr: graphs are off -- from now on if the capture failed or too many were taken --
  // and the caller launches the step directly.
  template <class Body>
  Entry* get(drb_ctx* ctx, const StepGraphKey& key, Body&& body) {
    if (off) return nullptr;
    for (int i = 0; i < n_live; i++)
      if (slots[i].key == key) return &slots[i];
    if (++n_captures <= kMaxCaptures &&
        (stream || cudaStreamCreateWithFlags(&stream, cudaStreamNonBlocking) == cudaSuccess)) {
      cudaStream_t user = ctx->stream;
      const int64_t before = ctx->launches;
      cudaGraph_t graph = nullptr;
      cudaGraphExec_t exec = nullptr;
      int r = DRB_OK;
      cudaError_t e = cudaStreamBeginCapture(stream, cudaStreamCaptureModeThreadLocal);
      if (e == cudaSuccess) {
        ctx->stream = stream;
        r = body();
        ctx->stream = user;
        e = cudaStreamEndCapture(stream, &graph);
      }
      if (e == cudaSuccess && r == DRB_OK) e = cudaGraphInstantiate(&exec, graph, 0);
      if (graph) cudaGraphDestroy(graph);
      const int64_t captured = ctx->launches - before;
      ctx->launches = before;
      if (e == cudaSuccess && r == DRB_OK) {
        if (n_live == kSlots) cudaGraphExecDestroy(slots[next % kSlots].exec);
        Entry& s = slots[n_live < kSlots ? n_live++ : next++ % kSlots];
        s = Entry{key, exec, captured};
        return &s;
      }
    }
    cudaGetLastError();   // e.g. a driver without capture support for some node, or too many captures
    ctx->sticky = 0;
    off = true;
    return nullptr;
  }

  // refresh the n per-step scalars at scal_dev, then replay; counts k_set_scalars and the captured launches
  int replay(drb_ctx* ctx, const Entry* g, float* scal_dev, const float* vals, int n) {
    int r = launch_set_scalars(ctx, scal_dev, vals, n);
    if (r) return r;
    DRB_CUDA_TRY(ctx, cudaGraphLaunch(g->exec, ctx->stream));
    ctx->launches += g->launches;
    return DRB_OK;
  }

  void clear() {   // drops every graph; the capture count stays
    for (int i = 0; i < n_live; i++) cudaGraphExecDestroy(slots[i].exec);
    n_live = next = 0;
  }
};

// ========================================================================================== CDAE
struct CdaeWs {
  float *h, *dz, *dh_part, *dz1, *col_b2, *col_b, *loss_part, *reg_part, *label_count, *loss_scalar;
  // tcgen05 path: tf32 hi/lo operand splits (dz doubles as dz_hi)
  float *h_hi, *h_lo, *hT_hi, *hT_lo, *w2t_hi, *w2t_lo, *wT_hi, *wT_lo, *dzt_hi, *dzt_lo;   // dzt_*: tile-major dz
  int64_t hT_floats, wT_floats;
  uint32_t* label_bits;
  uint32_t* row_touched;         // bit u: dV[u] received a gradient row this step (see AdamArgs::row_mask)
  int32_t *uids, *keep_off, *aux_i32, *chunk_off;
  uint8_t* keep;
  int64_t bytes;
};

struct drb_cdae {
  drb_ctx* ctx;
  drb_cdae_desc d;
  drb_cdae_layout_t L;
  CdaeWs ws;
  int splits, words_per_row;
  int64_t keep_cap;
  bool use_umma;
  bool half;           // tensor-core operands are fp16 hi/lo pairs (kind::f16, per-tensor power-of-two scaling); else tf32 hi/lo
  int ldh, bp8, ip8;   // fp16 row pitches in halfs (multiples of 8): h / W' rows, transposed h, transposed W'
  bool v_grad_clean;   // the dV region of the gradient arena is known to be all zero
  int n_loss_blocks;
  const int32_t* rows_uids; int rows_n;   // user rows added by the last drb_cdae_scatter_user_rows (re-zeroed after Adam)
  bool reg_slots_clear;                   // the three reg_part slots were zeroed in PREP (split UPDATE of this step)
  int n2, batch_pad;   // tcgen05 path: N of the backward GEMMs (hidden + ones feature, rounded to 16), padded batch
  float* z_dbg;        // tests only: drb_debug_cdae_capture_logits
  drb_optim_desc opt;  // drb_cdae_set_optimizer (opt_set == false: Adam with the step args' beta1 / beta2 / epsilon)
  bool opt_set;
  // the whole step of the launch-bound shapes (ml-100k: ~15 launches) replayed from the uids / keep_off / keep
  // buffers above, with the five Adam step sizes and the philox step at ws.loss_scalar + 8
  StepGraphs graphs;
};

// N of the backward GEMMs: hidden plus the constant-one feature that folds db' = colsum(dz) into dW'^T, rounded to 16.
// tcgen05 tiles are at most 256 wide: for hidden = 256 the feature does not fit and the loss kernel accumulates db'
// itself (cdae_colsum_in_loss); for hidden in 241..255 it is the last column of a 256-wide tile.
static bool cdae_colsum_in_loss(int hidden) { return drb_round_up(hidden + 1, 16) > 256 && hidden <= 256; }
static int cdae_n2(int hidden) { return (int)drb_round_up(hidden + (cdae_colsum_in_loss(hidden) ? 0 : 1), 16); }

static int64_t cdae_keep_cap(int32_t n_items, int32_t max_batch) {
  // every sampled user can hold at most n_items positives; cap the staging buffer at 1 GiB
  return std::min<int64_t>((int64_t)max_batch * n_items, (int64_t)1 << 30);
}

static CdaeWs cdae_carve(void* base, const drb_cdae_layout_t& L, int n_users, int n_items, int hidden, int max_batch,
                         int label_mode, int splits, int sm_count, bool umma, bool sampled = false) {
  Carver c(base);
  CdaeWs w{};
  const int64_t B = max_batch;
  const int mt = (max_batch + 127) / 128;
  w.h = c.take<float>(B * L.ld);
  w.row_touched = c.take<uint32_t>((n_users + 31) / 32 + 8);
  // sampled-output models never form batch x items matrices: no dz, no per-tile column partials, a batch-sized loss buffer
  w.dz = c.take<float>(sampled ? 64 : B * L.items_pad);
  if (sampled) {
    w.dh_part = c.take<float>(B * L.ld);
    w.dz1 = c.take<float>(B * L.ld);
    w.col_b2 = c.take<float>(64);
    w.col_b = c.take<float>((int64_t)colpart_blocks(max_batch) * L.ld);
    w.loss_part = c.take<float>(B);
    w.reg_part = c.take<float>((int64_t)sm_count * 16 * 3);
    w.label_count = c.take<float>(64);
    w.loss_scalar = c.take<float>(64);
    w.label_bits = c.take<uint32_t>(1);
    w.uids = c.take<int32_t>(B);
    w.keep_off = c.take<int32_t>(B + 1);
    w.aux_i32 = c.take<int32_t>(3 * B + 64);
    w.chunk_off = c.take<int32_t>(B + 64);
    w.keep = c.take<uint8_t>(cdae_keep_cap(n_items, max_batch));
    w.bytes = c.off;
    return w;
  }
  w.dh_part = c.take<float>((int64_t)splits * B * L.ld);
  w.dz1 = c.take<float>(B * L.ld);
  w.col_b2 = c.take<float>((int64_t)mt * L.items_pad);
  w.col_b = c.take<float>((int64_t)colpart_blocks(max_batch) * L.ld);
  w.loss_part = c.take<float>((int64_t)mt * ((L.items_pad + 63) / 64));
  w.reg_part = c.take<float>((int64_t)sm_count * 16 * 3);   // three slots: split UPDATE launches (data parallel)
  w.label_count = c.take<float>(L.items_pad);
  w.loss_scalar = c.take<float>(64);
  const int64_t words = (L.items_pad + 31) / 32;
  w.label_bits = c.take<uint32_t>(label_mode == DRB_LABEL_PER_USER ? B * words : 1);
  w.uids = c.take<int32_t>(B);
  w.keep_off = c.take<int32_t>(B + 1);
  w.aux_i32 = c.take<int32_t>(3 * B + 64);
  w.chunk_off = c.take<int32_t>(B + 64);
  w.keep = c.take<uint8_t>(cdae_keep_cap(n_items, max_batch));
  if (umma) {
    // sized for tf32 hi/lo floats; the fp16 hi/lo forms (pitches rounded up to 8 halfs) need at most as many bytes
    const int64_t n2 = cdae_n2(hidden), bp = drb_round_up(max_batch, 8);
    w.h_hi = c.take<float>(B * (L.ld + 4));
    w.h_lo = c.take<float>(B * (L.ld + 4));
    w.hT_floats = n2 * bp;
    w.hT_hi = c.take<float>(w.hT_floats);
    w.hT_lo = c.take<float>(w.hT_floats);
    w.w2t_hi = c.take<float>((int64_t)n_items * (L.ld + 4));
    w.w2t_lo = c.take<float>((int64_t)n_items * (L.ld + 4));
    w.wT_floats = n2 * (int64_t)drb_round_up(L.items_pad, 8);
    w.wT_hi = c.take<float>(w.wT_floats);
    w.wT_lo = c.take<float>(w.wT_floats);
    w.dzt_hi = c.take<float>(drb_dz_tiled_floats(max_batch, n_items));
    w.dzt_lo = c.take<float>(drb_dz_tiled_floats(max_batch, n_items));
  }
  w.bytes = c.off;
  return w;
}

extern "C" {

int drb_cdae_layout(int32_t n_users, int32_t n_items, int32_t hidden, drb_cdae_layout_t* out) {
  if (!out || n_users <= 0 || n_items <= 0 || hidden <= 0 || hidden > 512)
    return drb_fail(DRB_E_INVALID, "drb_cdae_layout: need n_users, n_items > 0 and 0 < hidden <= 512");
  const int64_t ld = drb_round_up(hidden, 4), ip = drb_round_up(n_items, 4);
  out->ld = (int32_t)ld;
  out->items_pad = (int32_t)ip;
  out->off_w2t = 0;
  out->off_w = out->off_w2t + (int64_t)n_items * ld;
  out->off_b = out->off_w + (int64_t)n_items * ld;
  out->off_b2 = out->off_b + ld;
  out->off_v = out->off_b2 + ip;          // V last: everything before it is all-reduced densely when data parallel
  out->total = out->off_v + (int64_t)n_users * ld;
  return DRB_OK;
}

int64_t drb_cdae_workspace_bytes(int32_t n_users, int32_t n_items, int32_t hidden, int32_t max_batch) {
  drb_cdae_layout_t L;
  if (drb_cdae_layout(n_users, n_items, hidden, &L) || max_batch <= 0) return -1;
  // worst case over label modes and split counts (splits <= 32, 148+ SMs -> use 256 as an upper bound)
  return cdae_carve(nullptr, L, n_users, n_items, hidden, max_batch, DRB_LABEL_PER_USER, 32, 256, true).bytes;
}

int64_t drb_cdae_workspace_bytes_sampled(int32_t n_users, int32_t n_items, int32_t hidden, int32_t max_batch) {
  drb_cdae_layout_t L;
  if (drb_cdae_layout(n_users, n_items, hidden, &L) || max_batch <= 0) return -1;
  return cdae_carve(nullptr, L, n_users, n_items, hidden, max_batch, DRB_LABEL_PER_USER, 1, 256, false, true).bytes;
}

int drb_cdae_create(drb_ctx* ctx, const drb_cdae_desc* desc, drb_cdae** out) {
  if (!ctx || !desc || !out) return drb_fail(DRB_E_INVALID, "drb_cdae_create: NULL argument");
  drb_cdae_layout_t L;
  int r = drb_cdae_layout(desc->n_users, desc->n_items, desc->hidden, &L);
  if (r) return r;
  if (!desc->params || !desc->csr_indptr || !desc->csr_indices || !desc->workspace || desc->max_batch <= 0)
    return drb_fail(DRB_E_INVALID, "drb_cdae_create: params, csr and workspace are required");
  if (((uintptr_t)desc->params | (uintptr_t)desc->adam_m | (uintptr_t)desc->adam_v | (uintptr_t)desc->grads |
       (uintptr_t)desc->workspace) & 15)
    return drb_fail(DRB_E_INVALID, "drb_cdae_create: arenas and workspace must be 16-byte aligned");
  if (!(desc->corruption_level >= 0.f && desc->corruption_level < 1.f))
    return drb_fail(DRB_E_INVALID, "drb_cdae_create: corruption_level must be in [0, 1)");
  if (desc->loss_kind != DRB_LOSS_BCE && desc->loss_kind != DRB_LOSS_MSE)
    return drb_fail(DRB_E_INVALID, "Loss function is not supported. Supported losses: \"mse\", \"bce\".");
  drb_cdae* m = new (std::nothrow) drb_cdae;
  if (!m) return drb_fail(DRB_E_NOMEM, "out of memory");
  m->ctx = ctx;
  m->d = *desc;
  if (!m->d.seen_indptr) { m->d.seen_indptr = m->d.csr_indptr; m->d.seen_indices = m->d.csr_indices; }
  m->L = L;
  m->splits = gemm_splits(ctx, desc->max_batch, L.ld, desc->n_items);
  m->words_per_row = (L.items_pad + 31) / 32;
  m->n2 = cdae_n2(desc->hidden);
  m->batch_pad = (int)drb_round_up(desc->max_batch, 8);
  const bool sampled = desc->output_mode == DRB_OUTPUT_SAMPLED;
  if (sampled && (desc->neg_per_group < 1 || desc->neg_groups < 1)) {
    delete m;
    return drb_fail(DRB_E_INVALID, "drb_cdae_create: sampled outputs need neg_per_group >= 1 and neg_groups >= 1");
  }
  const bool umma_ok = umma_available() && m->n2 <= 256 && !sampled;
  if ((desc->gemm_path == DRB_GEMM_TCGEN05 || desc->gemm_path == DRB_GEMM_TCGEN05_TF32) && !umma_ok) {
    delete m;
    return drb_fail(DRB_E_INVALID, "drb_cdae_create: the tcgen05 path needs hidden <= 256 and a driver with TMA support");
  }
  m->use_umma = umma_ok && desc->gemm_path != DRB_GEMM_FFMA;
  {   // DRB_GEMM_SPLIT=tf32 keeps the 3xTF32 products (profiling / comparison); default: 3xFP16 at twice the MMA rate
    const char* se = getenv("DRB_GEMM_SPLIT");
    m->half = m->use_umma && desc->gemm_path != DRB_GEMM_TCGEN05_TF32 && !(se && !strcmp(se, "tf32"));
  }
  m->ldh = (int)drb_round_up(L.ld, 8);
  m->bp8 = (int)drb_round_up(desc->max_batch, 8);
  m->ip8 = (int)drb_round_up(L.items_pad, 8);
  m->v_grad_clean = false;
  m->z_dbg = nullptr;
  std::memset(&m->opt, 0, sizeof(m->opt));
  m->opt_set = false;
  m->rows_uids = nullptr; m->rows_n = 0; m->reg_slots_clear = false;
  if (m->use_umma) {
    // dh = dz W'^T on the tensor cores has one 128 x n2 tile per 128 users: split the item range so that the grid
    // is ~2 waves of the SM count (the kernel is L2/HBM bandwidth bound, one CTA per SM)
    const int mt = (desc->max_batch + 127) / 128;
    m->splits = std::max(1, std::min(32, std::min((2 * ctx->sm_count) / mt, desc->n_items / 256)));
    if (getenv("DRB_DH_SPLITS")) m->splits = std::max(1, std::min(32, atoi(getenv("DRB_DH_SPLITS"))));   // tuning override
  }
  if (sampled) m->splits = 1;
  m->ws = cdae_carve(desc->workspace, L, desc->n_users, desc->n_items, desc->hidden, desc->max_batch, desc->label_mode,
                     m->splits, ctx->sm_count, m->use_umma, sampled);
  m->keep_cap = cdae_keep_cap(desc->n_items, desc->max_batch);
  if (m->ws.bytes <= desc->workspace_bytes)
    cudaMemsetAsync(m->ws.row_touched, 0, ((size_t)(desc->n_users + 31) / 32 + 8) * 4, ctx->stream);
  if (m->ws.bytes > desc->workspace_bytes) {
    int64_t need = m->ws.bytes;
    delete m;
    return drb_fail(DRB_E_INVALID, "drb_cdae_create: workspace too small (%lld < %lld bytes)",
                    (long long)desc->workspace_bytes, (long long)need);
  }
  if (cudaMemsetAsync(m->ws.loss_scalar, 0, 64 * sizeof(float), ctx->stream) != cudaSuccess) {   // loss, scales, ticket
    delete m;
    return drb_fail(DRB_E_CUDA, "drb_cdae_create: workspace clear failed");
  }
  if (m->use_umma) {   // transposed operand buffers: rows >= hidden stay zero (the ones row is rewritten every step)
    cudaError_t e = cudaMemsetAsync(m->ws.hT_hi, 0, (size_t)m->ws.hT_floats * 4, ctx->stream);
    if (e == cudaSuccess) e = cudaMemsetAsync(m->ws.hT_lo, 0, (size_t)m->ws.hT_floats * 4, ctx->stream);
    if (e == cudaSuccess) e = cudaMemsetAsync(m->ws.wT_hi, 0, (size_t)m->ws.wT_floats * 4, ctx->stream);
    if (e == cudaSuccess) e = cudaMemsetAsync(m->ws.wT_lo, 0, (size_t)m->ws.wT_floats * 4, ctx->stream);
    if (e != cudaSuccess) {
      delete m;
      return drb_fail(DRB_E_CUDA, "drb_cdae_create: workspace clear failed: %s", cudaGetErrorString(e));
    }
  }
  *out = m;
  return DRB_OK;
}
int drb_cdae_set_optimizer(drb_cdae* m, const drb_optim_desc* opt) {
  if (!m) return drb_fail(DRB_E_INVALID, "drb_cdae_set_optimizer: NULL model");
  int r = optim_check(opt, "drb_cdae_set_optimizer");
  if (r) return r;
  m->opt = *opt;
  m->opt_set = true;
  m->graphs.clear();   // captured steps hold the previous rule's kernel and hyper-parameters: never replay them for this one
  return DRB_OK;
}

int drb_cdae_destroy(drb_cdae* m) {
  delete m;
  return DRB_OK;
}

static int cdae_hidden_into(drb_cdae* m, const int32_t* uids, int n, const int32_t* keep_off, const uint8_t* keep,
                            float scale, float* h, int act = DRB_ACT_SIGMOID, const int32_t* bias_rows = nullptr,
                            const int32_t* chunk_off = nullptr) {
  GatherArgs g{};
  g.indptr = m->d.csr_indptr; g.indices = m->d.csr_indices; g.values = nullptr;
  g.rows = uids; g.keep_off = keep_off; g.keep = keep;
  g.table = m->d.params + m->L.off_w; g.ld = m->L.ld;
  g.rowbias = m->d.params + m->L.off_v; g.bias = m->d.params + m->L.off_b;
  g.row_scale = nullptr; g.scale = scale; g.act = act; g.width = m->d.hidden;
  g.bias_rows = bias_rows;
  g.out = h;
  g.chunk_off = chunk_off;
  return launch_gather(m->ctx, g, n);
}

int drb_cdae_step(drb_cdae* m, const int32_t* uids, const int32_t* keep_off, const uint8_t* keep, int32_t batch,
                  const drb_cdae_step_args* a, float* loss_out) {
  return drb_cdae_step_phases(m, uids, keep_off, keep, batch, a, loss_out, DRB_PHASE_ALL);
}

int drb_cdae_loss_buffer(drb_cdae* m, float** ptr) {
  if (!m || !ptr) return drb_fail(DRB_E_INVALID, "drb_cdae_loss_buffer: NULL argument");
  *ptr = m->ws.loss_scalar;
  return DRB_OK;
}

int drb_cdae_h_buffer(drb_cdae* m, float** ptr, int64_t* count) {
  if (!m || !ptr || !count) return drb_fail(DRB_E_INVALID, "drb_cdae_h_buffer: NULL argument");
  *ptr = m->ws.h;
  *count = (int64_t)m->d.max_batch * m->L.ld;
  return DRB_OK;
}

int drb_cdae_dz1_buffer(drb_cdae* m, float** ptr, int64_t* count) {
  if (!m || !ptr || !count) return drb_fail(DRB_E_INVALID, "drb_cdae_dz1_buffer: NULL argument");
  *ptr = m->ws.dz1;
  *count = (int64_t)m->d.max_batch * m->L.ld;
  return DRB_OK;
}

int drb_cdae_scatter_user_rows(drb_cdae* m, const int32_t* uids, const float* rows, int32_t n) {
  if (!m || !uids || !rows || n < 0) return drb_fail(DRB_E_INVALID, "drb_cdae_scatter_user_rows: bad argument");
  m->rows_uids = uids; m->rows_n = n;     // borrowed until the UPDATE of this step: those rows are re-zeroed after Adam
  return launch_row_scatter(m->ctx, uids, rows, n, m->L.ld, m->d.grads + m->L.off_v, m->ws.row_touched);
}

int drb_debug_cdae_capture_logits(drb_cdae* m, float* z_out) {
  if (!m) return drb_fail(DRB_E_INVALID, "drb_debug_cdae_capture_logits: NULL argument");
  if (z_out && !m->use_umma) return drb_fail(DRB_E_STATE, "drb_debug_cdae_capture_logits: the model runs the FFMA path");
  m->z_dbg = z_out;
  return DRB_OK;
}

int drb_cdae_label_count_buffer(drb_cdae* m, float** ptr, int64_t* count) {
  if (!m || !ptr || !count) return drb_fail(DRB_E_INVALID, "drb_cdae_label_count_buffer: NULL argument");
  *ptr = m->ws.label_count;
  *count = m->L.items_pad;
  return DRB_OK;
}

}  // extern "C"

// the optimizer a step runs: the model's descriptor, or Adam with the step args' hyper-parameters when none was set
static drb_optim_desc effective_optim(bool set, const drb_optim_desc& d, float beta1, float beta2, float eps) {
  if (set) return d;
  drb_optim_desc o{};
  o.kind = DRB_OPT_ADAM; o.beta1 = beta1; o.beta2 = beta2; o.epsilon = eps;
  return o;
}

// scal_dev != NULL (graph capture): the five Adam step sizes are read from scal_dev[0..4] (reference variable order
// [W, W_, V, b, b_]) and the philox step from scal_dev[5..6] (lo, hi words) -- the only per-step scalars of a step
static int cdae_step_impl(drb_cdae* m, const int32_t* uids, const int32_t* keep_off, const uint8_t* keep,
                          int32_t batch, const drb_cdae_step_args* a, float* loss_out, int32_t phases,
                          const float* scal_dev) {
  if (!m || !uids || !keep_off || !a || !loss_out) return drb_fail(DRB_E_INVALID, "drb_cdae_step: NULL argument");
  if (batch <= 0 || batch > m->d.max_batch)
    return drb_fail(DRB_E_INVALID, "drb_cdae_step: batch %d outside (0, max_batch=%d]", batch, m->d.max_batch);
  if (!m->d.adam_m || !m->d.adam_v || !m->d.grads)
    return drb_fail(DRB_E_STATE, "drb_cdae_step: model was created without optimizer arenas");
  drb_ctx* ctx = m->ctx;
  if (ctx->sticky) return drb_fail(DRB_E_CUDA, "context has a sticky CUDA error (%d)", ctx->sticky);
  const drb_cdae_layout_t& L = m->L;
  CdaeWs& w = m->ws;
  const int I = m->d.n_items, ld = L.ld;
  float* P = m->d.params;
  float* G = m->d.grads;
  const bool per_user = (m->d.label_mode == DRB_LABEL_PER_USER);
  const int gbatch = a->global_batch > 0 ? a->global_batch : batch;   // data parallel: labels / loss / reg use it
  if (gbatch < batch) return drb_fail(DRB_E_INVALID, "drb_cdae_step: global_batch %d < batch %d", gbatch, batch);
  const uint8_t* keep_used = keep ? keep : w.keep;
  if (m->d.corruption_level == 0.f) keep_used = nullptr;
  const float s = (float)(1.0 / (1.0 - (double)m->d.corruption_level));
  const bool sharded = a->shard_items != 0;       // item-sharded weights: this model holds items [item_offset, +I)
  const double items_global = sharded && a->n_items_global > 0 ? (double)a->n_items_global : (double)I;
  const bool sampled = m->d.output_mode == DRB_OUTPUT_SAMPLED;   // positives + drawn items only (extension, sampled.cu)
  const float inv_count = sampled ? (float)(1.0 / ((double)gbatch * m->d.neg_groups * m->d.neg_per_group))
                                  : (float)(1.0 / ((double)gbatch * items_global));
  int r;

  if (phases & DRB_PHASE_PREP) {
  // 0. clear sparse-gradient regions [W | V | b | b2] (W2T's gradient is fully overwritten by the GEMM)
  // (the tcgen05 path accumulates dW'^T from two reduction halves with vector atomics, so it clears that too)
  const int64_t clear_from = (m->use_umma || sampled) ? 0 : L.off_w;
  // dV (U x K, the largest gradient) is only touched in the rows of the sampled users: on the plain single-process
  // step those rows are re-zeroed after the update (k_zero_rows) instead of clearing the whole table every step
  const bool sparse_clear_v = !sharded && m->v_grad_clean;
  const int64_t clear_to = sparse_clear_v ? L.off_v : L.total;
  DRB_CUDA_TRY(ctx, cudaMemsetAsync(G + clear_from, 0, (size_t)(clear_to - clear_from) * sizeof(float), ctx->stream));
  if (!sparse_clear_v)   // dV was cleared as a whole: no row holds a gradient
    DRB_CUDA_TRY(ctx, cudaMemsetAsync(w.row_touched, 0, ((size_t)(m->d.n_users + 31) / 32 + 8) * 4, ctx->stream));
  m->v_grad_clean = false;
  m->rows_uids = nullptr; m->rows_n = 0;
  m->reg_slots_clear = false;
  if (sampled) {
    // labels are looked up per scored item; nothing to prepare but the philox mask
  } else if (per_user)
    DRB_CUDA_TRY(ctx, cudaMemsetAsync(w.label_bits, 0, (size_t)batch * m->words_per_row * 4, ctx->stream));
  else
    DRB_CUDA_TRY(ctx, cudaMemsetAsync(w.label_count, 0, (size_t)L.items_pad * 4, ctx->stream));

  // 1. labels of the batch (cdae.py:61-62) and, in counter mode, the corruption mask (cdae.py:63-64)
  BatchPrepArgs bp{};
  bp.indptr = m->d.csr_indptr; bp.indices = m->d.csr_indices; bp.rows = uids; bp.keep_off = keep_off;
  bp.count = (per_user || sampled) ? nullptr : w.label_count;
  bp.label_bits = (per_user && !sampled) ? w.label_bits : nullptr;
  bp.words_per_row = m->words_per_row;
  bp.keep_out = keep ? nullptr : w.keep;
  bp.seed = a->philox_seed; bp.step = a->philox_step; bp.q = m->d.corruption_level;
  bp.step_dev = scal_dev ? reinterpret_cast<const uint32_t*>(scal_dev + 5) : nullptr;
  bp.slot_offset = a->slot_offset;
  bp.item_offset = sharded ? a->item_offset : 0;
  if (!sampled || bp.keep_out) {
    if ((r = launch_batch_prep(ctx, bp, batch))) return r;
  }
  }  // PREP (data parallel: the caller all-reduces the label histogram here)

  const int n2 = m->n2, bp = m->batch_pad;
  if (phases & DRB_PHASE_GRADS_A) {
  // 2. K1: h = sigmoid(s * sum_kept W[i] + V[u] + b)   (needs no labels: overlaps the label all-reduce when DP).
  //    Item-sharded: the partial pre-activation over the local items (+ V_u + b on the user's owner rank); the caller
  //    all-reduces drb_cdae_h_buffer() and GRADS_A2 applies the sigmoid.
  //    Balanced over 256-entry pieces of the users' rows (training only; k_chunk_scan builds the piece map that the
  //    scatter of this step reuses).
  if ((r = launch_chunk_scan(ctx, m->d.csr_indptr, uids, batch, w.chunk_off))) return r;
  if ((r = cdae_hidden_into(m, uids, batch, keep_off, keep_used, s, w.h, sharded ? DRB_ACT_NONE : DRB_ACT_SIGMOID,
                            sharded ? a->v_rows : nullptr, w.chunk_off)))
    return r;
  }
  if ((phases & DRB_PHASE_GRADS_A2) || ((phases & DRB_PHASE_GRADS_A) && !sharded)) {
  if (sharded && (r = launch_sigmoid_rows(ctx, w.h, batch, ld, m->d.hidden))) return r;
  if (m->use_umma && m->half) {
    // fp16 hi/lo operand splits.  h is in (0, 1): fixed scale 2^15.  W' is scaled by a power of two alpha_w that puts its
    // largest magnitude in [2^14, 2^15) (k_absmax, then k_publish_scale: scales[0] = alpha_w, scales[1] = 1 / alpha_w).
    float* scales = w.loss_scalar + 32;
    const int ones = cdae_colsum_in_loss(m->d.hidden) ? -1 : m->d.hidden;
    if ((r = launch_split_f16(ctx, w.h, batch, ld, ld, DRB_H_F16_SCALE, nullptr, w.h_hi, w.h_lo, m->ldh, w.hT_hi, w.hT_lo,
                              m->bp8, ones)))
      return r;
    if ((r = launch_absmax_scale(ctx, P + L.off_w2t, I, m->d.hidden, ld, scales))) return r;
    if ((r = launch_split_f16(ctx, P + L.off_w2t, I, ld, ld, 1.0f, scales, w.w2t_hi, w.w2t_lo, m->ldh, w.wT_hi, w.wT_lo,
                              m->ip8, -1)))
      return r;
  } else if (m->use_umma) {   // tf32 hi/lo operand splits for the tensor-core GEMMs (umma.cu)
    if ((r = launch_split_tf32(ctx, w.h, batch, ld, ld, w.h_hi, w.h_lo, w.hT_hi, w.hT_lo, bp,
                               cdae_colsum_in_loss(m->d.hidden) ? -1 : m->d.hidden)))
      return r;
    if ((r = launch_split_tf32(ctx, P + L.off_w2t, I, ld, ld, w.w2t_hi, w.w2t_lo, w.wT_hi, w.wT_lo, L.items_pad, -1)))
      return r;
  }
  }

  // fp16 dz: two tile-major copies inside the dzt buffers (kernels.h: DzHalf), hi in the first half, lo in the second
  DzHalf dzh{};
  const float* inv_alpha_w = w.loss_scalar + 33;
  if (m->use_umma && m->half) {
    const int64_t half_bytes = drb_dz_tiled_floats(m->d.max_batch, I) * 2;     // bytes of one hi (or lo) copy
    dzh.row_tiles = (m->d.max_batch + 127) / 128; dzh.item_tiles = (I + 127) / 128;
    dzh.nib64 = drb_dz_nib64(I); dzh.nub = 2 * dzh.row_tiles;
    dzh.u_hi = w.dzt_hi; dzh.u_lo = reinterpret_cast<char*>(w.dzt_hi) + half_bytes;
    // one copy of dz (U) serves both backward GEMMs: dh reads it K-major, dW'^T reads it transposed through the MN-major
    // descriptor.  DRB_DZ_COPIES=2 also writes the [item tile][user block] copy and feeds dW'^T from it (the round's
    // first form: 0.1 ms of extra store time in the loss kernel).
    static const bool two_copies = getenv("DRB_DZ_COPIES") && atoi(getenv("DRB_DZ_COPIES")) == 2;
    if (two_copies) { dzh.i_hi = w.dzt_lo; dzh.i_lo = reinterpret_cast<char*>(w.dzt_lo) + half_bytes; }
  }
  const float dz_unscale = inv_count / DRB_DZ_F16_SCALE;      // fp16 dz holds dL/dz2 * 2^14 / inv_count

  UmmaOperands o2{w.dzt_hi, w.dzt_lo, 32, w.hT_hi, w.hT_lo, bp, n2};
  o2.a_tiled_nib = drb_dz_nib(I);
  o2.a_tiled_rows = (int64_t)((m->d.max_batch + 127) / 128) * o2.a_tiled_nib * 128;
  if ((phases & DRB_PHASE_GRADS_B) && sampled) {
    // 3-5 in one kernel: output layer over positives + drawn items, loss terms, dW'^T / db' (atomics), dh
    SampledOutArgs so{};
    so.indptr = m->d.csr_indptr; so.indices = m->d.csr_indices; so.rows = uids;
    so.h = w.h; so.ld = ld; so.w2t = P + L.off_w2t; so.b2 = P + L.off_b2;
    so.g_w2t = G + L.off_w2t; so.g_b2 = G + L.off_b2; so.dh = w.dh_part; so.loss_part = w.loss_part;
    so.n_items_total = sharded && a->n_items_global > 0 ? (int)a->n_items_global : I;
    so.n_groups_total = m->d.neg_groups;
    so.n_groups = sharded ? 1 : m->d.neg_groups;
    so.item_offset = sharded ? a->item_offset : 0;
    const int per_g = (so.n_items_total + so.n_groups_total - 1) / so.n_groups_total;
    so.group_id0 = sharded ? a->item_offset / per_g : 0;
    if (sharded && (a->item_offset % per_g != 0 || I > per_g))
      return drb_fail(DRB_E_INVALID, "drb_cdae_step: item-sharded sampled outputs need one negative-sampling group per shard");
    so.neg_per_group = m->d.neg_per_group;
    so.seed = a->philox_seed; so.step = a->philox_step;
    so.step_dev = scal_dev ? reinterpret_cast<const uint32_t*>(scal_dev + 5) : nullptr;
    so.slot_offset = a->slot_offset; so.loss_kind = m->d.loss_kind; so.inv_count = inv_count;
    if ((r = launch_sampled_out(ctx, so, batch))) return r;
    m->n_loss_blocks = batch;
  } else
  if (phases & DRB_PHASE_GRADS_B) {
  int n_blocks = 0;
  if (m->use_umma) {
    // 3-4 on the tensor cores: fp32-accurate split products (3xFP16 or 3xTF32), TMA-fed, TMEM accumulators
    UmmaOperands o1{w.h_hi, w.h_lo, m->half ? m->ldh : ld, w.w2t_hi, w.w2t_lo, m->half ? m->ldh : ld, I};
    if (m->half) { o1.half = true; o1.out_scale = 1.0f / DRB_H_F16_SCALE; o1.out_scale_dev = inv_alpha_w; }
    dzh.row_tiles = (batch + 127) / 128;        // row tiles that exist for THIS batch (the layout pitch is nub / nib64)
    if ((r = launch_umma_cdae_loss(ctx, o1, batch, I, ld, w.dzt_hi, w.dzt_lo, L.items_pad, P + L.off_b2,
                                   per_user ? nullptr : w.label_count, per_user ? w.label_bits : nullptr,
                                   m->words_per_row, m->d.loss_kind, inv_count, gbatch, w.loss_part,
                                   cdae_colsum_in_loss(m->d.hidden) ? G + L.off_b2 : nullptr, &n_blocks, m->z_dbg,
                                   L.items_pad, m->half ? &dzh : nullptr)))
      return r;
    // dW'^T = dz^T h (I x K); the constant-one feature at column `hidden` yields db' = colsum(dz)
    // e.g. 209 item tiles on 148 SMs would run as two uneven waves: split the batch reduction so the grid is ~2 waves
    // (the partial products accumulate with vector atomics into the pre-zeroed gradient)
    const int mt2 = (I + 127) / 128;
    static const int s2_env = getenv("DRB_DW_SPLITS") ? atoi(getenv("DRB_DW_SPLITS")) : 0;             // tuning override
    const int s2 = batch >= 1024 ? std::max(1, std::min({16, s2_env > 0 ? s2_env : (2 * ctx->sm_count + mt2 - 1) / mt2, batch / 512})) : 1;
    const bool colsum = cdae_colsum_in_loss(m->d.hidden);
    if (m->half && dzh.i_hi) {      // A = the [item tile][user block] copy of dz (K-major over users), B = h^T
      UmmaOperands oh{dzh.i_hi, dzh.i_lo, 64, w.hT_hi, w.hT_lo, m->bp8, n2};
      oh.a_tiled_nib = dzh.nub; oh.a_tiled_rows = (int64_t)dzh.item_tiles * dzh.nub * 128;
      oh.half = true; oh.out_scale = dz_unscale / DRB_H_F16_SCALE; oh.name = "k_umma_gemm_dw";
      if ((r = launch_umma_store(ctx, oh, false, I, n2, batch, s2, G + L.off_w2t, ld, ld, m->d.hidden,
                                 colsum ? nullptr : G + L.off_b2, colsum ? -1 : m->d.hidden, s2 > 1)))
        return r;
    } else if (m->half) {           // A = the one [user tile][item block] copy of dz, read MN-major (m = items contiguous)
      UmmaOperands oh{dzh.u_hi, dzh.u_lo, 64, w.hT_hi, w.hT_lo, m->bp8, n2};
      oh.a_tiled_nib = dzh.nib64; oh.a_tiled_rows = (int64_t)((m->d.max_batch + 127) / 128) * dzh.nib64 * 128;
      oh.half = true; oh.out_scale = dz_unscale / DRB_H_F16_SCALE; oh.name = "k_umma_gemm_dw";
      if ((r = launch_umma_store(ctx, oh, true, I, n2, batch, s2, G + L.off_w2t, ld, ld, m->d.hidden,
                                 colsum ? nullptr : G + L.off_b2, colsum ? -1 : m->d.hidden, s2 > 1)))
        return r;
    } else
    if ((r = launch_umma_store(ctx, o2, true, I, n2, batch, s2, G + L.off_w2t, ld, ld, m->d.hidden,
                               colsum ? nullptr : G + L.off_b2, colsum ? -1 : m->d.hidden, s2 > 1)))
      return r;
  } else {
  // 3. K2: z2 = h W'^T + b', p = sigmoid, loss terms, dL/dz2 (never materialises p)
  GemmArgs g1{};
  g1.A = w.h; g1.lda = ld; g1.B = P + L.off_w2t; g1.ldb = ld; g1.C = w.dz; g1.ldc = L.items_pad;
  g1.M = batch; g1.N = I; g1.Kred = ld; g1.splits = 1;
  g1.bias = P + L.off_b2;
  g1.label_count = per_user ? nullptr : w.label_count;
  g1.label_bits = per_user ? w.label_bits : nullptr; g1.words_per_row = m->words_per_row;
  g1.loss_kind = m->d.loss_kind; g1.inv_count = inv_count; g1.batch = gbatch;
  g1.loss_part = w.loss_part; g1.col_part = w.col_b2;
  int n_mtiles = 0;
  if ((r = launch_gemm(ctx, LAYOUT_KK, EPI_CDAE_LOSS, g1, &n_mtiles, &n_blocks))) return r;
  if ((r = launch_reduce_partials(ctx, w.col_b2, n_mtiles, L.items_pad, G + L.off_b2, L.items_pad))) return r;

  // 4. K3: dW'^T = dz^T h   (I x K)
  GemmArgs g2{};
  g2.A = w.dz; g2.lda = L.items_pad; g2.B = w.h; g2.ldb = ld; g2.C = G + L.off_w2t; g2.ldc = ld;
  g2.M = I; g2.N = ld; g2.Kred = batch; g2.splits = 1;
  if ((r = launch_gemm(ctx, LAYOUT_MN, EPI_STORE, g2))) return r;
  }
  m->n_loss_blocks = n_blocks;
  }  // GRADS_B (data parallel: dW'^T and db' can be all-reduced from here on)

  if (phases & DRB_PHASE_GRADS_C) {
  // 5. K3: dh = dz W'^T  (B x K), split over the item range, partials reduced by the dz1 kernel
  if (sampled) {
    // dh already sits in plane 0 of dh_part (k_sampled_out)
  } else if (m->use_umma && m->half) {      // A = the [user tile][item block] copy of dz (K-major over items), B = W'^T
    UmmaOperands o3{dzh.u_hi, dzh.u_lo, 64, w.wT_hi, w.wT_lo, m->ip8, n2};
    o3.a_tiled_nib = dzh.nib64; o3.a_tiled_rows = (int64_t)((m->d.max_batch + 127) / 128) * dzh.nib64 * 128;
    o3.half = true; o3.out_scale = dz_unscale; o3.out_scale_dev = inv_alpha_w; o3.name = "k_umma_gemm_dh";
    if ((r = launch_umma_store(ctx, o3, false, batch, n2, I, m->splits, w.dh_part, ld, ld, m->d.hidden, nullptr, -1)))
      return r;
  } else if (m->use_umma) {
    UmmaOperands o3{w.dzt_hi, w.dzt_lo, 32, w.wT_hi, w.wT_lo, L.items_pad, n2};
    o3.a_tiled_nib = o2.a_tiled_nib;
    o3.a_tiled_rows = o2.a_tiled_rows;
    if ((r = launch_umma_store(ctx, o3, false, batch, n2, I, m->splits, w.dh_part, ld, ld, m->d.hidden, nullptr, -1)))
      return r;
  } else {
  GemmArgs g3{};
  g3.A = w.dz; g3.lda = L.items_pad; g3.B = P + L.off_w2t; g3.ldb = ld; g3.C = w.dh_part; g3.ldc = ld;
  g3.M = batch; g3.N = ld; g3.Kred = I; g3.splits = m->splits;
  if ((r = launch_gemm(ctx, LAYOUT_KN, EPI_STORE, g3))) return r;
  }
  if (sharded) {   // dh partial over the local items -> one plane; the caller all-reduces drb_cdae_dz1_buffer()
    if ((r = launch_sum_planes(ctx, w.dh_part, m->splits, (int64_t)batch * ld, w.dz1))) return r;
  }
  }
  if ((phases & DRB_PHASE_GRADS_C2) || ((phases & DRB_PHASE_GRADS_C) && !sharded)) {
  int nb = sharded ? launch_dz1(ctx, w.dz1, 1, w.h, w.dz1, batch, ld, w.col_b)
                   : launch_dz1(ctx, w.dh_part, m->splits, w.h, w.dz1, batch, ld, w.col_b);
  if (nb < 0) return nb;
  if ((r = launch_reduce_partials(ctx, w.col_b, nb, ld, G + L.off_b, ld))) return r;

  // 6. K3: scatter dz1 rows into dW (kept items, scaled by s) and dV[u]
  ScatterArgs sc{};
  sc.indptr = m->d.csr_indptr; sc.indices = m->d.csr_indices; sc.values = nullptr; sc.rows = uids;
  sc.keep_off = keep_off; sc.keep = keep_used; sc.row_scale = nullptr; sc.scale = s;
  sc.d = w.dz1; sc.ld = ld; sc.gtable = G + L.off_w;
  sc.growbias = a->skip_user_grad ? nullptr : G + L.off_v;   // data parallel: user rows are exchanged instead
  sc.bias_rows = sharded ? a->v_rows : nullptr;              // item-sharded: only owned users' rows of V
  sc.chunk_off = w.chunk_off;                                // piece map of this batch (built in GRADS_A)
  // plain single-process step: remember which rows of dV get a gradient, the Adam launch reads only those (the rest of
  // dV is zero: it is re-zeroed row by row after every update)
  const bool mask_rows = !sharded && !a->skip_user_grad;
  sc.row_touched = mask_rows ? w.row_touched : nullptr;
  if ((r = launch_scatter(ctx, sc, batch))) return r;
  }  // GRADS_C / GRADS_C2 (data parallel: the caller exchanges dz1 rows and all-reduces dW, db here)

  const int upd = phases & (DRB_PHASE_UPDATE | DRB_PHASE_UPDATE_V | DRB_PHASE_UPDATE_W2T | DRB_PHASE_UPDATE_REST);
  if (!upd) return DRB_OK;
  // 7. K4: fused Adam + L2 over the arena; t per reference variable [W, W_, V, b, b_].  DRB_PHASE_UPDATE = one launch
  //    over everything.  Data parallel: three launches, each as soon as ITS gradient is final -- V after the user rows
  //    have been added, W2T after its all-reduce, the rest (W, b, b2) after theirs -- so the last all-reduce runs under
  //    the V update (72 % of the Adam bytes at the ml-20m shape).
  AdamArgs ad{};
  ad.w = P; ad.m = m->d.adam_m; ad.v = m->d.adam_v; ad.g = G;
  const drb_optim_desc opt = effective_optim(m->opt_set, m->opt, a->beta1, a->beta2, a->epsilon);
  OptimExtra ox;
  optim_fill_args(opt, ad, ox);    // update rule, its hyper-parameters and slots (Adam: beta1 / beta2 / eps only)
  ad.alpha_dev = scal_dev;
  const float c = a->reg_rate / (float)gbatch;                      // cdae.py:82
  const int64_t offs[6] = {L.off_w2t, L.off_w, L.off_b, L.off_b2, L.off_v, L.total};   // arena order
  const int tmap[5] = {1, 0, 3, 4, 2};                                                  // -> [W, W_, V, b, b_]
  const bool l2seg[5] = {true, true, false, false, true};
  const int R = ctx->sm_count * 16;                                  // one reg_part slot
  auto run_adam = [&](int first, int last, int slot, int* n_out) -> int {   // arena segments [first, last]
    int ns = 0;
    for (int sidx = first; sidx <= last; sidx++, ns++) {
      ad.seg[ns].off4 = offs[sidx] / 4;
      ad.seg[ns].n4 = (offs[sidx + 1] - offs[sidx]) / 4;
      ad.seg[ns].alpha = drb_optim_step_size(opt, a->learning_rate, a->t[tmap[sidx]]);
      ad.seg[ns].alpha_idx = tmap[sidx];
      ad.seg[ns].l2 = l2seg[sidx] ? c : 0.f;
      ad.seg[ns].regw = l2seg[sidx] ? 0.5f * c : 0.f;
    }
    ad.nseg = ns;
    ad.row_mask = nullptr; ad.row_seg = -1;
    // segment 4 = V: only the sampled users' rows carry a gradient (data parallel: the rows added from the all-gathered list)
    if (!sharded && (!a->skip_user_grad || m->rows_uids) && first <= 4 && last >= 4) {
      ad.row_mask = w.row_touched; ad.row_seg = 4 - first; ad.row_len4 = ld / 4;
    }
    ad.reg_part = w.reg_part + (int64_t)slot * R;
    return launch_adam(ctx, ad, n_out, ox);
  };
  auto rezero_user_rows = [&]() -> int {      // leave dV all-zero again for the next step (see PREP)
    if (sharded) return DRB_OK;
    if (!a->skip_user_grad) {
      if ((r = launch_zero_rows(ctx, G + L.off_v, uids, batch, ld, w.row_touched))) return r;
      m->v_grad_clean = true;
    } else if (m->rows_uids) {                // data parallel: the rows every rank added from the all-gathered list
      if ((r = launch_zero_rows(ctx, G + L.off_v, m->rows_uids, m->rows_n, ld, w.row_touched))) return r;
      m->v_grad_clean = true;
    }
    return DRB_OK;
  };
  int n_reg = 0;
  auto fuse_finalize = [&](int n_regs) {      // the last Adam block also writes the loss (one launch less)
    ad.fin_loss_part = w.loss_part; ad.fin_n_loss = m->n_loss_blocks; ad.fin_scale = inv_count; ad.fin_n_reg = n_regs;
    ad.fin_reg_part = w.reg_part; ad.fin_loss_out = loss_out;
    ad.fin_ticket = reinterpret_cast<unsigned int*>(w.loss_scalar + 48);
  };
  if (phases & DRB_PHASE_UPDATE) {
    fuse_finalize(0);
    if ((r = run_adam(0, 4, 0, &n_reg))) return r;
    return rezero_user_rows();
  }
  if (!m->reg_slots_clear) {   // split form: unused entries of the three partial-sum slots must read as zero
    DRB_CUDA_TRY(ctx, cudaMemsetAsync(w.reg_part, 0, (size_t)3 * R * sizeof(float), ctx->stream));
    m->reg_slots_clear = true;
  }
  if (phases & DRB_PHASE_UPDATE_V) {
    if ((r = run_adam(4, 4, 0, &n_reg))) return r;
    if ((r = rezero_user_rows())) return r;
  }
  if (phases & DRB_PHASE_UPDATE_W2T) {
    if ((r = run_adam(0, 0, 1, &n_reg))) return r;
  }
  if (phases & DRB_PHASE_UPDATE_REST) {
    fuse_finalize(3 * R);
    if ((r = run_adam(1, 3, 2, &n_reg))) return r;
  }
  return DRB_OK;
}

extern "C" {

int drb_cdae_step_phases(drb_cdae* m, const int32_t* uids, const int32_t* keep_off, const uint8_t* keep,
                         int32_t batch, const drb_cdae_step_args* a, float* loss_out, int32_t phases) {
  if (!m || !uids || !keep_off || !a || !loss_out) return drb_fail(DRB_E_INVALID, "drb_cdae_step: NULL argument");
  drb_ctx* ctx = m->ctx;
  // Graph replay: only the plain single-process step of a launch-bound shape, in steady state (dV known clean, so the
  // captured step is the sparse-clear variant), with inputs that can be staged in the model's own buffers.
  const bool own_inputs = uids == m->ws.uids && keep_off == m->ws.keep_off && (!keep || keep == m->ws.keep);
  const bool small = (int64_t)batch * m->d.n_items <= ((int64_t)8 << 20);
  const bool eligible = !m->graphs.off && !ctx->profile && small && phases == DRB_PHASE_ALL && m->v_grad_clean &&
                        a->global_batch == 0 && !a->shard_items && !a->skip_user_grad && !m->z_dbg &&
                        batch > 0 && batch <= m->d.max_batch && m->d.adam_m && !ctx->sticky &&
                        (own_inputs || !keep || a->keep_bytes > 0);
  if (!eligible) return cdae_step_impl(m, uids, keep_off, keep, batch, a, loss_out, phases, nullptr);
  CdaeWs& w = m->ws;
  if (!own_inputs) {      // stage the caller's device arrays (outside the graph)
    if (keep && a->keep_bytes > m->keep_cap)
      return drb_fail(DRB_E_INVALID, "drb_cdae_step: keep_bytes %lld exceeds the staging capacity", (long long)a->keep_bytes);
    DRB_CUDA_TRY(ctx, cudaMemcpyAsync(w.uids, uids, (size_t)batch * 4, cudaMemcpyDeviceToDevice, ctx->stream));
    DRB_CUDA_TRY(ctx, cudaMemcpyAsync(w.keep_off, keep_off, (size_t)(batch + 1) * 4, cudaMemcpyDeviceToDevice, ctx->stream));
    if (keep)
      DRB_CUDA_TRY(ctx, cudaMemcpyAsync(w.keep, keep, (size_t)a->keep_bytes, cudaMemcpyDeviceToDevice, ctx->stream));
  }
  const uint8_t* gkeep = keep ? w.keep : nullptr;
  float* scal = w.loss_scalar + 8;      // [8..14]: five step sizes + philox step (lo, hi)
  const StepGraphKey key{loss_out, batch, 0, 0, keep ? 1 : 0, a->beta1, a->beta2, a->epsilon, a->reg_rate, a->philox_seed};
  const StepGraphs::Entry* g = m->graphs.get(ctx, key, [&] {
    const bool clean_before = m->v_grad_clean;
    int r = cdae_step_impl(m, w.uids, w.keep_off, gkeep, batch, a, loss_out, phases, scal);
    m->v_grad_clean = clean_before;      // nothing ran during capture
    return r;
  });
  if (!g) return cdae_step_impl(m, w.uids, w.keep_off, gkeep, batch, a, loss_out, phases, nullptr);
  float vals[7];
  const drb_optim_desc opt = effective_optim(m->opt_set, m->opt, a->beta1, a->beta2, a->epsilon);
  for (int j = 0; j < 5; j++) vals[j] = drb_optim_step_size(opt, a->learning_rate, a->t[j]);
  const uint32_t slo = (uint32_t)a->philox_step, shi = (uint32_t)(a->philox_step >> 32);
  std::memcpy(&vals[5], &slo, 4);
  std::memcpy(&vals[6], &shi, 4);
  int r = m->graphs.replay(ctx, g, scal, vals, 7);
  if (r) return r;
  m->v_grad_clean = true;      // the captured step ends with the sparse re-zero of the sampled users' rows
  m->rows_uids = nullptr; m->rows_n = 0;
  return DRB_OK;
}

int drb_cdae_step_host(drb_cdae* m, const int32_t* uids, const int32_t* keep_off, const uint8_t* keep,
                       int32_t batch, const drb_cdae_step_args* a, float* loss_host) {
  if (!m || !uids || !keep_off) return drb_fail(DRB_E_INVALID, "drb_cdae_step_host: NULL argument");
  if (batch <= 0 || batch > m->d.max_batch)
    return drb_fail(DRB_E_INVALID, "drb_cdae_step_host: batch %d outside (0, max_batch=%d]", batch, m->d.max_batch);
  drb_ctx* ctx = m->ctx;
  CdaeWs& w = m->ws;
  const int64_t nnz = keep_off[batch];
  if (nnz > m->keep_cap) return drb_fail(DRB_E_INVALID, "drb_cdae_step_host: batch nnz %lld exceeds staging capacity", (long long)nnz);
  DRB_CUDA_TRY(ctx, cudaMemcpyAsync(w.uids, uids, (size_t)batch * 4, cudaMemcpyHostToDevice, ctx->stream));
  DRB_CUDA_TRY(ctx, cudaMemcpyAsync(w.keep_off, keep_off, (size_t)(batch + 1) * 4, cudaMemcpyHostToDevice, ctx->stream));
  if (keep && nnz > 0)
    DRB_CUDA_TRY(ctx, cudaMemcpyAsync(w.keep, keep, (size_t)nnz, cudaMemcpyHostToDevice, ctx->stream));
  int r = drb_cdae_step(m, w.uids, w.keep_off, keep ? w.keep : nullptr, batch, a, w.loss_scalar);
  if (r) return r;
  if (loss_host) {
    DRB_CUDA_TRY(ctx, cudaMemcpyAsync(loss_host, w.loss_scalar, 4, cudaMemcpyDeviceToHost, ctx->stream));
    DRB_CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
  }
  return DRB_OK;
}

int drb_cdae_hidden(drb_cdae* m, const int32_t* uids, int32_t n, float* h_out) {
  if (!m || !uids || !h_out || n < 0) return drb_fail(DRB_E_INVALID, "drb_cdae_hidden: bad argument");
  // prediction path: plain 0/1 input, no corruption, no 1/(1-q) scaling (cdae.py:67-71)
  return cdae_hidden_into(m, uids, n, nullptr, nullptr, 1.0f, h_out);
}

static int cdae_scores_chunk(drb_cdae* m, const int32_t* uids, int n, float* out) {
  int r = cdae_hidden_into(m, uids, n, nullptr, nullptr, 1.0f, m->ws.h);
  if (r) return r;
  GemmArgs g{};
  g.A = m->ws.h; g.lda = m->L.ld; g.B = m->d.params + m->L.off_w2t; g.ldb = m->L.ld; g.C = out;
  g.ldc = m->L.items_pad; g.M = n; g.N = m->d.n_items; g.Kred = m->L.ld; g.splits = 1;
  g.bias = m->d.params + m->L.off_b2; g.act = DRB_ACT_SIGMOID;
  return launch_gemm(m->ctx, LAYOUT_KK, EPI_BIAS_ACT, g);
}

int drb_cdae_predict_all(drb_cdae* m, const int32_t* uids, int32_t n, float* out) {
  if (!m || !uids || !out || n < 0) return drb_fail(DRB_E_INVALID, "drb_cdae_predict_all: bad argument");
  for (int32_t o = 0; o < n; o += m->d.max_batch) {
    const int c = std::min(m->d.max_batch, n - o);
    int r = cdae_scores_chunk(m, uids + o, c, out + (int64_t)o * m->L.items_pad);
    if (r) return r;
  }
  return DRB_OK;
}

int drb_cdae_predict_pairs(drb_cdae* m, const int32_t* users, int32_t n_users, const int64_t* pair_off,
                           const int32_t* pair_iid, const int32_t* pair_dst, int32_t n, float* out) {
  if (!m || (n > 0 && !out)) return drb_fail(DRB_E_INVALID, "drb_cdae_predict_pairs: NULL argument");
  const PairArgs p{users, n_users, pair_off, pair_iid, pair_dst, n};
  if (n_users == 0 && n == 0) return DRB_OK;
  int r = pair_args_check(m->ctx, "drb_cdae_predict_pairs", p, m->d.n_users, m->d.n_items,
                          reinterpret_cast<int*>(m->ws.dz));
  if (r) return r;
  for (int32_t o = 0; o < n_users; o += m->d.max_batch) {
    const int c = std::min(m->d.max_batch, n_users - o);
    // h exactly as cdae_scores_chunk forms it for drb_cdae_predict_all
    if ((r = cdae_hidden_into(m, users + o, c, nullptr, nullptr, 1.0f, m->ws.h))) return r;
    if ((r = launch_cdae_pair_scores(m->ctx, p, o, c, m->ws.h, m->d.params + m->L.off_w2t, m->d.params + m->L.off_b2,
                                     m->L.ld, out)))
      return r;
  }
  return DRB_OK;
}

int drb_cdae_rank_candidates(drb_cdae* m, const int32_t* uids, int32_t n, const int32_t* cand,
                             const int32_t* cand_count, int32_t max_cand, int32_t novelty, int32_t* out_iid,
                             float* out_score, int32_t* n_out) {
  if (!m || !uids || !cand || !cand_count || !out_iid || !out_score || !n_out || n < 0 || max_cand < 1)
    return drb_fail(DRB_E_INVALID, "drb_cdae_rank_candidates: bad argument");
  // lists longer than the shared-memory sorter takes (recommend(n=None): the whole catalog) sort their keys in the
  // dz workspace, as many users per launch as fit there
  void* scratch = m->ws.dz;
  const int64_t scratch_bytes = m->d.output_mode == DRB_OUTPUT_SAMPLED ? 256 : (int64_t)m->d.max_batch * m->L.items_pad * 4;
  int64_t per = m->d.max_batch;
  if (max_cand > 4096) {
    per = std::min<int64_t>(per, rank_scratch_rows(scratch_bytes, max_cand));
    if (per < 1) return drb_fail(DRB_E_INVALID, "drb_cdae_rank_candidates: max_cand %d does not fit the workspace", max_cand);
  }
  for (int32_t o = 0; o < n; o += (int32_t)per) {
    const int c = (int)std::min<int64_t>(per, n - o);
    int r = cdae_hidden_into(m, uids + o, c, nullptr, nullptr, 1.0f, m->ws.h);
    if (r) return r;
    CandScoreArgs a{};
    a.urep = m->ws.h; a.ld_u = m->L.ld; a.table = m->d.params + m->L.off_w2t; a.ld_t = m->L.ld;
    a.bias = m->d.params + m->L.off_b2; a.width = m->d.hidden; a.mode = 0;
    a.uids = uids + o; a.cand = cand + (int64_t)o * max_cand; a.cand_count = cand_count + o; a.max_cand = max_cand;
    a.seen_indptr = m->d.seen_indptr; a.seen_indices = m->d.seen_indices; a.novelty = novelty;
    a.out_iid = out_iid + (int64_t)o * max_cand; a.out_score = out_score + (int64_t)o * max_cand; a.n_out = n_out + o;
    if ((r = launch_rank_candidates(m->ctx, a, c, scratch, scratch_bytes))) return r;
  }
  return DRB_OK;
}

// Scratch of the tensor-core top-k, carved from the dz workspace (max_batch x items_pad floats):
//   lists [B][cap] u64 | seen bitmap [B][words] u32 | cnt [B] | tau [B] | tau_z [B] | fallback: count, users [FB],
//   rows [FB][items_pad]
struct TopkScratch {
  uint64_t* lists; uint32_t* bits; int32_t* cnt; uint32_t* tau; float* tau_z; int32_t* fb_count; int32_t* fb_users;
  int32_t* big_users;                // users whose list is longer than the first select launch takes (score.cu)
  float* fb_rows;
  int cap, fb_max; bool ok;
  int n_stages; int bounds[12];      // item ranges [bounds[i-1], bounds[i]) of the filter passes (bounds[-1] = 0)
};
static constexpr int kTopkFallbackRows = 32;

static TopkScratch topk_scratch(drb_cdae* m, int cap) {
  TopkScratch t{};
  const int64_t B = m->d.max_batch, words = m->words_per_row;
  Carver c(m->ws.dz);
  t.lists = c.take<uint64_t>(B * cap);
  t.bits = c.take<uint32_t>(B * words);
  t.cnt = c.take<int32_t>(B);
  t.tau = c.take<uint32_t>(B);
  t.tau_z = c.take<float>(B);
  t.fb_count = c.take<int32_t>(64);
  t.fb_users = c.take<int32_t>(kTopkFallbackRows);
  t.big_users = c.take<int32_t>(B);
  t.fb_rows = c.take<float>((int64_t)kTopkFallbackRows * m->L.items_pad);
  t.cap = cap; t.fb_max = kTopkFallbackRows;
  t.ok = c.off <= B * (int64_t)m->L.items_pad * 4;
  return t;
}

// Full-catalog top-k on the tensor cores for one block of users (see umma_score.cu for the selection scheme).
static int cdae_topk_umma_chunk(drb_cdae* m, const TopkScratch& S, const int32_t* uids, int c, int k, int novelty,
                                int32_t* out_iid, float* out_score, int32_t* n_out) {
  drb_ctx* ctx = m->ctx;
  CdaeWs& w = m->ws;
  const int I = m->d.n_items, ld = m->L.ld, words = m->words_per_row;
  int r;
  if ((r = cdae_hidden_into(m, uids, c, nullptr, nullptr, 1.0f, w.h))) return r;
  if (m->half) {
    if ((r = launch_split_f16(ctx, w.h, c, ld, ld, DRB_H_F16_SCALE, nullptr, w.h_hi, w.h_lo, m->ldh, nullptr, nullptr, 0, -1)))
      return r;
  } else if ((r = launch_split_tf32(ctx, w.h, c, ld, ld, w.h_hi, w.h_lo, nullptr, nullptr, 0, -1))) return r;
  DRB_CUDA_TRY(ctx, cudaMemsetAsync(S.cnt, 0, (size_t)c * 4, ctx->stream));
  DRB_CUDA_TRY(ctx, cudaMemsetAsync(S.tau, 0, (size_t)c * 4, ctx->stream));
  DRB_CUDA_TRY(ctx, cudaMemsetAsync(S.fb_count, 0, 64 * 4, ctx->stream));   // [0] fallback rows, [16 + stage] long lists
  const uint32_t* bits = nullptr;
  if (novelty) {     // the user's stored items as a bitmap (cdae.py:93-98): built like the per-user label bitmap
    DRB_CUDA_TRY(ctx, cudaMemsetAsync(S.bits, 0, (size_t)c * words * 4, ctx->stream));
    BatchPrepArgs bp{};
    bp.indptr = m->d.seen_indptr; bp.indices = m->d.seen_indices; bp.rows = uids;
    bp.label_bits = S.bits; bp.words_per_row = words;
    if ((r = launch_batch_prep(ctx, bp, c))) return r;
    bits = S.bits;
  }
  UmmaOperands o{w.h_hi, w.h_lo, m->half ? m->ldh : ld, w.w2t_hi, w.w2t_lo, m->half ? m->ldh : ld, I};
  if (m->half) { o.half = true; o.out_scale = 1.0f / DRB_H_F16_SCALE; o.out_scale_dev = w.loss_scalar + 33; }
  const float* b2 = m->d.params + m->L.off_b2;
  // Stage 0: the first slice, every unseen item is listed; tau = the k-th best of the slice.  Every further stage
  // lists only what reaches the current tau (a logit pre-filter decides for most elements, umma_score.cu) and the
  // select that follows tightens tau to the k-th best of everything seen so far: with item ranges growing
  // geometrically each stage adds about (growth - 1) * k keys per user.  The last select emits the ranked lists.
  for (int st = 0, lo = 0; st < S.n_stages; lo = S.bounds[st], st++) {
    const bool last = st == S.n_stages - 1;
    if ((r = launch_umma_score_filter(ctx, o, c, I, lo, S.bounds[st], ld, b2, bits, words, S.tau, st ? S.tau_z : nullptr,
                                      S.cnt, S.lists, S.cap)))
      return r;
    if ((r = launch_select_lists(ctx, S.lists, S.cap, S.cnt, S.tau, S.tau_z, k, last, last ? out_iid : nullptr,
                                 last ? out_score : nullptr, last ? n_out : nullptr, S.fb_users, S.fb_count, S.fb_max,
                                 S.big_users, S.fb_count + 16 + st, c)))
      return r;
  }
  // users whose list overflowed (n_out == -1, scratch rows claimed by the last select): exact fp32 scores + radix
  // select, on the device, no host round trip
  TopkArgs t{};
  t.ld = m->L.items_pad; t.n_items = I; t.uids = uids;
  t.seen_indptr = m->d.seen_indptr; t.seen_indices = m->d.seen_indices; t.novelty = novelty; t.k = k;
  t.out_iid = out_iid; t.out_score = out_score; t.n_out = n_out;
  return launch_topk_fallback(ctx, t, c, w.h, ld, m->d.params + m->L.off_w2t, ld, b2, m->d.hidden, S.fb_rows, S.fb_users,
                              S.fb_count, S.fb_max);
}

static int cdae_topk_impl(drb_cdae* m, const int32_t* uids, int32_t n, int32_t k, int32_t novelty, int32_t* out_iid,
                          float* out_score, int32_t* n_out, bool exact_only) {
  if (!m || !uids || !out_iid || !out_score || !n_out || n < 0)
    return drb_fail(DRB_E_INVALID, "drb_cdae_topk: bad argument");
  if (m->d.output_mode == DRB_OUTPUT_SAMPLED)
    return drb_fail(DRB_E_STATE, "drb_cdae_topk: a model created for sampled-output training carries no score workspace");
  if (k < 1 || k > 2048) return drb_fail(DRB_E_INVALID, "drb_cdae_topk: k must be in [1, 2048]");
  // Tensor-core path: wide catalogs, blocks of >= 128 users.  DRB_TOPK_PATH=ffma forces the exact-fp32 GEMM + radix
  // select path; DRB_TOPK_CAP / DRB_TOPK_NS / DRB_TOPK_GROWTH shrink the list capacity / set the first slice / the growth
  // of the item ranges from stage to stage (tests of the overflow fallback: a huge growth = two passes).
  const char* path_env = getenv("DRB_TOPK_PATH");
  const int cap_env = getenv("DRB_TOPK_CAP") ? atoi(getenv("DRB_TOPK_CAP")) : 0;
  const int ns_env = getenv("DRB_TOPK_NS") ? atoi(getenv("DRB_TOPK_NS")) : 0;
  const int growth = getenv("DRB_TOPK_GROWTH") ? std::max(2, atoi(getenv("DRB_TOPK_GROWTH"))) : 3;
  const int I = m->d.n_items;
  const int cap = cap_env ? cap_env : 4096;
  // first slice: at least 4 k items (its k-th best is then a usable threshold); a stage over (growth - 1) times the
  // items seen so far is expected to add (growth - 1) k keys to the k kept ones, three times that must fit the list
  const int n_s = ns_env ? ns_env : (int)drb_round_up(std::max<int64_t>(1024, 4ll * k), 256);
  TopkScratch S{};
  bool fast = !exact_only && m->use_umma && n >= 128 && !(path_env && !strcmp(path_env, "ffma")) && (cap & (cap - 1)) == 0 &&
              n_s + k <= cap && n_s < I;
  if (fast && !ns_env && !cap_env) fast = I >= 8192 && n_s <= I / 3 && (3ll * (growth - 1) + 1) * k <= cap;
  if (fast) { S = topk_scratch(m, cap); fast = S.ok; }
  if (fast) {
    int64_t b = n_s;
    while (true) {
      S.bounds[S.n_stages++] = (int)b;
      if (b >= I) break;
      int64_t nx = drb_round_up(b * growth, 128);
      if (S.n_stages == 11 || nx + nx / 4 >= I) nx = I;     // no short last stage
      b = nx;
    }
  }
  if (fast) {   // hi/lo split of W' once per call (the weights do not change while scoring)
    int r;
    if (m->half) {
      float* scales = m->ws.loss_scalar + 32;
      if ((r = launch_absmax_scale(m->ctx, m->d.params + m->L.off_w2t, I, m->d.hidden, m->L.ld, scales))) return r;
      r = launch_split_f16(m->ctx, m->d.params + m->L.off_w2t, I, m->L.ld, m->L.ld, 1.0f, scales, m->ws.w2t_hi,
                           m->ws.w2t_lo, m->ldh, nullptr, nullptr, 0, -1);
    } else {
      r = launch_split_tf32(m->ctx, m->d.params + m->L.off_w2t, I, m->L.ld, m->L.ld, m->ws.w2t_hi, m->ws.w2t_lo, nullptr,
                            nullptr, 0, -1);
    }
    if (r) return r;
  }
  for (int32_t o = 0; o < n; o += m->d.max_batch) {
    const int c = std::min(m->d.max_batch, n - o);
    int r;
    if (fast && c >= 128) {
      if ((r = cdae_topk_umma_chunk(m, S, uids + o, c, k, novelty, out_iid + (int64_t)o * k,
                                    out_score + (int64_t)o * k, n_out + o)))
        return r;
      continue;
    }
    if ((r = cdae_scores_chunk(m, uids + o, c, m->ws.dz))) return r;
    TopkArgs t{};
    t.scores = m->ws.dz; t.ld = m->L.items_pad; t.n_items = m->d.n_items; t.uids = uids + o;
    t.seen_indptr = m->d.seen_indptr; t.seen_indices = m->d.seen_indices; t.novelty = novelty; t.k = k;
    t.out_iid = out_iid + (int64_t)o * k; t.out_score = out_score + (int64_t)o * k; t.n_out = n_out + o;
    if ((r = launch_topk(m->ctx, t, c))) return r;
  }
  return DRB_OK;
}

int drb_cdae_topk(drb_cdae* m, const int32_t* uids, int32_t n, int32_t k, int32_t novelty, int32_t* out_iid,
                  float* out_score, int32_t* n_out) {
  return cdae_topk_impl(m, uids, n, k, novelty, out_iid, out_score, n_out, false);
}

int drb_cdae_topk_exact(drb_cdae* m, const int32_t* uids, int32_t n, int32_t k, int32_t novelty, int32_t* out_iid,
                        float* out_score, int32_t* n_out) {
  return cdae_topk_impl(m, uids, n, k, novelty, out_iid, out_score, n_out, true);
}

}  // extern "C"

// ========================================================================================== DMF
struct DmfTower {
  int n_layers; int in_dim;
  int width[DRB_DMF_MAX_LAYERS], ld[DRB_DMF_MAX_LAYERS];
  int64_t off_k[DRB_DMF_MAX_LAYERS], off_b[DRB_DMF_MAX_LAYERS];
  const int64_t* indptr; const int32_t* indices; const float* values; const float* row_scale;
  float* act[DRB_DMF_MAX_LAYERS];    // [max_batch, ld_l] post-relu activations
  float* dpre[DRB_DMF_MAX_LAYERS];   // [max_batch, ld_l] gradient w.r.t. pre-activations
};

struct drb_dmf {
  drb_ctx* ctx;
  drb_dmf_desc d;
  drb_dmf_layout_t L;
  DmfTower tw[2];  // 0 = user tower (rows over items), 1 = item tower (rows over users)
  float *col_part, *loss_part, *reg_part, *loss_scalar, *labels, *p_tmp, *item_rep, *user_rep;
  int32_t *uids, *iids;
  void* rank_scratch; int64_t rank_scratch_bytes;   // sort keys of candidate lists longer than 4096 (score.cu)
  bool item_rep_valid;                               // item_rep holds the item tower of the CURRENT weights
  int64_t ws_bytes;
  // the training step replayed from the uids / iids / labels buffers above (a caller's device arrays are copied there
  // first), with the two Adam step sizes -- the only per-step scalars -- at step_scalars
  StepGraphs graphs;
  float* step_scalars;
  drb_optim_desc opt;          // drb_dmf_set_optimizer (opt_set == false: Adam with the step args' hyper-parameters)
  bool opt_set;
};

static int dmf_fill_layout(int32_t n_users, int32_t n_items, const int32_t* uf, int32_t nu, const int32_t* itf,
                           int32_t ni, drb_dmf_layout_t* L) {
  if (!L || !uf || !itf || nu < 1 || ni < 1 || nu > DRB_DMF_MAX_LAYERS || ni > DRB_DMF_MAX_LAYERS)
    return drb_fail(DRB_E_INVALID, "drb_dmf_layout: between 1 and %d layers per tower are supported", DRB_DMF_MAX_LAYERS);
  if (uf[nu - 1] != itf[ni - 1])
    return drb_fail(DRB_E_INVALID, "The last user and item factors dimension must be equal (%d != %d)", uf[nu - 1], itf[ni - 1]);
  std::memset(L, 0, sizeof(*L));
  L->n_layers_user = nu; L->n_layers_item = ni;
  int64_t off = 0;
  for (int t = 0; t < 2; t++) {
    const int32_t* f = t ? itf : uf;
    const int n = t ? ni : nu;
    int64_t in = t ? n_users : n_items;
    for (int l = 0; l < n; l++) {
      if (f[l] <= 0 || f[l] > 512) return drb_fail(DRB_E_INVALID, "drb_dmf_layout: layer widths must be in (0, 512]");
      const int ld = (int)drb_round_up(f[l], 4);
      (t ? L->ld_item : L->ld_user)[l] = ld;
      (t ? L->off_kernel_item : L->off_kernel_user)[l] = off; off += in * ld;
      (t ? L->off_bias_item : L->off_bias_user)[l] = off; off += ld;
      in = f[l];
    }
  }
  L->total = off;
  return DRB_OK;
}

static int64_t dmf_carve(drb_dmf* m, void* base, const drb_dmf_layout_t& L, int n_users, int n_items, int max_batch,
                         int sm_count) {
  Carver c(base);
  const int64_t B = max_batch;
  int maxld = 4;
  for (int t = 0; t < 2; t++) {
    const int n = t ? L.n_layers_item : L.n_layers_user;
    for (int l = 0; l < n; l++) {
      const int ld = (t ? L.ld_item : L.ld_user)[l];
      maxld = std::max(maxld, ld);
      float* a = c.take<float>(B * ld);
      float* dp = c.take<float>(B * ld);
      if (m) { m->tw[t].act[l] = a; m->tw[t].dpre[l] = dp; }
    }
  }
  const int ldl = L.ld_user[L.n_layers_user - 1];
  float* col = c.take<float>((int64_t)colpart_blocks(max_batch) * maxld);
  float* lp = c.take<float>(B);
  float* rp = c.take<float>((int64_t)sm_count * 16);
  float* ls = c.take<float>(64);
  float* lab = c.take<float>(B);
  float* pt = c.take<float>(B);
  float* irep = c.take<float>((int64_t)n_items * ldl);
  float* urep = c.take<float>(B * ldl);
  int32_t* u = c.take<int32_t>(B);
  int32_t* i = c.take<int32_t>(B);
  // key scratch for catalog-long candidate lists: 8 users x next_pow2(n_items) 64-bit keys
  int64_t p2 = 32;
  while (p2 < n_items) p2 <<= 1;
  const int64_t rs_bytes = 8 * p2 * 8;
  void* rs = c.take<uint8_t>(rs_bytes);
  if (m) { m->rank_scratch = rs; m->rank_scratch_bytes = rs_bytes; }
  if (m) {
    m->col_part = col; m->loss_part = lp; m->reg_part = rp; m->loss_scalar = ls; m->labels = lab; m->p_tmp = pt;
    m->item_rep = irep; m->user_rep = urep; m->uids = u; m->iids = i;
    m->step_scalars = ls + 16;   // inside the 64-float scalar block, clear of the loss outputs
  }
  (void)n_users;
  return c.off;
}

// forward of one tower for n rows (n <= max_batch); result in tw.act[last]
static int dmf_tower_fwd(drb_dmf* m, int t, const int32_t* ids, int n) {
  DmfTower& T = m->tw[t];
  float* P = m->d.params;
  GatherArgs g{};
  g.indptr = T.indptr; g.indices = T.indices; g.values = T.values; g.rows = ids;
  g.table = P + T.off_k[0]; g.ld = T.ld[0]; g.bias = P + T.off_b[0];
  g.row_scale = T.row_scale; g.scale = 1.0f; g.act = DRB_ACT_RELU; g.width = T.width[0]; g.out = T.act[0];
  int r = launch_gather(m->ctx, g, n);
  if (r) return r;
  for (int l = 1; l < T.n_layers; l++) {
    GemmArgs a{};
    a.A = T.act[l - 1]; a.lda = T.ld[l - 1]; a.B = P + T.off_k[l]; a.ldb = T.ld[l]; a.C = T.act[l]; a.ldc = T.ld[l];
    a.M = n; a.N = T.width[l]; a.Kred = T.width[l - 1]; a.splits = 1; a.bias = P + T.off_b[l]; a.act = DRB_ACT_RELU;
    if ((r = launch_gemm(m->ctx, LAYOUT_KN, EPI_BIAS_ACT, a))) return r;
  }
  return DRB_OK;
}

static int dmf_tower_bwd(drb_dmf* m, int t, const int32_t* ids, int n) {
  DmfTower& T = m->tw[t];
  float* P = m->d.params;
  float* G = m->d.grads;
  int r;
  for (int l = T.n_layers - 1; l >= 1; l--) {
    GemmArgs gk{};  // dK_l = act_{l-1}^T dpre_l
    gk.A = T.act[l - 1]; gk.lda = T.ld[l - 1]; gk.B = T.dpre[l]; gk.ldb = T.ld[l]; gk.C = G + T.off_k[l];
    gk.ldc = T.ld[l]; gk.M = T.width[l - 1]; gk.N = T.ld[l]; gk.Kred = n; gk.splits = 1;
    if ((r = launch_gemm(m->ctx, LAYOUT_MN, EPI_STORE, gk))) return r;
    int nb = launch_colpart(m->ctx, T.dpre[l], n, T.ld[l], m->col_part);
    if (nb < 0) return nb;
    if ((r = launch_reduce_partials(m->ctx, m->col_part, nb, T.ld[l], G + T.off_b[l], T.ld[l]))) return r;
    GemmArgs gd{};  // dpre_{l-1} = (dpre_l K_l^T) * [act_{l-1} > 0]
    gd.A = T.dpre[l]; gd.lda = T.ld[l]; gd.B = P + T.off_k[l]; gd.ldb = T.ld[l]; gd.C = T.dpre[l - 1];
    gd.ldc = T.ld[l - 1]; gd.M = n; gd.N = T.width[l - 1]; gd.Kred = T.ld[l]; gd.splits = 1; gd.mask = T.act[l - 1];
    if ((r = launch_gemm(m->ctx, LAYOUT_KK, EPI_MASK_POS, gd))) return r;
  }
  int nb = launch_colpart(m->ctx, T.dpre[0], n, T.ld[0], m->col_part);
  if (nb < 0) return nb;
  if ((r = launch_reduce_partials(m->ctx, m->col_part, nb, T.ld[0], G + T.off_b[0], T.ld[0]))) return r;
  ScatterArgs sc{};
  sc.indptr = T.indptr; sc.indices = T.indices; sc.values = T.values; sc.rows = ids;
  sc.row_scale = T.row_scale; sc.scale = 1.0f; sc.d = T.dpre[0]; sc.ld = T.ld[0];
  sc.gtable = G + T.off_k[0]; sc.growbias = nullptr;
  return launch_scatter(m->ctx, sc, n);
}

extern "C" {

int drb_dmf_layout(int32_t n_users, int32_t n_items, const int32_t* user_factors, int32_t n_user_layers,
                   const int32_t* item_factors, int32_t n_item_layers, drb_dmf_layout_t* out) {
  if (n_users <= 0 || n_items <= 0) return drb_fail(DRB_E_INVALID, "drb_dmf_layout: n_users, n_items must be > 0");
  return dmf_fill_layout(n_users, n_items, user_factors, n_user_layers, item_factors, n_item_layers, out);
}

int64_t drb_dmf_workspace_bytes(int32_t n_users, int32_t n_items, const int32_t* user_factors, int32_t n_user_layers,
                                const int32_t* item_factors, int32_t n_item_layers, int32_t max_batch) {
  drb_dmf_layout_t L;
  if (drb_dmf_layout(n_users, n_items, user_factors, n_user_layers, item_factors, n_item_layers, &L) || max_batch <= 0)
    return -1;
  return dmf_carve(nullptr, nullptr, L, n_users, n_items, max_batch, 256);
}

int drb_dmf_create(drb_ctx* ctx, const drb_dmf_desc* d, drb_dmf** out) {
  if (!ctx || !d || !out) return drb_fail(DRB_E_INVALID, "drb_dmf_create: NULL argument");
  drb_dmf_layout_t L;
  int r = drb_dmf_layout(d->n_users, d->n_items, d->user_factors, d->n_layers_user, d->item_factors,
                         d->n_layers_item, &L);
  if (r) return r;
  if (!d->params || !d->csr_indptr || !d->csr_indices || !d->csr_values || !d->csc_indptr || !d->csc_indices ||
      !d->csc_values || !d->workspace || d->max_batch <= 0)
    return drb_fail(DRB_E_INVALID, "drb_dmf_create: params, csr, csc and workspace are required");
  if (((uintptr_t)d->params | (uintptr_t)d->adam_m | (uintptr_t)d->adam_v | (uintptr_t)d->grads |
       (uintptr_t)d->workspace) & 15)
    return drb_fail(DRB_E_INVALID, "drb_dmf_create: arenas and workspace must be 16-byte aligned");
  drb_dmf* m = new (std::nothrow) drb_dmf();
  if (!m) return drb_fail(DRB_E_NOMEM, "out of memory");
  m->ctx = ctx; m->d = *d; m->L = L;
  for (int t = 0; t < 2; t++) {
    DmfTower& T = m->tw[t];
    T.n_layers = t ? L.n_layers_item : L.n_layers_user;
    T.in_dim = t ? d->n_users : d->n_items;
    for (int l = 0; l < T.n_layers; l++) {
      T.width[l] = (t ? d->item_factors : d->user_factors)[l];
      T.ld[l] = (t ? L.ld_item : L.ld_user)[l];
      T.off_k[l] = (t ? L.off_kernel_item : L.off_kernel_user)[l];
      T.off_b[l] = (t ? L.off_bias_item : L.off_bias_user)[l];
    }
    T.indptr = t ? d->csc_indptr : d->csr_indptr;
    T.indices = t ? d->csc_indices : d->csr_indices;
    T.values = t ? d->csc_values : d->csr_values;
    T.row_scale = t ? d->csc_row_scale : d->csr_row_scale;
  }
  m->ws_bytes = dmf_carve(m, d->workspace, L, d->n_users, d->n_items, d->max_batch, ctx->sm_count);
  if (m->ws_bytes > d->workspace_bytes) {
    int64_t need = m->ws_bytes;
    delete m;
    return drb_fail(DRB_E_INVALID, "drb_dmf_create: workspace too small (%lld < %lld bytes)",
                    (long long)d->workspace_bytes, (long long)need);
  }
  if (cudaMemsetAsync(m->loss_scalar, 0, 64 * sizeof(float), ctx->stream) != cudaSuccess) {   // loss, step sizes, ticket
    delete m;
    return drb_fail(DRB_E_CUDA, "drb_dmf_create: workspace clear failed");
  }
  *out = m;
  return DRB_OK;
}
int drb_dmf_set_optimizer(drb_dmf* m, const drb_optim_desc* opt) {
  if (!m) return drb_fail(DRB_E_INVALID, "drb_dmf_set_optimizer: NULL model");
  int r = optim_check(opt, "drb_dmf_set_optimizer");
  if (r) return r;
  m->opt = *opt;
  m->opt_set = true;
  m->graphs.clear();   // captured steps hold the previous rule: never replay them for this one
  return DRB_OK;
}

int drb_dmf_destroy(drb_dmf* m) {
  delete m;
  return DRB_OK;
}

// Both towers have exactly two Dense layers of equal first width that fit the fused kernels: the forward pass of BOTH
// towers is one launch (row gather + first layer, second layer fused in the same CTA) and so are the dense part of
// the backward pass and the scatter into the first-layer kernels: memset + 5 kernels per step instead of 22.
static bool dmf_fused_ok(const drb_dmf* m) {
  const DmfTower& A = m->tw[0];
  const DmfTower& B = m->tw[1];
  return A.n_layers == 2 && B.n_layers == 2 && A.ld[0] == B.ld[0] && dmf_tower_bwd_fits(A.width[0], A.ld[0], A.width[1]) &&
         dmf_tower_bwd_fits(B.width[0], B.ld[0], B.width[1]) && !getenv("DRB_DMF_UNFUSED");
}

static GatherArgs dmf_gather_args(drb_dmf* m, int t, const int32_t* ids, bool fuse_next) {
  DmfTower& T = m->tw[t];
  float* P = m->d.params;
  GatherArgs g{};
  g.indptr = T.indptr; g.indices = T.indices; g.values = T.values; g.rows = ids;
  g.table = P + T.off_k[0]; g.ld = T.ld[0]; g.bias = P + T.off_b[0];
  g.row_scale = T.row_scale; g.scale = 1.0f; g.act = DRB_ACT_RELU; g.width = T.width[0]; g.out = T.act[0];
  if (fuse_next) {
    g.next_k = P + T.off_k[1]; g.next_b = P + T.off_b[1]; g.next_ld = T.ld[1]; g.next_width = T.width[1];
    g.next_act = DRB_ACT_RELU; g.next_out = T.act[1];
  }
  return g;
}

static int dmf_towers_fwd_fused(drb_dmf* m, const int32_t* uids, const int32_t* iids, int n) {
  return launch_gather_pair(m->ctx, dmf_gather_args(m, 0, uids, true), dmf_gather_args(m, 1, iids, true), n);
}

static int dmf_towers_bwd_fused(drb_dmf* m, const int32_t* uids, const int32_t* iids, int n) {
  float* P = m->d.params;
  float* G = m->d.grads;
  DmfTowerBwd tb[2];
  ScatterArgs sc[2];
  for (int t = 0; t < 2; t++) {
    DmfTower& T = m->tw[t];
    tb[t] = DmfTowerBwd{T.act[0], T.dpre[1], P + T.off_k[1], T.dpre[0], G + T.off_k[1], G + T.off_b[1], G + T.off_b[0],
                        T.width[0], T.ld[0], T.width[1], T.ld[1]};
    sc[t] = ScatterArgs{};
    sc[t].indptr = T.indptr; sc[t].indices = T.indices; sc[t].values = T.values; sc[t].rows = t ? iids : uids;
    sc[t].row_scale = T.row_scale; sc[t].scale = 1.0f; sc[t].d = T.dpre[0]; sc[t].ld = T.ld[0];
    sc[t].gtable = G + T.off_k[0];
  }
  int r = launch_dmf_tower_bwd(m->ctx, tb[0], tb[1], n);
  if (r) return r;
  return launch_scatter_pair(m->ctx, sc[0], sc[1], n);
}

enum { DMF_PHASE_GRADS = 1, DMF_PHASE_UPDATE = 2 };

// one training step enqueued on ctx->stream; alpha_dev != NULL: Adam step sizes come from device memory (graph capture).
// phases: GRADS = forward + backward into the gradient arena (data parallel: the caller all-reduces it), UPDATE = Adam
// + loss.  global_batch > 0: the loss mean and its gradient use it instead of `batch`.
static int dmf_step_body(drb_dmf* m, const int32_t* uids, const int32_t* iids, const float* labels, int32_t batch,
                         const drb_dmf_step_args* a, float* loss_out, const float* alpha_dev, int phases = 3,
                         int global_batch = 0) {
  drb_ctx* ctx = m->ctx;
  int r;
  const bool fused = dmf_fused_ok(m);
  if (phases & DMF_PHASE_GRADS) {
  DRB_CUDA_TRY(ctx, cudaMemsetAsync(m->d.grads, 0, (size_t)m->L.total * sizeof(float), ctx->stream));
  if (fused) {
    if ((r = dmf_towers_fwd_fused(m, uids, iids, batch))) return r;
  } else {
    if ((r = dmf_tower_fwd(m, 0, uids, batch))) return r;
    if ((r = dmf_tower_fwd(m, 1, iids, batch))) return r;
  }
  const int lu = m->tw[0].n_layers - 1, li = m->tw[1].n_layers - 1;
  DmfHeadArgs h{};
  h.a = m->tw[0].act[lu]; h.e = m->tw[1].act[li]; h.ld = m->tw[0].ld[lu]; h.width = m->tw[0].width[lu];
  h.labels = labels; h.p_out = nullptr; h.da = m->tw[0].dpre[lu]; h.de = m->tw[1].dpre[li];
  h.loss_part = m->loss_part; h.n = batch; h.n_global = global_batch;
  if ((r = launch_dmf_head(ctx, h))) return r;
  if (fused) {
    if ((r = dmf_towers_bwd_fused(m, uids, iids, batch))) return r;
  } else {
    if ((r = dmf_tower_bwd(m, 0, uids, batch))) return r;
    if ((r = dmf_tower_bwd(m, 1, iids, batch))) return r;
  }
  }
  if (!(phases & DMF_PHASE_UPDATE)) return DRB_OK;
  AdamArgs ad{};
  ad.w = m->d.params; ad.m = m->d.adam_m; ad.v = m->d.adam_v; ad.g = m->d.grads;
  const drb_optim_desc opt = effective_optim(m->opt_set, m->opt, a->beta1, a->beta2, a->epsilon);
  OptimExtra ox;
  optim_fill_args(opt, ad, ox);
  ad.alpha_dev = alpha_dev;
  int ns = 0;
  for (int t = 0; t < 2; t++) {
    const float alpha = drb_optim_step_size(opt, a->learning_rate, a->t[t]);
    DmfTower& T = m->tw[t];
    int64_t in = T.in_dim;
    for (int l = 0; l < T.n_layers; l++) {
      ad.seg[ns].off4 = T.off_k[l] / 4; ad.seg[ns].n4 = in * T.ld[l] / 4; ad.seg[ns].alpha = alpha;
      ad.seg[ns].alpha_idx = t;
      ad.seg[ns].l2 = 2.0f * a->reg_rate; ad.seg[ns].regw = a->reg_rate;       // regularizers.l2: reg * sum(w^2)
      ns++;
      ad.seg[ns].off4 = T.off_b[l] / 4; ad.seg[ns].n4 = T.ld[l] / 4; ad.seg[ns].alpha = alpha;
      ad.seg[ns].alpha_idx = t;
      ad.seg[ns].l2 = 0.f; ad.seg[ns].regw = 0.f;
      ns++;
      in = T.width[l];
    }
  }
  ad.nseg = ns;
  ad.reg_part = m->reg_part;
  // the last Adam block also reduces the per-pair loss terms and the L2 partials into loss_out (one launch less)
  ad.fin_loss_part = m->loss_part; ad.fin_n_loss = batch; ad.fin_scale = 1.0f / (float)(global_batch > 0 ? global_batch : batch);
  ad.fin_n_reg = 0; ad.fin_reg_part = nullptr; ad.fin_loss_out = loss_out;
  ad.fin_ticket = reinterpret_cast<unsigned int*>(m->loss_scalar + 48);
  int n_reg = 0;
  return launch_adam(ctx, ad, &n_reg, ox);
}

int drb_dmf_step(drb_dmf* m, const int32_t* uids, const int32_t* iids, const float* labels, int32_t batch,
                 const drb_dmf_step_args* a, float* loss_out) {
  return drb_dmf_step_phases(m, uids, iids, labels, batch, a, loss_out, DRB_DMF_PHASE_ALL, 0);
}

int drb_dmf_grads_buffer(drb_dmf* m, float** ptr, int64_t* count) {
  if (!m || !ptr || !count) return drb_fail(DRB_E_INVALID, "drb_dmf_grads_buffer: NULL argument");
  *ptr = m->d.grads;
  *count = m->L.total;
  return DRB_OK;
}

int drb_dmf_step_phases(drb_dmf* m, const int32_t* uids, const int32_t* iids, const float* labels, int32_t batch,
                        const drb_dmf_step_args* a, float* loss_out, int32_t phases, int32_t global_batch) {
  if (!m || !uids || !iids || !labels || !a || !loss_out) return drb_fail(DRB_E_INVALID, "drb_dmf_step: NULL argument");
  if (!(phases & DRB_DMF_PHASE_ALL) || global_batch < 0 || (global_batch && global_batch < batch))
    return drb_fail(DRB_E_INVALID, "drb_dmf_step_phases: bad phases / global_batch");
  if (batch <= 0 || batch > m->d.max_batch)
    return drb_fail(DRB_E_INVALID, "drb_dmf_step: batch %d outside (0, max_batch=%d]", batch, m->d.max_batch);
  if (!m->d.adam_m || !m->d.adam_v || !m->d.grads)
    return drb_fail(DRB_E_STATE, "drb_dmf_step: model was created without optimizer arenas");
  drb_ctx* ctx = m->ctx;
  if (ctx->sticky) return drb_fail(DRB_E_CUDA, "context has a sticky CUDA error (%d)", ctx->sticky);
  m->item_rep_valid = false;           // the weights are about to change
  if (m->graphs.off || ctx->profile)    // per-kernel profiling brackets every launch with events: direct launches
    return dmf_step_body(m, uids, iids, labels, batch, a, loss_out, nullptr, phases, global_batch);

  if (uids != m->uids) DRB_CUDA_TRY(ctx, cudaMemcpyAsync(m->uids, uids, (size_t)batch * 4, cudaMemcpyDeviceToDevice, ctx->stream));
  if (iids != m->iids) DRB_CUDA_TRY(ctx, cudaMemcpyAsync(m->iids, iids, (size_t)batch * 4, cudaMemcpyDeviceToDevice, ctx->stream));
  if (labels != m->labels)
    DRB_CUDA_TRY(ctx, cudaMemcpyAsync(m->labels, labels, (size_t)batch * 4, cudaMemcpyDeviceToDevice, ctx->stream));
  const StepGraphKey key{loss_out, batch, phases, global_batch, 0, a->beta1, a->beta2, a->epsilon, a->reg_rate, 0};
  const StepGraphs::Entry* g = m->graphs.get(ctx, key, [&] {
    return dmf_step_body(m, m->uids, m->iids, m->labels, batch, a, loss_out, m->step_scalars, phases, global_batch);
  });
  if (!g) return dmf_step_body(m, m->uids, m->iids, m->labels, batch, a, loss_out, nullptr, phases, global_batch);
  const drb_optim_desc opt = effective_optim(m->opt_set, m->opt, a->beta1, a->beta2, a->epsilon);
  const float alphas[2] = {drb_optim_step_size(opt, a->learning_rate, a->t[0]),
                           drb_optim_step_size(opt, a->learning_rate, a->t[1])};
  return m->graphs.replay(ctx, g, m->step_scalars, alphas, 2);
}

int drb_dmf_loss_buffer(drb_dmf* m, float** ptr) {
  if (!m || !ptr) return drb_fail(DRB_E_INVALID, "drb_dmf_loss_buffer: NULL argument");
  *ptr = m->loss_scalar;
  return DRB_OK;
}

int drb_dmf_step_host(drb_dmf* m, const int32_t* uids, const int32_t* iids, const float* labels, int32_t batch,
                      const drb_dmf_step_args* a, float* loss_host) {
  if (!m || !uids || !iids || !labels) return drb_fail(DRB_E_INVALID, "drb_dmf_step_host: NULL argument");
  if (batch <= 0 || batch > m->d.max_batch)
    return drb_fail(DRB_E_INVALID, "drb_dmf_step_host: batch %d outside (0, max_batch=%d]", batch, m->d.max_batch);
  drb_ctx* ctx = m->ctx;
  DRB_CUDA_TRY(ctx, cudaMemcpyAsync(m->uids, uids, (size_t)batch * 4, cudaMemcpyHostToDevice, ctx->stream));
  DRB_CUDA_TRY(ctx, cudaMemcpyAsync(m->iids, iids, (size_t)batch * 4, cudaMemcpyHostToDevice, ctx->stream));
  DRB_CUDA_TRY(ctx, cudaMemcpyAsync(m->labels, labels, (size_t)batch * 4, cudaMemcpyHostToDevice, ctx->stream));
  int r = drb_dmf_step(m, m->uids, m->iids, m->labels, batch, a, m->loss_scalar);
  if (r) return r;
  if (loss_host) {
    DRB_CUDA_TRY(ctx, cudaMemcpyAsync(loss_host, m->loss_scalar, 4, cudaMemcpyDeviceToHost, ctx->stream));
    DRB_CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
  }
  return DRB_OK;
}

int drb_dmf_forward_pairs(drb_dmf* m, const int32_t* uids, const int32_t* iids, int32_t n, float* p_out) {
  if (!m || !uids || !iids || !p_out || n < 0) return drb_fail(DRB_E_INVALID, "drb_dmf_forward_pairs: bad argument");
  const int lu = m->tw[0].n_layers - 1, li = m->tw[1].n_layers - 1;
  for (int32_t o = 0; o < n; o += m->d.max_batch) {
    const int c = std::min(m->d.max_batch, n - o);
    int r;
    if ((r = dmf_tower_fwd(m, 0, uids + o, c))) return r;
    if ((r = dmf_tower_fwd(m, 1, iids + o, c))) return r;
    DmfHeadArgs h{};
    h.a = m->tw[0].act[lu]; h.e = m->tw[1].act[li]; h.ld = m->tw[0].ld[lu]; h.width = m->tw[0].width[lu];
    h.labels = nullptr; h.p_out = p_out + o; h.n = c;
    if ((r = launch_dmf_head(m->ctx, h))) return r;
  }
  return DRB_OK;
}

}  // extern "C"

// Item tower once for every item of the catalog, chunk by chunk, into m->item_rep; the representations stay valid
// until the next training step or drb_dmf_invalidate_cache (a single-user rank() does not recompute the whole catalog).
static int dmf_refresh_item_rep(drb_dmf* m) {
  if (m->item_rep_valid) return DRB_OK;
  drb_ctx* ctx = m->ctx;
  const int li = m->tw[1].n_layers - 1;
  const int ldl = m->tw[1].ld[li];
  int r;
  for (int32_t o = 0; o < m->d.n_items; o += m->d.max_batch) {
    const int c = std::min(m->d.max_batch, m->d.n_items - o);
    if ((r = launch_iota(ctx, m->iids, c, o))) return r;
    if ((r = dmf_tower_fwd(m, 1, m->iids, c))) return r;
    DRB_CUDA_TRY(ctx, cudaMemcpyAsync(m->item_rep + (int64_t)o * ldl, m->tw[1].act[li], (size_t)c * ldl * 4,
                                      cudaMemcpyDeviceToDevice, ctx->stream));
  }
  m->item_rep_valid = true;
  return DRB_OK;
}

// Plan of a drb_dmf_topk call: list capacity, item ranges of the filter passes (swept from the highest item id down)
// and the scratch layout.  DRB_TOPK_CAP / DRB_TOPK_NS / DRB_TOPK_GROWTH (read per call, as drb_cdae_topk reads them)
// set the list capacity, the first range and the growth of the ranges from pass to pass.
struct DmfTopkPlan {
  int cap, growth, n_s, i_pad, words, w32;
  int n_stages; int lo[12];          // pass s covers items [lo[s], s ? lo[s - 1] : n_items)
  int64_t bytes;
};
static constexpr int kDmfTopkFallbackRows = 32;

struct DmfTopkScratch {
  float* irep_t; float* item_inv; uint64_t* lists; uint32_t* bits; int32_t* cnt; uint32_t* tau; float* tau_z;
  int32_t* fb_count; int32_t* fb_users; int32_t* big_users; float* fb_rows;
};

static int64_t dmf_topk_carve(const drb_dmf* m, const DmfTopkPlan& P, void* base, DmfTopkScratch* s) {
  const int64_t B = m->d.max_batch;
  Carver c(base);
  DmfTopkScratch t{};
  t.irep_t = c.take<float>((int64_t)P.w32 * P.i_pad);
  t.item_inv = c.take<float>(P.i_pad);
  t.lists = c.take<uint64_t>(B * P.cap);
  t.bits = c.take<uint32_t>(B * P.words);
  t.cnt = c.take<int32_t>(B);
  t.tau = c.take<uint32_t>(B);
  t.tau_z = c.take<float>(B);
  t.fb_count = c.take<int32_t>(64);        // [0] claimed fallback rows, [16 + pass] long lists of that pass's select
  t.fb_users = c.take<int32_t>(kDmfTopkFallbackRows);
  t.big_users = c.take<int32_t>(B);
  t.fb_rows = c.take<float>((int64_t)kDmfTopkFallbackRows * P.i_pad);
  if (s) *s = t;
  return c.off;
}

static int dmf_topk_plan(const drb_dmf* m, int k, DmfTopkPlan* P) {
  if (k < 1 || k > 2048) return drb_fail(DRB_E_INVALID, "drb_dmf_topk: k must be in [1, 2048] (got %d)", k);
  const int cap_env = getenv("DRB_TOPK_CAP") ? atoi(getenv("DRB_TOPK_CAP")) : 0;
  const int ns_env = getenv("DRB_TOPK_NS") ? atoi(getenv("DRB_TOPK_NS")) : 0;
  const int g_env = getenv("DRB_TOPK_GROWTH") ? atoi(getenv("DRB_TOPK_GROWTH")) : 0;
  const int I = m->d.n_items;
  // a pass over (growth - 1) times the items seen so far adds about (growth - 1) k keys to the >= k kept ones; room
  // for three times that (the capacity follows k up to the 8192 keys the select kernels take)
  int cap = 2048;
  while (cap < 8 * k && cap < 8192) cap <<= 1;
  if (cap_env) cap = cap_env;
  if (cap < 32 || cap > 8192 || (cap & (cap - 1)))
    return drb_fail(DRB_E_INVALID, "drb_dmf_topk: DRB_TOPK_CAP must be a power of two in [32, 8192] (got %d)", cap);
  P->cap = cap;
  P->growth = g_env ? std::max(2, g_env) : ((3ll * 2 + 1) * k <= cap ? 3 : 2);
  // first range: at least 4 k items (its k-th best is then a usable threshold), at most half the list
  P->n_s = ns_env > 0 ? ns_env : (int)std::min<int64_t>(drb_round_up(std::max(1024, 4 * k), 128), cap / 2);
  P->i_pad = (int)drb_round_up(I, 128);
  P->words = P->i_pad / 32;
  P->w32 = 32 * dmf_topk_nj(m->tw[0].width[m->tw[0].n_layers - 1]);
  P->n_stages = 0;
  int64_t b = P->n_s;
  while (true) {                                   // b = items covered from the top after this pass
    const int lo = b >= I ? 0 : (int)((I - b) / 128 * 128);
    P->lo[P->n_stages++] = lo;
    if (lo == 0) break;
    int64_t nx = drb_round_up((int64_t)(I - lo) * P->growth, 128);
    if (P->n_stages == 11 || nx + nx / 4 >= I) nx = I;     // no short last pass
    b = nx;
  }
  P->bytes = dmf_topk_carve(m, *P, nullptr, nullptr);
  return DRB_OK;
}

extern "C" {

int64_t drb_dmf_topk_scratch_bytes(drb_dmf* m, int32_t k) {
  if (!m) return drb_fail(DRB_E_INVALID, "drb_dmf_topk_scratch_bytes: NULL model"), -1;
  DmfTopkPlan P;
  if (dmf_topk_plan(m, k, &P)) return -1;
  return P.bytes;
}

int drb_dmf_topk(drb_dmf* m, const int32_t* uids, int32_t n, int32_t k, int32_t novelty, void* scratch,
                 int64_t scratch_bytes, int32_t* out_iid, float* out_score, int32_t* n_out) {
  if (!m || !uids || !out_iid || !out_score || !n_out || !scratch || n < 0)
    return drb_fail(DRB_E_INVALID, "drb_dmf_topk: bad argument");
  DmfTopkPlan P;
  int r;
  if ((r = dmf_topk_plan(m, k, &P))) return r;
  if (scratch_bytes < P.bytes)
    return drb_fail(DRB_E_INVALID, "drb_dmf_topk: scratch of %lld bytes, k = %d needs %lld (drb_dmf_topk_scratch_bytes)",
                    (long long)scratch_bytes, k, (long long)P.bytes);
  if (n == 0) return DRB_OK;
  drb_ctx* ctx = m->ctx;
  DmfTopkScratch S;
  dmf_topk_carve(m, P, scratch, &S);
  const int lu = m->tw[0].n_layers - 1, li = m->tw[1].n_layers - 1;
  const int I = m->d.n_items, width = m->tw[0].width[lu], ldl = m->tw[1].ld[li];
  if ((r = dmf_refresh_item_rep(m))) return r;
  if ((r = launch_dmf_topk_prep(ctx, m->item_rep, ldl, width, I, P.i_pad, S.irep_t, S.item_inv))) return r;
  for (int32_t o = 0; o < n; o += m->d.max_batch) {
    const int c = std::min(m->d.max_batch, n - o);
    if ((r = dmf_tower_fwd(m, 0, uids + o, c))) return r;
    int32_t* b_iid = out_iid + (int64_t)o * k;
    float* b_score = out_score + (int64_t)o * k;
    DRB_CUDA_TRY(ctx, cudaMemsetAsync(S.cnt, 0, (size_t)c * 4, ctx->stream));
    DRB_CUDA_TRY(ctx, cudaMemsetAsync(S.tau, 0, (size_t)c * 4, ctx->stream));
    DRB_CUDA_TRY(ctx, cudaMemsetAsync(S.fb_count, 0, 64 * 4, ctx->stream));
    const uint32_t* bits = nullptr;
    if (novelty) {     // the user's stored items (the rank path's `seen` rows) as a bitmap
      DRB_CUDA_TRY(ctx, cudaMemsetAsync(S.bits, 0, (size_t)c * P.words * 4, ctx->stream));
      BatchPrepArgs bp{};
      bp.indptr = m->d.csr_indptr; bp.indices = m->d.csr_indices; bp.rows = uids + o;
      bp.label_bits = S.bits; bp.words_per_row = P.words;
      if ((r = launch_batch_prep(ctx, bp, c))) return r;
      bits = S.bits;
    }
    DmfFilterArgs fa{};
    fa.urep = m->tw[0].act[lu]; fa.ld_u = m->tw[0].ld[lu]; fa.n_users = c;
    fa.irep_t = S.irep_t; fa.item_inv = S.item_inv; fa.i_pad = P.i_pad; fa.width = width;
    fa.seen_bits = bits; fa.words_per_row = P.words; fa.tau_ord = S.tau;
    fa.cnt = S.cnt; fa.lists = S.lists; fa.cap = P.cap;
    for (int st = 0; st < P.n_stages; st++) {
      const bool last = st == P.n_stages - 1;
      fa.item_lo = P.lo[st]; fa.item_hi = st ? P.lo[st - 1] : I;
      if ((r = launch_dmf_topk_filter(ctx, fa))) return r;
      if ((r = launch_select_lists(ctx, S.lists, P.cap, S.cnt, S.tau, S.tau_z, k, last, last ? b_iid : nullptr,
                                   last ? b_score : nullptr, last ? n_out + o : nullptr, S.fb_users, S.fb_count,
                                   kDmfTopkFallbackRows, S.big_users, S.fb_count + 16 + st, c)))
        return r;
    }
    // users whose list overflowed claimed fallback rows in the last select; almost always none, so one small read
    // back per block decides whether the exact fallback is launched at all
    int32_t claimed = 0;
    DRB_CUDA_TRY(ctx, cudaMemcpyAsync(&claimed, S.fb_count, 4, cudaMemcpyDeviceToHost, ctx->stream));
    DRB_CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    if (claimed == 0) continue;
    TopkArgs t{};
    t.ld = P.i_pad; t.n_items = I; t.uids = uids + o;
    t.seen_indptr = m->d.csr_indptr; t.seen_indices = m->d.csr_indices; t.novelty = novelty; t.k = k;
    t.out_iid = b_iid; t.out_score = b_score; t.n_out = n_out + o;
    if ((r = launch_dmf_topk_fallback(ctx, t, c, m->tw[0].act[lu], m->tw[0].ld[lu], m->item_rep, ldl, width, S.fb_rows,
                                      S.fb_users, S.fb_count, kDmfTopkFallbackRows)))
      return r;
  }
  return DRB_OK;
}

int drb_dmf_predict_pairs(drb_dmf* m, const int32_t* users, int32_t n_users, const int64_t* pair_off,
                          const int32_t* pair_iid, const int32_t* pair_dst, int32_t n, float* p_out) {
  if (!m || (n > 0 && !p_out)) return drb_fail(DRB_E_INVALID, "drb_dmf_predict_pairs: NULL argument");
  const PairArgs p{users, n_users, pair_off, pair_iid, pair_dst, n};
  if (n_users == 0 && n == 0) return DRB_OK;
  int r = pair_args_check(m->ctx, "drb_dmf_predict_pairs", p, m->d.n_users, m->d.n_items,
                          reinterpret_cast<int*>(m->rank_scratch));
  if (r) return r;
  const int lu = m->tw[0].n_layers - 1, li = m->tw[1].n_layers - 1;
  if ((r = dmf_refresh_item_rep(m))) return r;
  for (int32_t o = 0; o < n_users; o += m->d.max_batch) {
    const int c = std::min(m->d.max_batch, n_users - o);
    // a tower row depends on its own id only (one CTA per row in the gather, splits = 1 in the layer GEMMs), so the
    // rows equal those drb_dmf_forward_pairs computes for the same user / item
    if ((r = dmf_tower_fwd(m, 0, users + o, c))) return r;
    if ((r = launch_dmf_pair_head(m->ctx, p, o, c, m->tw[0].act[lu], m->tw[0].ld[lu], m->item_rep, m->tw[1].ld[li],
                                  m->tw[0].width[lu], p_out)))
      return r;
  }
  return DRB_OK;
}

int drb_dmf_rank_candidates(drb_dmf* m, const int32_t* uids, int32_t n, const int32_t* cand,
                            const int32_t* cand_count, int32_t max_cand, int32_t novelty, int32_t* out_iid,
                            float* out_score, int32_t* n_out) {
  if (!m || !uids || !cand || !cand_count || !out_iid || !out_score || !n_out || n < 0 || max_cand < 1)
    return drb_fail(DRB_E_INVALID, "drb_dmf_rank_candidates: bad argument");
  drb_ctx* ctx = m->ctx;
  const int lu = m->tw[0].n_layers - 1, li = m->tw[1].n_layers - 1;
  const int ldl = m->tw[1].ld[li];
  int r;
  if ((r = dmf_refresh_item_rep(m))) return r;
  int64_t per = m->d.max_batch;
  if (max_cand > 4096) {
    per = std::min<int64_t>(per, rank_scratch_rows(m->rank_scratch_bytes, max_cand));
    if (per < 1) return drb_fail(DRB_E_INVALID, "drb_dmf_rank_candidates: max_cand %d exceeds the catalog-sized key scratch", max_cand);
  }
  for (int32_t o = 0; o < n; o += (int32_t)per) {
    const int c = (int)std::min<int64_t>(per, n - o);
    if ((r = dmf_tower_fwd(m, 0, uids + o, c))) return r;
    CandScoreArgs a{};
    a.urep = m->tw[0].act[lu]; a.ld_u = m->tw[0].ld[lu]; a.table = m->item_rep; a.ld_t = ldl; a.bias = nullptr;
    a.width = m->tw[0].width[lu]; a.mode = 1;
    a.uids = uids + o; a.cand = cand + (int64_t)o * max_cand; a.cand_count = cand_count + o; a.max_cand = max_cand;
    a.seen_indptr = m->d.csr_indptr; a.seen_indices = m->d.csr_indices; a.novelty = novelty;
    a.out_iid = out_iid + (int64_t)o * max_cand; a.out_score = out_score + (int64_t)o * max_cand; a.n_out = n_out + o;
    if ((r = launch_rank_candidates(ctx, a, c, m->rank_scratch, m->rank_scratch_bytes))) return r;
  }
  return DRB_OK;
}

int drb_dmf_invalidate_cache(drb_dmf* m) {
  if (!m) return drb_fail(DRB_E_INVALID, "drb_dmf_invalidate_cache: NULL argument");
  m->item_rep_valid = false;
  return DRB_OK;
}

}  // extern "C"

// ========================================================================================== Caser
struct drb_caser {
  drb_ctx* ctx;
  drb_caser_desc d;
  drb_caser_layout_t L;
  CaserArgs base;              // sizes, offsets and device arrays of every launch; per-step fields are set per call
  float *urep, *scores, *loss_part, *reg_part, *loss_scalar, *eye;
  int32_t *ex_user, *ex_items, *flag;
  int n_loss_blocks;
  // the whole step replayed as one graph, with the step size and the philox step at step_scalars
  StepGraphs graphs;
  float* step_scalars;
  drb_optim_desc opt;
  bool opt_set;
};

// users per launch of the rank path: a one-hot user representation of this width carries the exact scores (below)
static constexpr int kCaserRankUsers = 32;

static int caser_fill_layout(int32_t n_users, int32_t n_items, int32_t L, int32_t T, int32_t d, int32_t n_v, int32_t n_h,
                             drb_caser_layout_t* o) {
  if (!o) return drb_fail(DRB_E_INVALID, "drb_caser_layout: NULL argument");
  if (n_users <= 0 || n_items <= 0) return drb_fail(DRB_E_INVALID, "drb_caser_layout: n_users, n_items must be > 0");
  if (L < 1 || L > 16) return drb_fail(DRB_E_INVALID, "Caser: L must be in [1, 16] (got %d)", L);
  if (T < 1 || T > 32) return drb_fail(DRB_E_INVALID, "Caser: T must be in [1, 32] (got %d)", T);
  if (d < 1 || d > 256) return drb_fail(DRB_E_INVALID, "Caser: d must be in [1, 256] (got %d)", d);
  if (n_v < 1 || n_v > 64) return drb_fail(DRB_E_INVALID, "Caser: n_v must be in [1, 64] (got %d)", n_v);
  if (n_h < 1 || n_h > 64) return drb_fail(DRB_E_INVALID, "Caser: n_h must be in [1, 64] (got %d)", n_h);
  std::memset(o, 0, sizeof(*o));
  o->ld_e = (int32_t)drb_round_up(d, 4);
  o->ld_x = (int32_t)drb_round_up(2 * d, 4);
  o->items_pad = (int32_t)drb_round_up(n_items, 4);
  const int64_t F = (int64_t)n_v * d + (int64_t)n_h * L;
  int64_t off = 0;
  auto take = [&](int64_t n) { const int64_t r = off; off += drb_round_up(n, 4); return r; };
  o->off_e = take((int64_t)n_items * o->ld_e);
  o->off_p = take((int64_t)n_users * o->ld_e);
  o->off_w2 = take((int64_t)n_items * o->ld_x);
  o->off_fv = take((int64_t)L * n_v);
  o->off_fh = take((int64_t)n_h * d * L * (L + 1) / 2);
  o->off_fc = take(F * d);
  o->off_bv = take(n_v);
  o->off_bh = take((int64_t)L * n_h);
  o->off_bfc = take(d);
  o->off_b2 = take(n_items);
  o->total = off;
  return DRB_OK;
}

static CaserArgs caser_args(const drb_caser_layout_t& Lo, int n_users, int n_items, int L, int T, int d, int n_v, int n_h,
                            int neg_ratio) {
  CaserArgs a{};
  a.n_users = n_users; a.n_items = n_items; a.L = L; a.T = T; a.d = d; a.n_v = n_v; a.n_h = n_h;
  a.n_tgt = T * (1 + neg_ratio);
  a.F = n_v * d + n_h * L; a.n_fh = n_h * d * L * (L + 1) / 2; a.n_conv = n_h * L * (L + 1) / 2;
  a.lde = Lo.ld_e; a.ldx = Lo.ld_x;
  a.off_e = Lo.off_e; a.off_p = Lo.off_p; a.off_w2 = Lo.off_w2; a.off_fv = Lo.off_fv; a.off_fh = Lo.off_fh;
  a.off_fc = Lo.off_fc; a.off_bv = Lo.off_bv; a.off_bh = Lo.off_bh; a.off_bfc = Lo.off_bfc; a.off_b2 = Lo.off_b2;
  return a;
}

static int64_t caser_carve(drb_caser* m, void* base, const drb_caser_layout_t& Lo, int n_items, int row, int max_batch) {
  Carver c(base);
  const int64_t B = max_batch;
  float* urep = c.take<float>(B * Lo.ld_x);
  float* scores = c.take<float>(B * Lo.items_pad);
  float* lp = c.take<float>(1024);
  float* rp = c.take<float>(256 * 16);
  float* ls = c.take<float>(64);
  float* eye = c.take<float>(kCaserRankUsers * kCaserRankUsers);
  int32_t* eu = c.take<int32_t>(B);
  int32_t* ei = c.take<int32_t>(B * row);
  int32_t* flag = c.take<int32_t>(4);
  if (m) {
    m->urep = urep; m->scores = scores; m->loss_part = lp; m->reg_part = rp; m->loss_scalar = ls; m->eye = eye;
    m->ex_user = eu; m->ex_items = ei; m->flag = flag;
    m->step_scalars = ls + 16;
  }
  (void)n_items;
  return c.off;
}

static int caser_check_sizes(const drb_caser_layout_t& Lo, int L, int T, int d, int n_v, int n_h, int neg_ratio) {
  if (neg_ratio < 0 || neg_ratio > 1000) return drb_fail(DRB_E_INVALID, "Caser: neg_ratio must be in [0, 1000] (got %d)", neg_ratio);
  const CaserArgs a = caser_args(Lo, 1, 1, L, T, d, n_v, n_h, neg_ratio);
  const int64_t smem = caser_smem_bytes(a, true);
  if (smem > kCaserMaxSmem)
    return drb_fail(DRB_E_INVALID, "Caser: L=%d, T=%d, d=%d, n_v=%d, n_h=%d, neg_ratio=%d need %lld bytes of shared memory "
                    "per CTA for the conv / fc weights and their gradients (at most %lld)", L, T, d, n_v, n_h, neg_ratio,
                    (long long)smem, (long long)kCaserMaxSmem);
  return DRB_OK;
}

extern "C" {

int drb_caser_layout(int32_t n_users, int32_t n_items, int32_t L, int32_t T, int32_t d, int32_t n_v, int32_t n_h,
                     drb_caser_layout_t* out) {
  int r = caser_fill_layout(n_users, n_items, L, T, d, n_v, n_h, out);
  if (r) return r;
  return caser_check_sizes(*out, L, T, d, n_v, n_h, 0);
}

int64_t drb_caser_workspace_bytes(int32_t n_users, int32_t n_items, int32_t L, int32_t T, int32_t d, int32_t n_v,
                                  int32_t n_h, int32_t neg_ratio, int32_t max_batch) {
  drb_caser_layout_t Lo;
  if (drb_caser_layout(n_users, n_items, L, T, d, n_v, n_h, &Lo) || max_batch <= 0 || neg_ratio < 0) return -1;
  return caser_carve(nullptr, nullptr, Lo, n_items, L + T * (1 + neg_ratio), max_batch);
}

int drb_caser_create(drb_ctx* ctx, const drb_caser_desc* d, drb_caser** out) {
  if (!ctx || !d || !out) return drb_fail(DRB_E_INVALID, "drb_caser_create: NULL argument");
  drb_caser_layout_t Lo;
  int r = drb_caser_layout(d->n_users, d->n_items, d->L, d->T, d->d, d->n_v, d->n_h, &Lo);
  if (r) return r;
  if ((r = caser_check_sizes(Lo, d->L, d->T, d->d, d->n_v, d->n_h, d->neg_ratio))) return r;
  if (!(d->dropout_rate >= 0.f && d->dropout_rate < 1.f))
    return drb_fail(DRB_E_INVALID, "drb_caser_create: dropout_rate must be in [0, 1)");
  if (!d->params || !d->seq || !d->seq_indptr || !d->win_off || !d->seen_indptr || !d->seen_indices || !d->workspace ||
      d->max_batch <= 0)
    return drb_fail(DRB_E_INVALID, "drb_caser_create: params, sequences, windows, stored rows and workspace are required");
  if (((uintptr_t)d->params | (uintptr_t)d->adam_m | (uintptr_t)d->adam_v | (uintptr_t)d->grads |
       (uintptr_t)d->workspace) & 15)
    return drb_fail(DRB_E_INVALID, "drb_caser_create: arenas and workspace must be 16-byte aligned");
  drb_caser* m = new (std::nothrow) drb_caser();
  if (!m) return drb_fail(DRB_E_NOMEM, "out of memory");
  m->ctx = ctx; m->d = *d; m->L = Lo;
  const int row = d->L + d->T * (1 + d->neg_ratio);
  const int64_t need = caser_carve(m, d->workspace, Lo, d->n_items, row, d->max_batch);
  if (need > d->workspace_bytes) {
    delete m;
    return drb_fail(DRB_E_INVALID, "drb_caser_create: workspace too small (%lld < %lld bytes)",
                    (long long)d->workspace_bytes, (long long)need);
  }
  CaserArgs& a = m->base;
  a = caser_args(Lo, d->n_users, d->n_items, d->L, d->T, d->d, d->n_v, d->n_h, d->neg_ratio);
  a.params = d->params; a.grads = d->grads;
  a.seq = d->seq; a.seq_off = d->seq_indptr; a.win_off = d->win_off; a.n_windows = d->n_windows;
  a.seen_indptr = d->seen_indptr; a.seen_indices = d->seen_indices;
  a.ex_user = m->ex_user; a.ex_items = m->ex_items;
  a.dropout = d->dropout_rate; a.keep_scale = 1.0f / (1.0f - d->dropout_rate);
  a.loss_part = m->loss_part;
  float eye[kCaserRankUsers * kCaserRankUsers] = {};
  for (int i = 0; i < kCaserRankUsers; i++) eye[i * kCaserRankUsers + i] = 1.f;
  if (cudaMemsetAsync(m->loss_scalar, 0, 64 * sizeof(float), ctx->stream) != cudaSuccess ||
      cudaMemcpyAsync(m->eye, eye, sizeof(eye), cudaMemcpyHostToDevice, ctx->stream) != cudaSuccess ||
      cudaStreamSynchronize(ctx->stream) != cudaSuccess) {
    delete m;
    return drb_fail(DRB_E_CUDA, "drb_caser_create: workspace initialisation failed");
  }
  *out = m;
  return DRB_OK;
}

int drb_caser_destroy(drb_caser* m) {
  delete m;
  return DRB_OK;
}

int drb_caser_set_optimizer(drb_caser* m, const drb_optim_desc* opt) {
  if (!m) return drb_fail(DRB_E_INVALID, "drb_caser_set_optimizer: NULL model");
  int r = optim_check(opt, "drb_caser_set_optimizer");
  if (r) return r;
  m->opt = *opt;
  m->opt_set = true;
  m->graphs.clear();
  return DRB_OK;
}

}  // extern "C"

// one step on ctx->stream; scal_dev != NULL: the step size and the philox step come from device memory (graph capture)
static int caser_step_body(drb_caser* m, int32_t batch, const drb_caser_step_args* s, float* loss_out, float* scal_dev) {
  drb_ctx* ctx = m->ctx;
  int r;
  DRB_CUDA_TRY(ctx, cudaMemsetAsync(m->d.grads, 0, (size_t)m->L.total * sizeof(float), ctx->stream));
  CaserArgs a = m->base;
  a.seed = s->philox_seed; a.step = s->philox_step;
  a.step_dev = scal_dev ? reinterpret_cast<const uint32_t*>(scal_dev + 1) : nullptr;
  a.inv_count = 1.0f / (float)((int64_t)batch * a.n_tgt);
  if ((r = launch_caser_sample(ctx, a, batch))) return r;
  int n_blocks = 0;
  if ((r = launch_caser_step(ctx, a, batch, &n_blocks))) return r;
  AdamArgs ad{};
  ad.w = m->d.params; ad.m = m->d.adam_m; ad.v = m->d.adam_v; ad.g = m->d.grads;
  const drb_optim_desc opt = effective_optim(m->opt_set, m->opt, s->beta1, s->beta2, s->epsilon);
  OptimExtra ox;
  optim_fill_args(opt, ad, ox);
  ad.alpha_dev = scal_dev;
  const float alpha = drb_optim_step_size(opt, s->learning_rate, s->t);
  ad.seg[0] = AdamSeg{0, m->L.off_bv / 4, alpha, 2.0f * s->reg_rate, s->reg_rate, 0};   // tensors under L2
  ad.seg[1] = AdamSeg{m->L.off_bv / 4, (m->L.total - m->L.off_bv) / 4, alpha, 0.f, 0.f, 0};
  ad.nseg = 2;
  ad.reg_part = m->reg_part;
  ad.fin_loss_part = m->loss_part; ad.fin_n_loss = n_blocks; ad.fin_scale = a.inv_count;
  ad.fin_n_reg = 0; ad.fin_reg_part = nullptr; ad.fin_loss_out = loss_out;
  ad.fin_ticket = reinterpret_cast<unsigned int*>(m->loss_scalar + 48);
  int n_reg = 0;
  return launch_adam(ctx, ad, &n_reg, ox);
}

extern "C" {

int drb_caser_step(drb_caser* m, int32_t batch, const drb_caser_step_args* s, float* loss_out) {
  if (!m || !s || !loss_out) return drb_fail(DRB_E_INVALID, "drb_caser_step: NULL argument");
  if (batch <= 0 || batch > m->d.max_batch)
    return drb_fail(DRB_E_INVALID, "drb_caser_step: batch %d outside (0, max_batch=%d]", batch, m->d.max_batch);
  if (!m->d.adam_m || !m->d.adam_v || !m->d.grads)
    return drb_fail(DRB_E_STATE, "drb_caser_step: model was created without optimizer arenas");
  if (m->d.n_windows <= 0) return drb_fail(DRB_E_STATE, "drb_caser_step: no user has L + T items");
  drb_ctx* ctx = m->ctx;
  if (ctx->sticky) return drb_fail(DRB_E_CUDA, "context has a sticky CUDA error (%d)", ctx->sticky);
  if (m->graphs.off || ctx->profile) return caser_step_body(m, batch, s, loss_out, nullptr);
  const StepGraphKey key{loss_out, batch, 0, 0, 0, s->beta1, s->beta2, s->epsilon, s->reg_rate, s->philox_seed};
  const StepGraphs::Entry* g = m->graphs.get(ctx, key, [&] { return caser_step_body(m, batch, s, loss_out, m->step_scalars); });
  if (!g) return caser_step_body(m, batch, s, loss_out, nullptr);
  const drb_optim_desc opt = effective_optim(m->opt_set, m->opt, s->beta1, s->beta2, s->epsilon);
  float vals[3];
  vals[0] = drb_optim_step_size(opt, s->learning_rate, s->t);
  const uint32_t slo = (uint32_t)s->philox_step, shi = (uint32_t)(s->philox_step >> 32);
  std::memcpy(&vals[1], &slo, 4);
  std::memcpy(&vals[2], &shi, 4);
  return m->graphs.replay(ctx, g, m->step_scalars, vals, 3);
}

int drb_caser_loss_buffer(drb_caser* m, float** ptr) {
  if (!m || !ptr) return drb_fail(DRB_E_INVALID, "drb_caser_loss_buffer: NULL argument");
  *ptr = m->loss_scalar;
  return DRB_OK;
}

int drb_caser_batch_buffer(drb_caser* m, int32_t** users, int32_t** items, int32_t* row_len) {
  if (!m || !users || !items || !row_len) return drb_fail(DRB_E_INVALID, "drb_caser_batch_buffer: NULL argument");
  *users = m->ex_user; *items = m->ex_items; *row_len = m->base.L + m->base.n_tgt;
  return DRB_OK;
}

int drb_caser_user_rep(drb_caser* m, const int32_t* uids, int32_t n, float* x_out) {
  if (!m || !uids || !x_out || n < 0 || n > m->d.max_batch) return drb_fail(DRB_E_INVALID, "drb_caser_user_rep: bad argument");
  return launch_caser_user_rep(m->ctx, m->base, uids, n, x_out);
}

}  // extern "C"

// sigmoid(x W2^T + b2) for c <= max_batch users into out [c][items_pad]: the fmaf chain every Caser score comes from
static int caser_scores_chunk(drb_caser* m, const int32_t* uids, int c, float* out) {
  int r = launch_caser_user_rep(m->ctx, m->base, uids, c, m->urep);
  if (r) return r;
  GemmArgs g{};
  g.A = m->urep; g.lda = m->L.ld_x; g.B = m->d.params + m->L.off_w2; g.ldb = m->L.ld_x; g.C = out;
  g.ldc = m->L.items_pad; g.M = c; g.N = m->d.n_items; g.Kred = m->L.ld_x; g.splits = 1;
  g.bias = m->d.params + m->L.off_b2; g.act = DRB_ACT_SIGMOID;
  return launch_gemm(m->ctx, LAYOUT_KK, EPI_BIAS_ACT, g);
}

extern "C" {

int drb_caser_predict_all(drb_caser* m, const int32_t* uids, int32_t n, float* out) {
  if (!m || !uids || !out || n < 0) return drb_fail(DRB_E_INVALID, "drb_caser_predict_all: bad argument");
  for (int32_t o = 0; o < n; o += m->d.max_batch) {
    const int c = std::min(m->d.max_batch, n - o);
    int r = caser_scores_chunk(m, uids + o, c, out + (int64_t)o * m->L.items_pad);
    if (r) return r;
  }
  return DRB_OK;
}

int drb_caser_predict_pairs(drb_caser* m, const int32_t* users, int32_t n_users, const int64_t* pair_off,
                            const int32_t* pair_iid, const int32_t* pair_dst, int32_t n, float* out) {
  if (!m || (n > 0 && !out)) return drb_fail(DRB_E_INVALID, "drb_caser_predict_pairs: NULL argument");
  const PairArgs p{users, n_users, pair_off, pair_iid, pair_dst, n};
  if (n_users == 0 && n == 0) return DRB_OK;
  int r = pair_args_check(m->ctx, "drb_caser_predict_pairs", p, m->d.n_users, m->d.n_items, m->flag);
  if (r) return r;
  for (int32_t o = 0; o < n_users; o += m->d.max_batch) {
    const int c = std::min(m->d.max_batch, n_users - o);
    if ((r = launch_caser_user_rep(m->ctx, m->base, users + o, c, m->urep))) return r;
    if ((r = launch_cdae_pair_scores(m->ctx, p, o, c, m->urep, m->d.params + m->L.off_w2, m->d.params + m->L.off_b2,
                                     m->L.ld_x, out)))
      return r;
  }
  return DRB_OK;
}

// The rank path takes its scores from the chain of drb_caser_predict_all: for a block of 32 users the GEMM forms the
// logits x W2^T transposed ([n_items][32], no bias), and k_rank_candidates scores candidate j of user u as the dot
// product of that row with the one-hot vector e_u (1 * logit plus zeros: exactly the logit), plus b2[j], through the
// same sigmoid.  Catalog-long candidate lists sort their keys in the score buffer.
int drb_caser_rank_candidates(drb_caser* m, const int32_t* uids, int32_t n, const int32_t* cand,
                              const int32_t* cand_count, int32_t max_cand, int32_t novelty, int32_t* out_iid,
                              float* out_score, int32_t* n_out) {
  if (!m || !uids || !cand || !cand_count || !out_iid || !out_score || !n_out || n < 0 || max_cand < 1)
    return drb_fail(DRB_E_INVALID, "drb_caser_rank_candidates: bad argument");
  const int U = kCaserRankUsers;
  const int64_t logit_floats = (int64_t)m->d.n_items * U;
  if (m->d.max_batch < U || logit_floats > (int64_t)m->d.max_batch * m->L.items_pad)
    return drb_fail(DRB_E_INVALID, "drb_caser_rank_candidates: max_batch must be >= %d", U);
  float* logits = m->scores;
  void* scratch = m->scores + drb_round_up(logit_floats, 64);
  const int64_t scratch_bytes = ((int64_t)m->d.max_batch * m->L.items_pad - drb_round_up(logit_floats, 64)) * 4;
  int64_t per = U;
  if (max_cand > 4096) {
    per = std::min<int64_t>(per, rank_scratch_rows(scratch_bytes, max_cand));
    if (per < 1) return drb_fail(DRB_E_INVALID, "drb_caser_rank_candidates: max_cand %d does not fit the workspace", max_cand);
  }
  for (int32_t o = 0; o < n; o += U) {
    const int c = std::min(U, n - o);
    int r = launch_caser_user_rep(m->ctx, m->base, uids + o, c, m->urep);
    if (r) return r;
    GemmArgs g{};
    g.A = m->d.params + m->L.off_w2; g.lda = m->L.ld_x; g.B = m->urep; g.ldb = m->L.ld_x; g.C = logits; g.ldc = U;
    g.M = m->d.n_items; g.N = c; g.Kred = m->L.ld_x; g.splits = 1;
    if ((r = launch_gemm(m->ctx, LAYOUT_KK, EPI_STORE, g))) return r;
    for (int q = 0; q < c; q += (int)per) {
      const int cc = std::min<int>((int)per, c - q);
      CandScoreArgs a{};
      a.urep = m->eye + q * U; a.ld_u = U; a.table = logits; a.ld_t = U;
      a.bias = m->d.params + m->L.off_b2; a.width = U; a.mode = 0;
      const int64_t u0 = o + q;
      a.uids = uids + u0; a.cand = cand + u0 * max_cand; a.cand_count = cand_count + u0; a.max_cand = max_cand;
      a.seen_indptr = m->d.seen_indptr; a.seen_indices = m->d.seen_indices; a.novelty = novelty;
      a.out_iid = out_iid + u0 * max_cand; a.out_score = out_score + u0 * max_cand; a.n_out = n_out + u0;
      if ((r = launch_rank_candidates(m->ctx, a, cc, scratch, scratch_bytes))) return r;
    }
  }
  return DRB_OK;
}

int drb_caser_topk(drb_caser* m, const int32_t* uids, int32_t n, int32_t k, int32_t novelty, int32_t* out_iid,
                   float* out_score, int32_t* n_out) {
  if (!m || !uids || !out_iid || !out_score || !n_out || n < 0) return drb_fail(DRB_E_INVALID, "drb_caser_topk: bad argument");
  if (k < 1 || k > 2048) return drb_fail(DRB_E_INVALID, "drb_caser_topk: k must be in [1, 2048]");
  for (int32_t o = 0; o < n; o += m->d.max_batch) {
    const int c = std::min(m->d.max_batch, n - o);
    int r;
    if ((r = caser_scores_chunk(m, uids + o, c, m->scores))) return r;
    TopkArgs t{};
    t.scores = m->scores; t.ld = m->L.items_pad; t.n_items = m->d.n_items; t.uids = uids + o;
    t.seen_indptr = m->d.seen_indptr; t.seen_indices = m->d.seen_indices; t.novelty = novelty; t.k = k;
    t.out_iid = out_iid + (int64_t)o * k; t.out_score = out_score + (int64_t)o * k; t.n_out = n_out + o;
    if ((r = launch_topk(m->ctx, t, c))) return r;
  }
  return DRB_OK;
}

}  // extern "C"
