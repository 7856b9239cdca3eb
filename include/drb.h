/*
 * drb.h -- C ABI of libdrb.so: the B200-native hot path behind DRecPy's CDAE / DMF recommenders.
 *
 * Every entry point replaces a piece of the reference's Python/TensorFlow hot path (cited per function as
 * "replaces <file>:<lines>", paths relative to the DRecPy source tree).  The reference has no FFI of its own
 * (it is pure Python); the binding a maintainer adds is the ctypes stub shown in INTEGRATION.md, which is what
 * drecpy_b200/_lib.py implements.
 *
 * Conventions
 *   - plain C, no C++ types, no exceptions across the boundary;
 *   - every function returns int: 0 = OK, <0 = error (DRB_E_*); the message is in drb_last_error()
 *     (thread-local);
 *   - device buffers are OWNED BY THE CALLER (PyTorch tensors on the Python side).  The library borrows raw
 *     device pointers until the owning object is destroyed; it never allocates or frees device memory;
 *   - there is NO CPU fallback: device entry points fail with DRB_E_NODEVICE without an sm_100 GPU;
 *   - a context is not re-entrant; serialise calls per context.  All device work is enqueued on the context's
 *     stream (drb_ctx_set_stream) and is asynchronous unless documented otherwise.
 */
#ifndef DRB_H
#define DRB_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DRB_VERSION 100 /* 0.1.0 */

enum {
  DRB_OK = 0,
  DRB_E_INVALID = -1,   /* bad argument (range, alignment, NULL) */
  DRB_E_NODEVICE = -2,  /* no CUDA device / not sm_100 */
  DRB_E_CUDA = -3,      /* CUDA runtime error (sticky per context) */
  DRB_E_STATE = -4,     /* object used in the wrong state */
  DRB_E_NOMEM = -5
};

enum { DRB_LOSS_BCE = 0, DRB_LOSS_MSE = 1 };
enum { DRB_LABEL_BATCH_MEAN = 0, DRB_LABEL_PER_USER = 1 };
enum { DRB_ACT_NONE = 0, DRB_ACT_SIGMOID = 1, DRB_ACT_RELU = 2 };
enum { DRB_OUTPUT_DENSE = 0, DRB_OUTPUT_SAMPLED = 1 };
enum { DRB_GEMM_AUTO = 0, DRB_GEMM_FFMA = 1, DRB_GEMM_TCGEN05 = 2, DRB_GEMM_TCGEN05_TF32 = 3 };

typedef struct drb_ctx drb_ctx;
typedef struct drb_rng drb_rng;
typedef struct drb_sampler drb_sampler;
typedef struct drb_cdae drb_cdae;
typedef struct drb_dmf drb_dmf;
typedef struct drb_caser drb_caser;

/* ------------------------------------------------------------------ diagnostics */
int drb_version(void);
const char* drb_last_error(void);

/* ------------------------------------------------------------------ context */
/* Creates a context on CUDA device `device`; fails with DRB_E_NODEVICE if it is not compute capability 10.x. */
int drb_ctx_create(int device, drb_ctx** out);
int drb_ctx_destroy(drb_ctx* ctx);
/* `stream` is a cudaStream_t (e.g. torch.cuda.current_stream().cuda_stream); NULL = legacy default stream. */
int drb_ctx_set_stream(drb_ctx* ctx, void* stream);
int drb_ctx_synchronize(drb_ctx* ctx);
/* number of kernel launches this context has enqueued so far (bench.py's gpu_launches claim) */
int64_t drb_ctx_launch_count(const drb_ctx* ctx);
/* Per-kernel device timing for the roofline report: when enabled, every kernel launch is bracketed by CUDA
 * events on the context's stream.  drb_ctx_profile_read synchronises, aggregates by kernel name and clears the
 * records: names = '\n'-separated list, total_ms[i] / counts[i] per name.  Never enable it inside a timed run. */
int drb_ctx_profile_enable(drb_ctx* ctx, int on);
int drb_ctx_profile_read(drb_ctx* ctx, char* names, int64_t names_cap, double* total_ms, int64_t* counts,
                         int32_t max_entries, int32_t* n_entries);

/* ------------------------------------------------------------------ host RNG: CPython random.Random replay
 * replaces: the three `random.Random(seed)` streams of DRecPy/Sampler/point_sampler.py:30,
 * DRecPy/Dataset/mem_dataset.py:113-114,135-136, the corruption stream DRecPy/Recommender/recommender_abc.py:74
 * and the per-user streams of DRecPy/Evaluation/Processes/ranking_evaluation.py:116.
 * MT19937 with CPython's init_by_array seeding of abs(seed); bit-exact with CPython >= 3.2. */
int drb_rng_create(uint64_t abs_seed, drb_rng** out);
int drb_rng_destroy(drb_rng* rng);
int drb_rng_seed(drb_rng* rng, uint64_t abs_seed);
double drb_rng_random(drb_rng* rng);                    /* random.random() */
uint64_t drb_rng_getrandbits(drb_rng* rng, int k);      /* random.getrandbits(k), 1 <= k <= 64 */
int64_t drb_rng_randbelow(drb_rng* rng, int64_t n);     /* random._randbelow(n), n >= 1 */
int drb_rng_random_fill(drb_rng* rng, int64_t n, double* out);
/* random.sample(range(n), k) (returns indices) and random.shuffle on an index vector (CPython 3.12 algorithms) */
int drb_rng_sample_indices(drb_rng* rng, int64_t n, int64_t k, int64_t* out);
int drb_rng_shuffle_i64(drb_rng* rng, int64_t n, int64_t* x);
/* state[0..623] = mt, state[624] = index (same layout as random.getstate()[1]) */
/* The next 624 untempered output words (generator not advanced) / the inverse; drb_rng_skip discards n outputs. */
int drb_rng_window(const drb_rng* rng, uint32_t window[624]);
int drb_rng_set_window(drb_rng* rng, const uint32_t window[624]);
int drb_rng_skip(drb_rng* rng, int64_t n_outputs);
int drb_rng_getstate(const drb_rng* rng, uint32_t state[625]);
int drb_rng_setstate(drb_rng* rng, const uint32_t state[625]);

/* ------------------------------------------------------------------ PointSampler
 * replaces: DRecPy/Sampler/point_sampler.py:44-96 and the two generators it pulls from,
 * DRecPy/Dataset/mem_dataset.py:119-129 (positives) and :154-163 (null pairs).
 * pos_* : per-user rows with interaction >= threshold (all rows if no threshold), in DataFrame row order;
 * all_* : per-user item ids of ALL rows, sorted ascending (membership test of :161).
 * Host arrays are borrowed until drb_sampler_destroy. */
int drb_sampler_create(int32_t max_uid, int32_t max_iid,
                       const int64_t* pos_indptr, const int32_t* pos_iid, const double* pos_val,
                       const int64_t* all_indptr, const int32_t* all_iid_sorted,
                       double neg_ratio, uint64_t abs_seed, drb_sampler** out);
int drb_sampler_destroy(drb_sampler* s);
/* fills n triples; val = 0 for null pairs, the stored interaction for positives */
int drb_sampler_sample(drb_sampler* s, int64_t n, int32_t* uid, int32_t* iid, double* val);
int drb_sampler_getstate(const drb_sampler* s, uint32_t state[3 * 625]);
int drb_sampler_setstate(drb_sampler* s, const uint32_t state[3 * 625]);

/* ------------------------------------------------------------------ CDAE corruption mask (host, MT19937)
 * replaces: DRecPy/Recommender/cdae.py:63-64 -- one rng.uniform(0,1) draw per item, in item order, for every
 * sampled user (n_items draws per user, zeros included).  Emits one keep byte per stored positive of each
 * sampled user: keep_off[b]..keep_off[b+1] index `keep` in CSR order of user uids[b] (csr = positives only,
 * column-sorted, host copy). */
int drb_cdae_corruption_keep_mt(drb_rng* rng, const int32_t* uids, int32_t batch, int32_t n_items, double q,
                                const int64_t* csr_indptr, const int32_t* csr_indices,
                                int32_t* keep_off /* [batch+1] */, uint8_t* keep /* [sum deg] */,
                                int64_t keep_capacity /* bytes available in keep; DRB_E_INVALID if too small */);
/* Device replay of the same stream (rng_mode='mt19937_device').  MT19937 is GF(2)-linear: a block of the stream J outputs
 * ahead is a fixed XOR-combination (the bits of t^J mod phi(t), phi = the characteristic polynomial) of the first
 * 19937 + 623 words of the stream.  drb_mtjump_create computes those polynomials once per (n_items, batch) for the
 * offsets seg_len * p, p = 1 .. n_seg (host, seconds); drb_mtjump_polys copies them out ([n_seg][312] uint64);
 * drb_mtjump_apply_host is the host reference of one jump (tests). */
typedef struct drb_mtjump drb_mtjump;
int drb_mtjump_create(int64_t seg_len, int32_t n_seg, drb_mtjump** out);
int drb_mtjump_destroy(drb_mtjump* j);
int drb_mtjump_polys(const drb_mtjump* j, uint64_t* out);
int drb_mtjump_apply_host(const drb_mtjump* j, int32_t p, const uint32_t* window_in, uint32_t* window_out);
/* One step of the stream on the device: keep[keep_off[b] + j] for every stored positive j of sampled user uids[b], exactly
 * what drb_cdae_corruption_keep_mt writes, from the 624-word window the step starts at (drb_rng_window); window_out
 * receives the window after batch * 2 * n_items outputs.  polys: (ceil(batch / users_per_cta) - 1) polynomials of the
 * offsets p * users_per_cta * 2 * n_items (drb_mtjump_create(users_per_cta * 2 * n_items, ...)), poly_total: the offset
 * batch * 2 * n_items; threshold = ceil(q * 2^53).  All pointers are device pointers; users_per_cta <= 64. */
int drb_mt_keep_device(drb_ctx* ctx, const uint32_t* window_in, uint32_t* window_out, const uint64_t* polys,
                       const uint64_t* poly_total, const int32_t* uids, const int32_t* keep_off, const int64_t* csr_indptr,
                       const int32_t* csr_indices, uint8_t* keep, int32_t batch, int32_t n_items, int32_t users_per_cta,
                       uint64_t threshold);
/* keep_off only (prefix of the sampled users' degrees), for the counter-based (philox) mask mode */
int drb_batch_offsets(const int32_t* uids, int32_t batch, const int64_t* csr_indptr, int32_t* keep_off);

/* ------------------------------------------------------------------ CDAE
 * Parameter arena layout (floats), all segments 16-byte aligned, row stride ld = K rounded up to a multiple of 4:
 *   [ W2T  n_items x ld | W  n_items x ld | b  ld | b2  n_items rounded up to a multiple of 4 | V  n_users x ld ]
 * W2T is the reference's W_ (cdae.py:37, [K, I]) stored item-major ([I, K]); pad columns k >= K stay zero.
 * params / adam_m / adam_v / grads share this layout.  Reference variable order for the per-variable Adam
 * step counters t[5] is [W, W_, V, b, b_] (cdae.py:43). */
typedef struct {
  int64_t off_w2t, off_w, off_v, off_b, off_b2, total; /* float offsets into the arena */
  int32_t ld, items_pad;
} drb_cdae_layout_t;
int drb_cdae_layout(int32_t n_users, int32_t n_items, int32_t hidden, drb_cdae_layout_t* out);
/* workspace bytes needed for batches up to max_batch (training) / max_score_users x max_candidates (scoring) */
int64_t drb_cdae_workspace_bytes(int32_t n_users, int32_t n_items, int32_t hidden, int32_t max_batch);
/* the same for a model created with output_mode = DRB_OUTPUT_SAMPLED (no batch x items buffers) */
int64_t drb_cdae_workspace_bytes_sampled(int32_t n_users, int32_t n_items, int32_t hidden, int32_t max_batch);

typedef struct {
  int32_t n_users, n_items, hidden;
  float* params;           /* device arenas (caller-owned) */
  float* adam_m;
  float* adam_v;
  float* grads;
  const int64_t* csr_indptr;   /* device CSR of positives (interaction >= threshold), column-sorted */
  const int32_t* csr_indices;
  const int64_t* seen_indptr;  /* device CSR of ALL stored rows (novelty filter of cdae.py:93-98); may alias csr_* */
  const int32_t* seen_indices;
  float corruption_level;      /* q */
  int32_t loss_kind;           /* DRB_LOSS_* */
  int32_t label_mode;          /* DRB_LABEL_* */
  void* workspace;             /* device, >= drb_cdae_workspace_bytes(...) */
  int64_t workspace_bytes;
  int32_t max_batch;
  int32_t gemm_path;           /* DRB_GEMM_AUTO (tcgen05 when hidden <= 256), DRB_GEMM_FFMA (exact fp32 on the CUDA cores),
                                  DRB_GEMM_TCGEN05 (fp32-accurate 3xFP16 split products), DRB_GEMM_TCGEN05_TF32 (3xTF32) */
  /* Sampled-output extension (NOT a reference behaviour: cdae.py:76 always scores the whole catalog; needed for catalogs
   * like BASELINE.json configs[4], 1 M items, where that is 1.5 GFLOP per sampled user).  output_mode DRB_OUTPUT_SAMPLED:
   * the training step scores each sampled user's positives plus neg_groups x neg_per_group uniformly drawn items (group
   * g = the g-th of neg_groups contiguous item ranges; one group per rank when the weights are item-sharded), with
   * per-user labels and the loss normalised by batch * neg_groups * neg_per_group.  Defined by
   * oracle/cdae.py: CDAESampledOracle.  Scoring entry points are unchanged (dense). */
  int32_t output_mode;         /* DRB_OUTPUT_DENSE (0, the reference) | DRB_OUTPUT_SAMPLED */
  int32_t neg_per_group, neg_groups;
} drb_cdae_desc;

typedef struct {
  float learning_rate, beta1, beta2, epsilon;  /* Keras Adam (recommender_abc.py:153): 1e-3, .9, .999, 1e-7 */
  float reg_rate;
  int32_t t[5];            /* Adam step counter per variable [W, W_, V, b, b_] (Q2: 5(s-1)+j+1) */
  uint64_t philox_seed;    /* used only when keep == NULL */
  uint64_t philox_step;
  int32_t global_batch;    /* data parallel: number of sampled users over all ranks (0 = batch) */
  int32_t slot_offset;     /* data parallel: global batch slot of local row 0 (philox counter) */
  int32_t skip_user_grad;  /* data parallel: leave dV to drb_cdae_scatter_user_rows (rows are all-gathered) */
  /* item-sharded weights (this model holds items [item_offset, item_offset + n_items) and a slice of V): */
  int32_t shard_items;     /* != 0 selects the item-sharded step */
  int32_t item_offset;     /* global id of local item 0 (philox counter) */
  int64_t n_items_global;  /* loss normalisation 1 / (global_batch * n_items_global) */
  const int32_t* v_rows;   /* device [batch]: local row of V for users this rank owns, -1 otherwise */
  int64_t keep_bytes;      /* optional: bytes of `keep` (= keep_off[batch]) when the caller knows it on the host; lets the
                              launch-bound small shapes replay the step as a CUDA graph from device-resident inputs */
} drb_cdae_step_args;

/* ------------------------------------------------------------------ optimizer of the dense update (K4)
 * replaces: the `optimizer=` keyword of recommender_abc.py:153 (any tf.keras optimizer, applied per variable at
 * :328-334).  Keras-2 / TF 2.0-2.3 OptimizerV2 dense updates in fp32; g is the gradient with the L2 term folded in:
 *   DRB_OPT_SGD      momentum == 0: w -= lr_t g;  else a = a momentum - lr_t g (slot adam_m), w += a, or with
 *                    nesterov w += a momentum - lr_t g
 *   DRB_OPT_RMSPROP  momentum == 0: ms = rho ms + (1-rho) g^2 (adam_m); centered: mg = rho mg + (1-rho) g (adam_v),
 *                    d = ms - mg^2, else d = ms; w -= lr_t g / (sqrt(d) + eps).
 *                    momentum > 0: ms += (g^2 - ms)(1-rho); centered: mg += (g - mg)(1-rho), d = ms - mg^2 + eps, else
 *                    d = ms + eps; mom = mom momentum + lr_t g / sqrt(d) (adam_v, or third_state when centered); w -= mom
 *   DRB_OPT_ADAGRAD  acc += g^2 (adam_m, which the caller initialises to initial_accumulator_value);
 *                    w -= lr_t g / (sqrt(acc) + eps)
 *   DRB_OPT_ADAMAX   m += (g - m)(1-beta1); u = max(beta2 u, |g|) (adam_v); w -= lr_t / (1 - beta1^t) m / (u + eps)
 *   DRB_OPT_ADAM     Keras Adam; amsgrad != 0: vhat = max(vhat, v) (third_state), w -= alpha_t m / (sqrt(vhat) + eps)
 * lr_t = learning_rate / (1 + decay (t - 1)) with learning_rate and the per-variable counters t of the step args.
 * A model that never calls drb_*_set_optimizer runs Adam with the beta1 / beta2 / epsilon of its step args; once it is
 * called, the descriptor's values are used instead (the step args then supply learning_rate and t only).  The slots are
 * the model's adam_m / adam_v arenas and, for AMSGrad and centered RMSprop with momentum only, third_state: a device
 * arena of the parameter arena's size and layout (caller-owned, 16-byte aligned, zero-initialised), borrowed until the
 * next call or the model's destruction.  Setting an optimizer does not touch any arena. */
enum { DRB_OPT_ADAM = 0, DRB_OPT_SGD = 1, DRB_OPT_RMSPROP = 2, DRB_OPT_ADAGRAD = 3, DRB_OPT_ADAMAX = 4 };
typedef struct {
  int32_t kind;            /* DRB_OPT_* */
  float momentum;          /* SGD, RMSprop: >= 0 */
  int32_t nesterov;        /* SGD */
  float rho;               /* RMSprop */
  int32_t centered;        /* RMSprop */
  float beta1, beta2;      /* Adam, Adamax: in [0, 1) */
  float epsilon;           /* > 0 for RMSprop, Adagrad, Adamax */
  int32_t amsgrad;         /* Adam */
  float decay;             /* Keras-2 time decay of the learning rate, >= 0 */
  float* third_state;      /* AMSGrad vhat / centered RMSprop with momentum: its momentum; else ignored (may be NULL) */
} drb_optim_desc;

enum {
  DRB_PHASE_PREP = 1,      /* clear gradients, label histogram / bitmap, philox mask */
  DRB_PHASE_GRADS_A = 2,   /* hidden layer (gather) + tf32 operand splits: needs no labels */
  DRB_PHASE_UPDATE = 4,    /* Adam + loss */
  DRB_PHASE_GRADS_B = 8,   /* output layer + loss epilogue, dW'^T, db' */
  DRB_PHASE_GRADS_C = 16,  /* dh, dz1, db, scatter into dW (and dV unless skip_user_grad) */
  DRB_PHASE_GRADS = 2 | 8 | 16,
  DRB_PHASE_ALL = 31,
  /* item-sharded step only: GRADS_A leaves the partial pre-activation in drb_cdae_h_buffer() (all-reduce it), then
   * GRADS_A2 applies the sigmoid; GRADS_C leaves the partial dh in drb_cdae_dz1_buffer() (all-reduce it), then
   * GRADS_C2 forms dz1 and scatters.  Rows of W / W' / V never travel, only batch x hidden activations do. */
  DRB_PHASE_GRADS_A2 = 32,
  DRB_PHASE_GRADS_C2 = 64,
  /* UPDATE in three launches (data parallel), each as soon as its gradient is final, so that the last gradient
   * all-reduce runs under the update of V: UPDATE_V (after drb_cdae_scatter_user_rows), UPDATE_W2T (after the
   * all-reduce of grads[0, off_w)), UPDATE_REST (W, b, b2 after the all-reduce of grads[off_w, off_v); writes the loss).
   * All three must run, UPDATE_REST last. */
  DRB_PHASE_UPDATE_V = 128,
  DRB_PHASE_UPDATE_W2T = 256,
  DRB_PHASE_UPDATE_REST = 512
};

int drb_cdae_create(drb_ctx* ctx, const drb_cdae_desc* desc, drb_cdae** out);
int drb_cdae_destroy(drb_cdae* m);
/* Selects the optimizer of every following step (see drb_optim_desc).  DRB_E_INVALID with a message for a descriptor
 * out of range.  Graphs captured for the previous optimizer are dropped. */
int drb_cdae_set_optimizer(drb_cdae* m, const drb_optim_desc* opt);
/* One training step on device-resident inputs.
 * replaces: recommender_abc.py:190-205 (tape, gradient, 5x apply_gradients) with cdae.py:50-82 inside.
 * uids[batch], keep_off[batch+1], keep[keep_off[batch]] are DEVICE pointers; keep == NULL selects the
 * counter-based mask (philox4x32-10 keyed by (seed, step, slot, item)).  loss_out: device float[2]
 * ([0] reported loss, [1] its batch term). */
int drb_cdae_step(drb_cdae* m, const int32_t* uids, const int32_t* keep_off, const uint8_t* keep,
                  int32_t batch, const drb_cdae_step_args* args, float* loss_out);
/* The same step in phases, for data parallelism over user mini-batches (one process per GPU, replicated weights):
 *   PREP   -> label histogram of the local batch; the caller all-reduces drb_cdae_label_count_buffer()
 *             (GRADS_A can run while that all-reduce is in flight, GRADS_C while dW'^T is being all-reduced)
 *   GRADS  -> (= GRADS_A | GRADS_B | GRADS_C) forward + backward with global_batch in the label mean / loss mean / L2 scale; the caller
 *             all-reduces the gradient arena [0, off_v) and, with skip_user_grad, all-gathers the (uid, dz1 row)
 *             pairs of drb_cdae_dz1_buffer() and adds them with drb_cdae_scatter_user_rows (rows of V never
 *             travel, only B x K activations' gradients do)
 *   UPDATE -> Adam + loss.  loss_out must hold TWO floats: [0] = batch term + regularisation, [1] = batch term of the
 *             local shard (sum [1] over ranks and add [0]-[1] for the global reported loss).
 * drb_cdae_step == all phases with loss_out[0..1]. */
int drb_cdae_step_phases(drb_cdae* m, const int32_t* uids, const int32_t* keep_off, const uint8_t* keep,
                         int32_t batch, const drb_cdae_step_args* args, float* loss_out, int32_t phases);
int drb_cdae_label_count_buffer(drb_cdae* m, float** ptr, int64_t* count);
int drb_cdae_dz1_buffer(drb_cdae* m, float** ptr, int64_t* count);   /* [max_batch][ld], rows 0..batch-1 valid */
int drb_cdae_h_buffer(drb_cdae* m, float** ptr, int64_t* count);     /* [max_batch][ld] hidden activations */
int drb_cdae_scatter_user_rows(drb_cdae* m, const int32_t* uids, const float* rows, int32_t n);
/* Same step with HOST inputs: copies uids / keep_off / keep to the device (inside the call), runs the step,
 * and, if loss_host != NULL, copies the loss back and synchronises. */
int drb_cdae_step_host(drb_cdae* m, const int32_t* uids, const int32_t* keep_off, const uint8_t* keep,
                       int32_t batch, const drb_cdae_step_args* args, float* loss_host);
/* Hidden representations h[n, ld] for n users, no corruption (cdae.py:67-76 first line).  uids: device. */
/* device float[2] that drb_cdae_step_host leaves the loss in (valid after the step's stream work) */
int drb_cdae_loss_buffer(drb_cdae* m, float** ptr);
int drb_cdae_hidden(drb_cdae* m, const int32_t* uids, int32_t n, float* h_out);
/* Candidate scoring + ranking.  replaces: cdae.py:84-103 (_predict over all items, filter, heapq.nlargest).
 * cand[n x max_cand] internal item ids (device), cand_count[n]; entries beyond the count are ignored.
 * If novelty != 0, candidates present in the user's `seen` row are dropped.  Output per user: n_out[u] ranked
 * entries, ordered by (score desc, iid desc) == heapq.nlargest on (score, iid) tuples. */
int drb_cdae_rank_candidates(drb_cdae* m, const int32_t* uids, int32_t n, const int32_t* cand,
                             const int32_t* cand_count, int32_t max_cand, int32_t novelty,
                             int32_t* out_iid, float* out_score, int32_t* n_out);
/* Full-catalog top-k.  replaces: recommender_abc.py:413-419 -> cdae.py:90-103 with iids = range(n_items), i.e. what
 * Evaluation/Processes/recommendation_evaluation.py:164 asks of the model for every user.
 * out_iid / out_score: [n x k]; n_out[u] <= k entries ordered by (score desc, iid desc).
 * Wide catalogs and blocks of >= 128 users run on the tensor cores (tcgen05 h W'^T tiles whose epilogue keeps only the
 * scores above a per-user threshold; no score is written to memory).  Its per-user candidate lists are bounded: a user
 * whose list overflowed is re-done on the device by the exact path; if more than 32 users of one block overflow, the
 * remaining ones are reported with n_out[u] == -1 and the caller re-runs them through drb_cdae_topk_exact. */
int drb_cdae_topk(drb_cdae* m, const int32_t* uids, int32_t n, int32_t k, int32_t novelty,
                  int32_t* out_iid, float* out_score, int32_t* n_out);
/* Same contract, always the exact-fp32 score rows + radix select (any catalog size, any number of users). */
int drb_cdae_topk_exact(drb_cdae* m, const int32_t* uids, int32_t n, int32_t k, int32_t novelty,
                        int32_t* out_iid, float* out_score, int32_t* n_out);
/* Dense scores for n users over all items: out[n x items_pad] (cdae.py:84-88 with iid=None). */
int drb_cdae_predict_all(drb_cdae* m, const int32_t* uids, int32_t n, float* out);
/* Scores of n (user, item) pairs.  replaces: recommender_abc.py:354-383 -> cdae.py:84-88 (_predict: the user's whole
 * score row, then one element of it) once per pair.  Pairs are grouped by user: users[n_users] internal uids, user b
 * owns pairs [pair_off[b], pair_off[b+1]) (pair_off[0] = 0, pair_off[n_users] = n, non-decreasing), pair q scores
 * internal item pair_iid[q] into out[pair_dst[q]].  All device pointers; the call synchronises the context's stream
 * once, to check the arguments (DRB_E_INVALID for an id or position out of range or a bad pair_off).  Every value is
 * bit for bit the element drb_cdae_predict_all gives for that user and item. */
int drb_cdae_predict_pairs(drb_cdae* m, const int32_t* users, int32_t n_users, const int64_t* pair_off,
                           const int32_t* pair_iid, const int32_t* pair_dst, int32_t n, float* out);

/* ------------------------------------------------------------------ DMF
 * Tower l has kernel [in_l, out_l] (row stride ld_l = out_l rounded up to a multiple of 4) and bias [ld_l].
 * Arena layout: user tower layers in order (kernel, bias), then item tower layers.  in_0 = n_items for the
 * user tower and n_users for the item tower (dmf.py:48-58). */
#define DRB_DMF_MAX_LAYERS 8
typedef struct {
  int32_t n_layers_user, n_layers_item;
  int64_t off_kernel_user[DRB_DMF_MAX_LAYERS], off_bias_user[DRB_DMF_MAX_LAYERS];
  int64_t off_kernel_item[DRB_DMF_MAX_LAYERS], off_bias_item[DRB_DMF_MAX_LAYERS];
  int32_t ld_user[DRB_DMF_MAX_LAYERS], ld_item[DRB_DMF_MAX_LAYERS];
  int64_t total;
} drb_dmf_layout_t;
int drb_dmf_layout(int32_t n_users, int32_t n_items, const int32_t* user_factors, int32_t n_user_layers,
                   const int32_t* item_factors, int32_t n_item_layers, drb_dmf_layout_t* out);
int64_t drb_dmf_workspace_bytes(int32_t n_users, int32_t n_items, const int32_t* user_factors,
                                int32_t n_user_layers, const int32_t* item_factors, int32_t n_item_layers,
                                int32_t max_batch);

typedef struct {
  int32_t n_users, n_items;
  int32_t n_layers_user, n_layers_item;
  int32_t user_factors[DRB_DMF_MAX_LAYERS], item_factors[DRB_DMF_MAX_LAYERS];
  float* params;
  float* adam_m;
  float* adam_v;
  float* grads;
  /* device CSR (user rows over items) and CSC (item rows over users) of ALL stored interactions with raw
   * values (duplicates summed), column-sorted; row_scale = rsqrt(max(sum v^2, 1e-12)) per row when
   * l2_norm_vectors (dmf.py:82-84), else NULL */
  const int64_t* csr_indptr; const int32_t* csr_indices; const float* csr_values; const float* csr_row_scale;
  const int64_t* csc_indptr; const int32_t* csc_indices; const float* csc_values; const float* csc_row_scale;
  void* workspace;
  int64_t workspace_bytes;
  int32_t max_batch;
} drb_dmf_desc;

typedef struct {
  float learning_rate, beta1, beta2, epsilon;
  float reg_rate;
  int32_t t[2];            /* Adam step counter per tower [user_nn, item_nn] (Q2: 2(s-1)+g+1) */
} drb_dmf_step_args;

int drb_dmf_create(drb_ctx* ctx, const drb_dmf_desc* desc, drb_dmf** out);
int drb_dmf_destroy(drb_dmf* m);
/* drb_cdae_set_optimizer for DMF (t of the step args: the per-tower counters) */
int drb_dmf_set_optimizer(drb_dmf* m, const drb_optim_desc* opt);
/* replaces: recommender_abc.py:190-205 with dmf.py:64-99 inside.  uids/iids/labels: device [batch];
 * loss_out: device float[2] ([0] reported loss, [1] its batch term). */
int drb_dmf_step(drb_dmf* m, const int32_t* uids, const int32_t* iids, const float* labels, int32_t batch,
                 const drb_dmf_step_args* args, float* loss_out);
/* The same step in two phases, for data parallelism over pair mini-batches (one process per GPU, replicated weights;
 * the reference is single-process, so this layer is new):
 *   DRB_DMF_PHASE_GRADS  forward + backward into the gradient arena (drb_dmf_grads_buffer), with the loss mean and its
 *                        gradient over global_batch pairs (0 = batch); the caller all-reduces the arena (2.5 MB at the
 *                        ml-1m shape) ...
 *   DRB_DMF_PHASE_UPDATE ... then Adam + loss.  loss_out[1] is this rank's share of the batch term (sum it over ranks
 *                        and add loss_out[0] - loss_out[1], the regularisation term, for the global reported loss). */
enum { DRB_DMF_PHASE_GRADS = 1, DRB_DMF_PHASE_UPDATE = 2, DRB_DMF_PHASE_ALL = 3 };
int drb_dmf_step_phases(drb_dmf* m, const int32_t* uids, const int32_t* iids, const float* labels, int32_t batch,
                        const drb_dmf_step_args* args, float* loss_out, int32_t phases, int32_t global_batch);
int drb_dmf_grads_buffer(drb_dmf* m, float** ptr, int64_t* count);
int drb_dmf_step_host(drb_dmf* m, const int32_t* uids, const int32_t* iids, const float* labels, int32_t batch,
                      const drb_dmf_step_args* args, float* loss_host);
int drb_dmf_loss_buffer(drb_dmf* m, float** ptr);
/* p[n] = max(1e-6, cos(user tower(uid), item tower(iid))) for n pairs (dmf.py:88-96, un-rescaled). device. */
int drb_dmf_forward_pairs(drb_dmf* m, const int32_t* uids, const int32_t* iids, int32_t n, float* p_out);
/* The same p for n pairs grouped by user, with the arguments of drb_cdae_predict_pairs.  replaces: recommender_abc.py:
 * 354-383 -> dmf.py:101-106 (_predict: both towers for one pair) once per pair.  The user tower runs once per entry of
 * users; the item side comes from the item-tower cache of drb_dmf_rank_candidates.  Every value is bit for bit what
 * drb_dmf_forward_pairs gives for that pair (un-rescaled). */
int drb_dmf_predict_pairs(drb_dmf* m, const int32_t* users, int32_t n_users, const int64_t* pair_off,
                          const int32_t* pair_iid, const int32_t* pair_dst, int32_t n, float* p_out);
/* replaces: recommender_abc.py:454-461 (one _predict per candidate + nlargest).  Same contract as
 * drb_cdae_rank_candidates; scores are the un-rescaled p (rescaling is monotone, done by the host). */
int drb_dmf_rank_candidates(drb_dmf* m, const int32_t* uids, int32_t n, const int32_t* cand,
                            const int32_t* cand_count, int32_t max_cand, int32_t novelty,
                            int32_t* out_iid, float* out_score, int32_t* n_out);
/* drb_dmf_rank_candidates keeps the item tower's output for the whole catalog until the next drb_dmf_step; a caller
 * that writes the parameter arena itself (weight injection, _revert_weights: recommender_abc.py:346-352) says so. */
int drb_dmf_invalidate_cache(drb_dmf* m);
/* replaces: recommender_abc.py:391-419 (recommend -> _recommend = _rank over range(n_items)) -> :454-461 (DMF: one
 * _predict per candidate, dmf.py:101-106, then nlargest), for n users at once.  uids: device [n]; out_iid / out_score
 * [n][k], n_out [n] (device).  Row u == drb_dmf_rank_candidates(uids[u], whole catalog) truncated to k, ids and fp32
 * scores bit for bit; n_out[u] == -1: list overflow beyond the device fallback, re-run the user through the rank path.
 * scratch: caller-owned device memory of drb_dmf_topk_scratch_bytes(m, k) bytes (-1: bad argument, see
 * drb_last_error).  1 <= k <= 2048.  Shares the item-tower cache of drb_dmf_rank_candidates. */
int64_t drb_dmf_topk_scratch_bytes(drb_dmf* m, int32_t k);
int drb_dmf_topk(drb_dmf* m, const int32_t* uids, int32_t n, int32_t k, int32_t novelty, void* scratch,
                 int64_t scratch_bytes, int32_t* out_iid, float* out_score, int32_t* n_out);

/* ------------------------------------------------------------------ Caser
 * Tang & Wang, "Personalized Top-N Sequential Recommendation via Convolutional Sequence Embedding" (WSDM 2018), the
 * third deep recommender of DRecPy.  The model, its batch sampler and its dropout stream are pinned by oracle/caser.py
 * (parity with DRecPy's TensorFlow Caser is unpinned, DESIGN.md section 8).  Supported sizes: 1 <= L <= 16,
 * 1 <= T <= 32, 1 <= d <= 256, 1 <= n_v, n_h <= 64, and the conv / fc weights with their gradients must fit the 227 KB
 * of shared memory of one CTA (drb_caser_layout fails with a message otherwise).
 * Arena layout (floats), every tensor 16-byte aligned, first the tensors under L2, then those without:
 *   [ E n_items x ld_e | P n_users x ld_e | W2 n_items x ld_x | Fv L x n_v | Fh | fc (n_v d + n_h L) x d ]
 *   [ bv n_v | bh L x n_h | b_fc d | b2 n_items ]
 * ld_e = d and ld_x = 2d rounded up to a multiple of 4 (pad columns stay zero); Fh holds the horizontal kernels
 * h = 1 .. L one after the other, kernel h [h][d][n_h] at n_h d (h - 1) h / 2; bh row h - 1 is the bias of kernel h;
 * fc is Keras-shaped [in][out], its input ordered [vertical output c d + k for c < n_v, k < d; pooled horizontal output
 * (h - 1) n_h + f].  The L2 tensors end at off_bv. */
typedef struct {
  int64_t off_e, off_p, off_w2, off_fv, off_fh, off_fc, off_bv, off_bh, off_bfc, off_b2, total;
  int32_t ld_e, ld_x, items_pad;
} drb_caser_layout_t;
int drb_caser_layout(int32_t n_users, int32_t n_items, int32_t L, int32_t T, int32_t d, int32_t n_v, int32_t n_h,
                     drb_caser_layout_t* out);
int64_t drb_caser_workspace_bytes(int32_t n_users, int32_t n_items, int32_t L, int32_t T, int32_t d, int32_t n_v,
                                  int32_t n_h, int32_t neg_ratio, int32_t max_batch);

typedef struct {
  int32_t n_users, n_items, L, T, d, n_v, n_h, neg_ratio;
  float dropout_rate;          /* in [0, 1) */
  float* params;               /* device arenas (caller-owned) */
  float* adam_m;
  float* adam_v;
  float* grads;
  /* device: the training sequences (CSR over users, each user's items in sequence order) and the prefix sums of the
   * windows of L + T consecutive items per user ([n_users + 1], win_off[n_users] = n_windows > 0) */
  const int32_t* seq; const int64_t* seq_indptr;
  const int64_t* win_off; int64_t n_windows;
  const int64_t* seen_indptr;  /* device CSR of ALL stored rows, column-sorted: negatives and the novelty filter */
  const int32_t* seen_indices;
  void* workspace;             /* device, >= drb_caser_workspace_bytes(...) */
  int64_t workspace_bytes;
  int32_t max_batch;           /* windows per step and users per scoring chunk */
} drb_caser_desc;

typedef struct {
  float learning_rate, beta1, beta2, epsilon;
  float reg_rate;
  int32_t t;                   /* optimizer step counter, the same for every tensor */
  uint64_t philox_seed;        /* key of the sampler and dropout streams */
  uint64_t philox_step;        /* counter words 2-3 of every draw of this step */
} drb_caser_step_args;

int drb_caser_create(drb_ctx* ctx, const drb_caser_desc* desc, drb_caser** out);
int drb_caser_destroy(drb_caser* m);
/* drb_cdae_set_optimizer for Caser */
int drb_caser_set_optimizer(drb_caser* m, const drb_optim_desc* opt);
/* One training step of `batch` windows, drawn on the device (nothing is read from the host): sampler, fused forward +
 * backward into the gradient arena (raw gradients, without the L2 term), the dense update of the whole arena, and the
 * loss.  loss_out: device float[2] ([0] reported loss = mean BCE + reg_rate sum w^2 over the L2 tensors, [1] the BCE
 * term).  Launch-bound shapes replay the step as one CUDA graph. */
int drb_caser_step(drb_caser* m, int32_t batch, const drb_caser_step_args* args, float* loss_out);
int drb_caser_loss_buffer(drb_caser* m, float** ptr);   /* device float[2] for loss_out */
/* The batch of the last step (device): users[max_batch], items[max_batch][row_len] = L inputs, T targets,
 * T * neg_ratio negatives. */
int drb_caser_batch_buffer(drb_caser* m, int32_t** users, int32_t** items, int32_t* row_len);
/* x[n][ld_x] = [z; P[u]] for n users (device), from the last L items of each sequence, left-padded with zero rows,
 * without dropout.  n <= max_batch. */
int drb_caser_user_rep(drb_caser* m, const int32_t* uids, int32_t n, float* x_out);
/* Scores sigmoid(x W2[j] + b2[j]) of n users over all items: out[n x items_pad] (one fmaf chain over ld_x). */
int drb_caser_predict_all(drb_caser* m, const int32_t* uids, int32_t n, float* out);
/* Pair scores with the arguments of drb_cdae_predict_pairs; bit for bit the elements of drb_caser_predict_all. */
int drb_caser_predict_pairs(drb_caser* m, const int32_t* users, int32_t n_users, const int64_t* pair_off,
                            const int32_t* pair_iid, const int32_t* pair_dst, int32_t n, float* out);
/* Contract of drb_cdae_rank_candidates; every score is bit for bit the drb_caser_predict_all element. */
int drb_caser_rank_candidates(drb_caser* m, const int32_t* uids, int32_t n, const int32_t* cand,
                              const int32_t* cand_count, int32_t max_cand, int32_t novelty,
                              int32_t* out_iid, float* out_score, int32_t* n_out);
/* Full-catalog top-k, contract of drb_cdae_topk_exact (1 <= k <= 2048); scores bit for bit those of
 * drb_caser_predict_all. */
int drb_caser_topk(drb_caser* m, const int32_t* uids, int32_t n, int32_t k, int32_t novelty,
                   int32_t* out_iid, float* out_score, int32_t* n_out);

/* ------------------------------------------------------------------ kernel-level test hooks (tests/ only)
 * The tcgen05 GEMM building blocks of the CDAE step, exposed so that tests can check them in isolation against
 * a float64 product.  All pointers are device pointers.
 * drb_debug_split_tf32: src[rows][ld] -> hi/lo (same layout; may be NULL) and transposed t_hi/t_lo[cols][ldt]
 * (may be NULL); ones_row >= 0 sets that transposed row to 1.
 * drb_debug_umma_gemm: C[m][n] = sum_k A(m,k) B(n,k) as 3 TF32 products.  a_mn_major == 0: A stored [M][lda] (k
 * contiguous); != 0: A stored [Kred][lda] (m contiguous).  B stored [b_rows][ldb] (k contiguous).  Partial z of a
 * split reduction is written at C + z*M*ldc; columns >= n_store are dropped; column extra_col_index goes to
 * extra_col[m] when extra_col != NULL. */
/* drb_debug_cdae_capture_logits: while z_out != NULL every following training step also stores the output-layer
 * logits z2 = h W'^T + b' (cdae.py:76 before the sigmoid) exactly as the tcgen05 loss kernel formed them, row-major
 * [batch][items_pad] floats at z_out (device).  NULL switches the capture off.  Only the tensor-core path. */
int drb_debug_cdae_capture_logits(drb_cdae* m, float* z_out);
int drb_debug_split_tf32(drb_ctx* ctx, const float* src, int32_t rows, int32_t cols, int32_t ld, float* hi, float* lo,
                         float* t_hi, float* t_lo, int32_t ldt, int32_t ones_row);
int drb_debug_umma_gemm(drb_ctx* ctx, const float* a_hi, const float* a_lo, int32_t lda, const float* b_hi,
                        const float* b_lo, int32_t ldb, int32_t b_rows, int32_t a_mn_major, int32_t M, int32_t N,
                        int32_t Kred, int32_t splits, float* C, int32_t ldc, int32_t n_store, float* extra_col,
                        int32_t extra_col_index);

/* The 3xFP16 forms of the same building blocks: x * alpha -> fp16 hi / lo ([rows][ldh halfs]; transposed [cols..][ldt
 * halfs], ones_row set to alpha), and C = out_scale * sum_k A(m,k) B(n,k) from K-major fp16 hi / lo operands
 * (A [M][lda halfs], or with a_mn_major != 0 A stored as [Kred][lda halfs] with m contiguous; B [b_rows][ldb halfs];
 * pitches are multiples of 8). */
int drb_debug_split_f16(drb_ctx* ctx, const float* src, int32_t rows, int32_t cols, int32_t ld, float alpha, void* hi,
                        void* lo, int32_t ldh, void* t_hi, void* t_lo, int32_t ldt, int32_t ones_row);
int drb_debug_umma_gemm_f16(drb_ctx* ctx, const void* a_hi, const void* a_lo, int32_t lda, const void* b_hi,
                            const void* b_lo, int32_t ldb, int32_t b_rows, int32_t a_mn_major, int32_t M, int32_t N, int32_t Kred,
                            int32_t splits, float out_scale, float* C, int32_t ldc, int32_t n_store, float* extra_col,
                            int32_t extra_col_index);

/* ------------------------------------------------------------------ ranking_evaluation candidate generation
 * replaces: DRecPy/Evaluation/Processes/ranking_evaluation.py:108-116,163-219 -- per-user
 * random.Random(seed+idx), rng.sample of positives / negatives, randint generation of extra negatives,
 * rng.shuffle.  Test rows are grouped by user in evaluation order (row order inside a user preserved):
 * test_indptr[n_users+1], test_item (raw ids), test_val.  Training positives (ignored when train_evaluation != 0
 * or black_row == NULL): black_row[u] = training-set row (internal uid) of evaluated user u or -1;
 * black_indptr / black_iid = the training CSR of positives over internal item ids (sorted per row);
 * raw_sorted[n_map] / raw_to_iid[n_map] = sorted raw item ids and their internal ids.
 * n_pos < 0 / n_neg < 0 mean "None"; user u is seeded with abs(seed + u); n_neg_is_frac != 0 means
 * n_neg = int(frac * n_positives).  Users are independent, so the work is split over n_threads host threads.
 * Outputs: cand_off[n_users+1] (caller passes capacity via cand_capacity), cand (raw ids, shuffled),
 * pos (raw ids of the sampled positives, pos_off[n_users+1]), skipped[u] != 0 when the reference returns early
 * for that user. */
int drb_eval_candidates(int64_t n_users, const int64_t* test_indptr, const int64_t* test_item,
                        const double* test_val, const int64_t* black_row, const int64_t* black_indptr,
                        const int32_t* black_iid, const int64_t* raw_sorted, const int32_t* raw_to_iid,
                        int64_t n_map, int32_t train_evaluation, int64_t n_items, double threshold, int64_t n_pos,
                        double n_neg, int32_t n_neg_is_frac, int32_t generate_negative_pairs, int64_t seed,
                        int32_t n_threads, int64_t cand_capacity, int64_t* cand_off, int64_t* cand, int64_t* pos_off,
                        int64_t* pos, uint8_t* skipped);

/* Grouped first-match lookup (replaces the per-candidate ds_test.select_one('uid == .., iid == ..') of
 * DRecPy/Evaluation/Processes/ranking_evaluation.py:222-223 and the `item in positives` tests of
 * Evaluation/Metrics/ranking.py:32-56).  For group g, out[q] = tab_val of the first row r in [tab_beg[g], tab_end[g])
 * with tab_key[r] == q_key[q] (1.0 when tab_val is NULL), else `miss`, for every q in [q_beg[g], q_end[g]).
 * Positions of `out` outside every query range are left untouched. */
int drb_eval_lookup(int64_t n_groups, const int64_t* tab_beg, const int64_t* tab_end, const int64_t* tab_key,
                    const double* tab_val, const int64_t* q_beg, const int64_t* q_end, const int64_t* q_key,
                    double miss, int32_t n_threads, double* out);

/* Per-user sums of the ranking metrics for every evaluated user at once (replaces the per-user metric calls of
 * DRecPy/Evaluation/Processes/ranking_evaluation.py:222-241 -> Evaluation/Metrics/ranking.py:20-114: DCG / NDCG with
 * strong relevancy, and the hit counts behind HitRatio / Recall / Precision).  For user g: the relevancy of an item is
 * the value of the first row r in [tab_beg[g], tab_end[g]) with tab_key[r] == item, else 0 (ranking_evaluation.py:223);
 * ranked[g * ld_ranked .. + n_out[g]) is the model's ranked list, [c_beg[g], c_end[g]) of c_key the candidate list and
 * [p_beg[g], p_end[g]) of p_key the sampled positives.  For every cut-off ks[j] (ascending or not):
 *   dcg[g * n_ks + j]  = sum_{i < min(ks[j], n_out[g])} (2^rel(ranked_i) - 1) / log2(2 + i), added in that order,
 *   idcg[g * n_ks + j] = the same sum over the candidates' relevancies in descending order (i < min(ks[j], #candidates)),
 *   hits[g * n_ks + j] = how many of the first min(ks[j], n_out[g]) ranked items are sampled positives.
 * Same float64 operations in the same order as the reference's Python loops (pow, log2 of the C library). */
int drb_eval_metrics(int64_t n_groups, const int64_t* tab_beg, const int64_t* tab_end, const int64_t* tab_key,
                     const double* tab_val, const int64_t* ranked, int64_t ld_ranked, const int32_t* n_out,
                     const int64_t* c_beg, const int64_t* c_end, const int64_t* c_key, const int64_t* p_beg,
                     const int64_t* p_end, const int64_t* p_key, const int64_t* ks, int32_t n_ks, int32_t n_threads,
                     double* dcg, double* idcg, int64_t* hits);

/* The same per-user sums for full-catalog top-k lists that are still on the device (replaces the per-user metric calls
 * of DRecPy/Evaluation/Processes/recommendation_evaluation.py:164-192 on model.recommend's list), enqueued on the
 * context's stream without synchronising.  All pointers are device pointers.  User u's list is top_iid / top_score
 * [u * ld .. + n_out[u]) as drb_cdae_topk / drb_dmf_topk leave it (internal item ids, descending scores); its valid
 * prefix is the first min(n_out[u], k_max) entries, cut at the first score < (float)threshold when use_threshold != 0.
 * lut_iid[lut_off[u] .. lut_off[u+1]) are the internal ids, sorted ascending, of the user's evaluated items with their
 * gain lut_gain (2^rel - 1) and lut_pos != 0 for a sampled positive; ideal_gain[ideal_off[u] .. ideal_off[u+1]) are the
 * gains of all the user's evaluated items (also those the model does not know); disc[i] = log2(2 + i) for i < k_max;
 * ks[n_ks] the cut-offs, 1 <= ks[j] <= k_max <= ld.  Outputs [n][n_ks]: dcg / hits over the first min(ks[j], n_valid)
 * entries, idcg over the largest min(ks[j], #ideal gains) gains in descending order, n_rec = min(ks[j], n_valid).  Bit
 * for bit what drb_eval_metrics computes for the same valid prefix, with the evaluated items as test table and
 * candidate list. */
int drb_eval_topk_metrics(drb_ctx* ctx, int32_t n, const int32_t* top_iid, const float* top_score, int32_t ld,
                          const int32_t* n_out, int32_t use_threshold, double threshold, const int64_t* lut_off,
                          const int32_t* lut_iid, const double* lut_gain, const uint8_t* lut_pos,
                          const int64_t* ideal_off, const double* ideal_gain, const double* disc, const int32_t* ks,
                          int32_t n_ks, int32_t k_max, double* dcg, double* idcg, int32_t* hits, int32_t* n_rec);

/* Leave-k-out split for every user at once (replaces DRecPy/Evaluation/Splits/leave_k_out.py:58-135: one
 * interaction_dataset.select('user == ...') plus rng.sample per user on a thread pool).  Rows are given grouped by
 * user in order of first appearance, each group in DataFrame order: group idx spans user_indptr[idx]..[idx+1].  User
 * idx draws from random.Random(seed + idx + 1) (the reference increments the seed before creating the generator,
 * leave_k_out.py:68-69).  k_fixed rows per user go to the test set (is_ratio: int(len * k_ratio), :98-99) when the
 * user has more than k rows (:119); users with fewer than min_user_interactions rows are removed (:115-117).
 * flags[pos] = 0 train, 1 test, 2 removed; the caller zero-fills flags.  The last_timestamps variant stays in Python. */
int drb_leave_k_out(int64_t n_users, const int64_t* user_indptr, int64_t k_fixed, double k_ratio, int32_t is_ratio,
                    int64_t min_user_interactions, int64_t seed, int32_t n_threads, uint8_t* flags);

#ifdef __cplusplus
}
#endif
#endif /* DRB_H */
