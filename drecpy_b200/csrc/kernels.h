// Launcher prototypes of the sm_100a kernels behind libdrb.so (internal, not part of the ABI).
// Kernel ids follow SURVEY.md section 2b: K1 gather, K2/K3 dense output layer + backward, K3 scatter,
// K4 fused Adam+L2, K5 DMF head, K6 scoring / top-k.
#ifndef DRB_KERNELS_H
#define DRB_KERNELS_H

#include "drb_internal.h"

// ------------------------------------------------------------------ sparse.cu
struct GatherArgs {
  const int64_t* indptr; const int32_t* indices; const float* values;  // values may be NULL (all ones)
  const int32_t* rows;                                                  // [n] CSR row of each output row
  const int32_t* keep_off; const uint8_t* keep;                         // may be NULL (keep everything)
  const float* table; int ld;                                           // gathered table [*, ld]
  const float* rowbias;                                                 // may be NULL; [*, ld] indexed by rows[b]
  const int32_t* bias_rows;                                             // may be NULL; else rowbias row per output row,
                                                                        // -1 = add neither rowbias nor bias (item-sharded)
  const float* bias;                                                    // may be NULL; [ld]
  const float* row_scale;                                               // may be NULL; per CSR row
  float scale; int act; int width;                                      // columns >= width are forced to 0
  float* out;                                                           // [n, ld]
  const int32_t* chunk_off;                                             // may be NULL; [n + 1] from launch_chunk_scan:
                                                                        // balanced form (pieces of 256 CSR entries,
                                                                        // atomics into out, then a finishing pass)
  // optional fused dense layer on the row just produced (second Dense layer of a DMF tower), one-CTA-per-row form only:
  // next_out[n, next_ld] = act(out . next_k[width x next_ld] + next_b); columns >= next_width are 0
  const float* next_k; const float* next_b; int next_ld, next_width, next_act; float* next_out;
};
struct GatherPair { GatherArgs a[2]; };
int launch_gather(drb_ctx* ctx, const GatherArgs& a, int n);
// two gathers of equal row width as ONE launch (blockIdx.y selects): the two towers of a DMF step
int launch_gather_pair(drb_ctx* ctx, const GatherArgs& a0, const GatherArgs& a1, int n);
// chunk_off[b] = number of 256-entry pieces of the CSR rows rows[0..b), chunk_off[n] = total
int launch_chunk_scan(drb_ctx* ctx, const int64_t* indptr, const int32_t* rows, int n, int32_t* chunk_off);

struct ScatterArgs {
  const int64_t* indptr; const int32_t* indices; const float* values;
  const int32_t* rows;
  const int32_t* keep_off; const uint8_t* keep;
  const float* row_scale; float scale;
  const float* d; int ld;             // [n, ld] row gradients
  float* gtable;                      // [*, ld] += w * d[b]   (vector atomics)
  float* growbias;                    // may be NULL; [*, ld] += d[b] at rows[b]
  const int32_t* bias_rows;           // may be NULL; else the growbias row per batch row, -1 = skip (item-sharded)
  const int32_t* chunk_off;           // may be NULL; balanced form, see GatherArgs
  uint32_t* row_touched = nullptr;    // may be NULL; bit r is set when growbias row r received a gradient (k_adam then
                                      // knows which rows of a zero-initialised gradient table it has to read)
};
struct ScatterPair { ScatterArgs a[2]; };
int launch_scatter(drb_ctx* ctx, const ScatterArgs& a, int n);
int launch_scatter_pair(drb_ctx* ctx, const ScatterArgs& a0, const ScatterArgs& a1, int n);

// gtable[ids[r]] += rows[r]  (one warp per row, vector atomics) -- data-parallel exchange of the user-row gradients
int launch_row_scatter(drb_ctx* ctx, const int32_t* ids, const float* rows, int n, int ld, float* gtable,
                       uint32_t* row_touched = nullptr);

// per batch row: label histogram (batch_mean) or bitmap (per_user) and, in philox mode, the keep bytes
struct BatchPrepArgs {
  const int64_t* indptr; const int32_t* indices; const int32_t* rows; const int32_t* keep_off;
  float* count;            // may be NULL; [items_pad] += 1 per stored positive
  uint32_t* label_bits;    // may be NULL; [n, words_per_row]
  int words_per_row;
  uint8_t* keep_out;       // may be NULL; philox keep bytes
  uint64_t seed, step; float q;
  const uint32_t* step_dev;  // may be NULL; else the step counter is {step_dev[0], step_dev[1]} (lo, hi): graph replay
  int slot_offset;         // global slot of local row 0 (data parallel), part of the philox counter
  int item_offset;         // global id of local item 0 (item-sharded), part of the philox counter
};
int launch_batch_prep(drb_ctx* ctx, const BatchPrepArgs& a, int n);

// dz1 = (sum_s dh_part[s]) * h * (1 - h); column partial sums per 32-row block -> colpart[nblk, ld]
int launch_dz1(drb_ctx* ctx, const float* dh_part, int splits, const float* h, float* dz1, int n, int ld,
               float* colpart);
// column partials of x[n, ld] per 32-row block (generic bias gradient)
int launch_colpart(drb_ctx* ctx, const float* x, int n, int ld, float* colpart);
// table[ids[r]][:] = 0 for r < n
int launch_zero_rows(drb_ctx* ctx, float* table, const int32_t* ids, int n, int ld, uint32_t* row_touched = nullptr);
// out[i] = start + i
int launch_iota(drb_ctx* ctx, int32_t* out, int n, int start);
// out[e] = sum_s part[s][e] (e < n_elems); in-place sigmoid of x[n][ld] with columns >= width forced to 0
int launch_sum_planes(drb_ctx* ctx, const float* part, int planes, int64_t n_elems, float* out);
int launch_sigmoid_rows(drb_ctx* ctx, float* x, int n, int ld, int width);
// out[j] = sum_p part[p, ld + j]
int launch_reduce_partials(drb_ctx* ctx, const float* part, int nparts, int ld, float* out, int n);

// ------------------------------------------------------------------ mt_device.cu
// Device replay of the reference's MT19937 corruption stream (cdae.py:63-64): keep bytes of the batch's positives.
struct MtKeepArgs {
  const uint32_t* window_in; uint32_t* window_out;     // 624-word windows: the stream at the start / end of this step
  const uint64_t* polys;                               // [n_cta - 1][312]: jump polynomials of offsets p * ups * 2 * n_items
  const uint64_t* poly_total;                          // [312]: offset batch * 2 * n_items
  const int32_t* uids; const int32_t* keep_off;        // [batch], [batch + 1]
  const int64_t* indptr; const int32_t* indices;       // CSR of positives, column-sorted
  uint8_t* keep;                                       // [keep_off[batch]]
  int batch, n_items, ups, n_cta;                      // ups = batch rows per CTA, n_cta = ceil(batch / ups)
  uint64_t threshold;                                  // ceil(q * 2^53): a draw below it drops the entry
};
int launch_mt_keep(drb_ctx* ctx, const MtKeepArgs& a);

// ------------------------------------------------------------------ sampled.cu
// Sampled-output layer (extension for configs[4], see sampled.cu / oracle.cdae.CDAESampledOracle): forward + backward of
// the output layer over each sampled user's positives and n_groups x neg_per_group drawn items.
struct SampledOutArgs {
  const int64_t* indptr; const int32_t* indices; const int32_t* rows;   // positives CSR over LOCAL item ids, column-sorted
  const float* h; int ld;                     // [n, ld] hidden activations
  const float* w2t; const float* b2;          // [n_items_local, ld], [n_items_local]
  float* g_w2t; float* g_b2;                  // their gradients (pre-zeroed; vector atomics)
  float* dh;                                  // [n, ld] written (partial over the local items when item-sharded)
  float* loss_part;                           // [n] raw sums of the loss terms
  int n_items_total, n_groups_total;          // the GLOBAL catalog and its partition into negative-sampling groups
  int n_groups, group_id0, item_offset;       // groups this model holds: [group_id0, group_id0 + n_groups); global id of local item 0
  int neg_per_group;
  uint64_t seed, step; const uint32_t* step_dev; int slot_offset;
  int loss_kind; float inv_count;             // 1 / (global batch * n_groups_total * neg_per_group)
};
int launch_sampled_out(drb_ctx* ctx, const SampledOutArgs& a, int n);

// ------------------------------------------------------------------ gemm.cu
enum { EPI_STORE = 0, EPI_BIAS_ACT = 1, EPI_MASK_POS = 2, EPI_CDAE_LOSS = 3 };
enum { LAYOUT_KK = 0,   // A[m][k] k-contiguous, B[n][k] k-contiguous      (C = A * B^T)
       LAYOUT_MN = 1,   // A[k][m] m-contiguous, B[k][n] n-contiguous      (C = A^T * B)
       LAYOUT_KN = 2 }; // A[m][k] k-contiguous, B[k][n] n-contiguous      (C = A * B)
struct GemmArgs {
  const float* A; const float* B; float* C;
  int M, N, Kred; int lda, ldb, ldc;
  int splits;                         // split the reduction range; partial s is written at C + s * M * ldc
  // epilogue
  const float* bias;                  // [N]  (EPI_BIAS_ACT, EPI_CDAE_LOSS)
  int act;                            // EPI_BIAS_ACT
  const float* mask;                  // [M, ldc] (EPI_MASK_POS: C = acc * (mask > 0))
  // EPI_CDAE_LOSS: C receives dL/dz2
  const float* label_count;           // [N] batch histogram (batch_mean) or NULL
  const uint32_t* label_bits; int words_per_row;   // per_user labels or NULL
  int loss_kind; float inv_count; int batch;
  float* loss_part;                   // [grid blocks]
  float* col_part;                    // [m tiles, ldc] column partial sums of C
};
int launch_gemm(drb_ctx* ctx, int layout, int epi, const GemmArgs& a, int* n_mtiles_out = nullptr,
                int* n_blocks_out = nullptr);

// ------------------------------------------------------------------ umma.cu (tcgen05 / TMA / TMEM path)
struct UmmaOperands {
  const void* a_hi; const void* a_lo; int lda;      // K-major: A[m][k]; MN-major (tf32 only): G[k][m]; pitch in elements
  const void* b_hi; const void* b_lo; int ldb;      // B[n][k], k contiguous
  int b_rows;                                       // rows of B that exist in memory (>= logical N is fine)
  int a_tiled_nib = 0;                              // > 0: A is dz in a tile-major layout: 128-row tiles of 32 floats
                                                    // (tf32, umma_loss.cu) or 64 halfs (fp16), nib column blocks per row tile
  int64_t a_tiled_rows = 0;                         //      total rows of the [rows, 32 | 64] view
  bool half = false;                                // operands are fp16 hi / lo pairs (kind::f16) instead of tf32 hi / lo
  float out_scale = 1.f;                            // accumulators are multiplied by out_scale * (*out_scale_dev)
  const float* out_scale_dev = nullptr;             //   (undoes the per-tensor power-of-two scaling of fp16 operands)
  const char* name = nullptr;                       // profiling name of the launch (drb_ctx_profile_read)
};
bool umma_available();
// src [rows][ld] -> tf32 hi / lo split, optionally also transposed ([cols..][ldt]); ones_row >= 0 sets that
// transposed row to 1 (constant feature used to fold the output-bias gradient into the dW' GEMM)
int launch_split_tf32(drb_ctx* ctx, const float* src, int rows, int cols, int ld, float* hi, float* lo, float* t_hi,
                      float* t_lo, int ldt, int ones_row);
// fp16 form: x * alpha * (*alpha_dev) -> hi = rn_f16(.), lo = rn_f16(. - hi); hi / lo [rows][ldh halfs] (may be NULL),
// transposed t_hi / t_lo [cols..][ldt halfs] (may be NULL).  alpha_dev may be NULL.  ones_row: that transposed row = alpha.
int launch_split_f16(drb_ctx* ctx, const float* src, int rows, int cols, int ld, float alpha, const float* alpha_dev,
                     void* hi, void* lo, int ldh, void* t_hi, void* t_lo, int ldt, int ones_row);
// scales[0] = alpha = 2^(14 - floor(log2(max |x|))) (so that max |x| * alpha is in [2^14, 2^15)), scales[1] = 1 / alpha;
// x [rows][ld], the first `cols` columns.  Two tiny launches (reduce, then publish).
int launch_absmax_scale(drb_ctx* ctx, const float* x, int64_t rows, int cols, int ld, float* scales);
// dz_hi / dz_lo are written in the tile-major layout: tile (row tile rt, column block cb) of 128 x 32 floats at
// float offset ((rt * nib + cb) * 128) * 32, nib = drb_dz_nib(N)
inline int drb_dz_nib(int n_cols) { return 4 * ((n_cols + 127) / 128); }
// fp16 dz: two tile-major copies, tiles of 128 rows x 64 halfs (16 KB): U = [user tile][item block] feeds dh = dz W'^T,
// I = [item tile][user block] feeds dW'^T = dz^T h; hi and lo of one copy share one buffer of drb_dz_tiled_floats floats
inline int drb_dz_nib64(int n_cols) { return 2 * ((n_cols + 127) / 128); }
struct DzHalf {
  void* u_hi; void* u_lo; int nib64;      // [ceil(B/128)][nib64] tiles
  void* i_hi; void* i_lo; int nub;        // [ceil(I/128)][nub] tiles, nub = 2 * ceil(B/128)
  int row_tiles, item_tiles;
};
inline int64_t drb_dz_tiled_floats(int rows, int n_cols) { return (int64_t)((rows + 127) / 128) * drb_dz_nib(n_cols) * 4096; }
int launch_umma_cdae_loss(drb_ctx* ctx, const UmmaOperands& o, int M, int N, int Kred, float* dz_hi, float* dz_lo,
                          int ldc, const float* bias, const float* label_count, const uint32_t* label_bits,
                          int words_per_row, int loss_kind, float inv_count, int batch, float* loss_part,
                          float* dz_colsum /* may be NULL: [N] += colsum(dz), i.e. db' */, int* n_blocks_out,
                          float* z_dbg = nullptr /* tests: logits as formed by the kernel, [M][ldz] */, int ldz = 0,
                          const DzHalf* dzh = nullptr /* o.half: dz goes here (fp16 hi/lo, scaled by 2^14 / inv_count) */);
constexpr float DRB_DZ_F16_SCALE = 16384.0f;   // |dL/dz2| / inv_count <= 1 -> scaled into [-2^14, 2^14]
constexpr float DRB_H_F16_SCALE = 32768.0f;    // h in (0, 1)
int launch_umma_store(drb_ctx* ctx, const UmmaOperands& o, bool a_mn_major, int M, int N, int Kred, int splits,
                      float* C, int ldc, int n_store, int n_valid, float* extra_col, int extra_col_index,
                      bool atomic_out = false);

// ------------------------------------------------------------------ optim.cu
#define DRB_MAX_SEGS 40
struct AdamSeg { int64_t off4, n4; float alpha, l2, regw; int alpha_idx; };
struct AdamArgs {
  float* w; float* m; float* v; const float* g;
  AdamSeg seg[DRB_MAX_SEGS]; int nseg;
  float beta1, beta2, eps;
  float* reg_part;                    // [blocks] partial sums of regw * w^2 (pre-update weights)
  const float* alpha_dev;             // may be NULL; else alpha of segment s = alpha_dev[seg[s].alpha_idx] (graph replay:
                                      // the step sizes are the only scalars of a step that change from step to step)
  // optional fused loss finalisation by the last block to finish (saves a launch on the latency-bound small shapes):
  // fin_loss_out[0] = sum(fin_loss_part) * fin_scale + sum(reg_part[0 .. fin_n_reg)), [1] = the batch term alone.
  // fin_n_reg == 0 means "the blocks of this launch".  fin_ticket: a zero-initialised device counter (self resetting).
  // fin_reg_part: start of the partials to sum (NULL = reg_part).
  const float* fin_loss_part; int fin_n_loss; float fin_scale; int fin_n_reg; const float* fin_reg_part;
  float* fin_loss_out; unsigned int* fin_ticket;
  // optional: segment `row_seg` is a [rows, 4 * row_len4] table whose gradient is zero except in the rows whose bit is
  // set in row_mask (the user table of CDAE: only the sampled users' rows): the gradient of the other rows is not read
  const uint32_t* row_mask = nullptr; int row_seg = -1; int row_len4 = 0;
};
// dst[i] = vals[i], i < n <= 8 (one tiny launch; the values travel as kernel arguments)
int launch_set_scalars(drb_ctx* ctx, float* dst, const float* vals, int n);
int launch_adam(drb_ctx* ctx, const AdamArgs& a, int* n_blocks_out);
// loss_out = sum(loss_part) * scale + sum(reg_part)
int launch_finalize_loss(drb_ctx* ctx, const float* loss_part, int n_loss, float scale, const float* reg_part,
                         int n_reg, float* loss_out);
float drb_adam_alpha(float lr, float beta1, float beta2, int t);

// ------------------------------------------------------------------ dmf.cu
// cosine head: p = max(1e-6, <a/|a|, e/|e|>), BCE vs label, backward through the normalisation and the last relu.
struct DmfHeadArgs {
  const float* a; const float* e; int ld; int width;    // last tower activations [n, ld]
  const float* labels;                                    // may be NULL (forward only)
  float* p_out;                                           // may be NULL
  float* da; float* de;                                   // may be NULL; d(pre-activation) of the last layers
  float* loss_part;                                       // [n] per-pair loss terms
  int n;
  int n_global;                                           // data parallel: pairs over all ranks (0 = n), the 1/B of the loss
};
int launch_dmf_head(drb_ctx* ctx, const DmfHeadArgs& a);
// dense part of the backward pass of a two-layer tower (Dense(w0, relu) -> Dense(w1, relu)), both towers in one launch:
//   dpre0 = (dpre1 K1^T) * [act0 > 0],  dK1 += act0^T dpre1,  db1 += colsum(dpre1),  db0 += colsum(dpre0)
// (gradient buffers pre-zeroed; partial sums per CTA, then atomics)
struct DmfTowerBwd {
  const float* act0; const float* dpre1; const float* k1;   // [n, ld0], [n, ld1], [w0 x ld1]
  float* dpre0;                                              // [n, ld0]
  float* g_k1; float* g_b1; float* g_b0;                     // gradients: [w0 x ld1], [ld1], [ld0]
  int w0, ld0, w1, ld1;
};
int launch_dmf_tower_bwd(drb_ctx* ctx, const DmfTowerBwd& t0, const DmfTowerBwd& t1, int n);
bool dmf_tower_bwd_fits(int w0, int ld0, int w1);

// ------------------------------------------------------------------ score.cu
struct CandScoreArgs {
  const float* urep; int ld_u;            // [n, ld] user representation (CDAE: h, DMF: user tower output)
  const float* table; int ld_t;           // [n_items, ld] item representation (CDAE: W2T, DMF: item tower out)
  const float* bias;                      // CDAE b2 or NULL
  int width; int mode;                    // mode 0: sigmoid(dot + bias) (CDAE); 1: max(1e-6, cosine) (DMF)
  const int32_t* uids;                    // [n]
  const int32_t* cand; const int32_t* cand_count; int max_cand;
  const int64_t* seen_indptr; const int32_t* seen_indices; int novelty;
  int32_t* out_iid; float* out_score; int32_t* n_out;     // [n, max_cand], [n]
};
// max_cand <= 4096: keys sorted in shared memory.  Longer lists (up to the whole catalog) sort in `scratch`
// (next_pow2(max_cand) 64-bit keys per user); rank_scratch_rows = users one call can take with that much scratch
int launch_rank_candidates(drb_ctx* ctx, const CandScoreArgs& a, int n, void* scratch = nullptr, int64_t scratch_bytes = 0);
int64_t rank_scratch_rows(int64_t scratch_bytes, int max_cand);

struct TopkArgs {
  const float* scores; int ld; int n_items;   // [n, ld]
  const int32_t* uids; const int64_t* seen_indptr; const int32_t* seen_indices; int novelty;
  int k; int32_t* out_iid; float* out_score; int32_t* n_out;
  // indirect form (exact fallback of the tensor-core top-k): block b ranks row b for user fb_users[b], b < *fb_count
  const int32_t* fb_users = nullptr; const int32_t* fb_count = nullptr; int fb_max = 0;
};
int launch_topk(drb_ctx* ctx, const TopkArgs& a, int n);
// tensor-core top-k (umma_score.cu + score.cu): filter pass over an item range, list selection, exact fallback
int launch_umma_score_filter(drb_ctx* ctx, const UmmaOperands& o, int n_users, int n_items, int item_begin, int item_end,
                             int Kred, const float* bias, const uint32_t* seen_bits, int words_per_row,
                             const uint32_t* tau_ord, const float* tau_z, int32_t* cnt, uint64_t* lists, int cap);
int launch_select_lists(drb_ctx* ctx, uint64_t* lists, int cap, int32_t* cnt, uint32_t* tau_ord, float* tau_z, int k, bool final,
                        int32_t* out_iid, float* out_score, int32_t* n_out, int32_t* fb_users, int32_t* fb_count, int fb_max,
                        int32_t* big_users, int32_t* big_count, int n);
// users with n_out == -1: scores by fp32 FMA into `rows` ([fb_max][a.ld]), then the radix-select top-k on those rows
int launch_topk_fallback(drb_ctx* ctx, const TopkArgs& a, int n, const float* h, int ld_h, const float* table, int ld_t,
                         const float* bias, int width, float* rows, int32_t* fb_users, int32_t* fb_count, int fb_max);

// ------------------------------------------------------------------ dmf_topk.cu (DMF full-catalog top-k, FFMA scores)
// vectors are zero-padded to 32 * dmf_topk_nj(width) components (1, 2, 4, 8 or 16 groups of 32)
int dmf_topk_nj(int width);
// irep [n_items][ld_i] -> irep_t [32 nj][i_pad] (k-major, zero-padded) and item_inv [i_pad] = 1 / |t| as the rank path
// forms it (0 past n_items); i_pad a multiple of 128
int launch_dmf_topk_prep(drb_ctx* ctx, const float* irep, int ld_i, int width, int n_items, int i_pad, float* irep_t,
                         float* item_inv);
struct DmfFilterArgs {
  const float* urep; int ld_u; int n_users;       // [n_users][ld_u] user tower output of the block
  const float* irep_t; const float* item_inv; int i_pad;   // from launch_dmf_topk_prep
  int width;
  int item_lo, item_hi;                           // item range of this pass (item_lo % 128 == 0)
  const uint32_t* seen_bits; int words_per_row;   // NULL (no novelty filter) or [n_users][words_per_row]
  const uint32_t* tau_ord;                        // [n_users] a key is listed when its orderable score is > tau
  int32_t* cnt; uint64_t* lists; int cap;         // [n_users], [n_users][cap] (cnt may exceed cap: overflow)
};
int launch_dmf_topk_filter(drb_ctx* ctx, const DmfFilterArgs& a);
// users with n_out == -1 (claimed by the final select): exact scores into `rows` ([fb_max][a.ld]), then k_topk on them
int launch_dmf_topk_fallback(drb_ctx* ctx, const TopkArgs& a, int n, const float* urep, int ld_u, const float* irep,
                             int ld_i, int width, float* rows, int32_t* fb_users, int32_t* fb_count, int fb_max);

#endif
