/* coda_b200 -- C ABI of the B200-native CODA acquisition hot path.
 *
 * Drop-in boundary (SURVEY.md 8b).  The reference (justinkay/coda) is pure Python/PyTorch
 * and has no FFI of its own; these entry points are what a ctypes binding inside
 * coda/coda.py would call in place of the ATen op chains on the acquisition path.  Each
 * declaration cites the reference lines it replaces (paths relative to the reference root).
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless the name ends in _host or the comment says "host struct";
 *   - `stream` is a cudaStream_t passed as void*; all work is enqueued, nothing synchronises;
 *   - return value: CODA_B200_OK or a negative error code, message via coda_b200_last_error();
 *   - numerical problems are reported through a device-side `flags` word (bits below) that the
 *     caller reads at its next host sync -- the reference raises RuntimeError('[NUMERIC ERROR]')
 *     from coda/util.py:17-25 at the same places;
 *   - layouts: preds [H][N][C] fp32 (coda/datasets.py:14), models `model_stride` floats apart (N*C when the
 *     shard is its own tensor; the full-task stride when it is an N-range view of a bigger slab);
 *   - 16-bit slabs: every entry point that reads preds has an `_f16` twin taking `const uint16_t* preds`, the IEEE
 *     binary16 bit patterns of the scores in the same layout (strides in elements).  The twins convert on load and
 *     compute in fp32: their results have the bits of the fp32 entry point on the upcast slab, and they choose
 *     between kernels exactly as the fp32 entry point does for the same shape and view;
 *     D (dirichlets) [H][C][C] fp32; U (un-normalised pi_hat_xi) [N][C] fp32; hard [N][H] u16;
 *     Hp = H rounded up to 32;
 *   - "rows": one row = one hypothetical (item, class) update.  Rows [0, T), T = C*(1+H), are the template rows
 *     (class-major: c*(1+H) + 0 = no model predicts c, + 1 + h = only model h predicts c); rows [T, T + n_heavy) are
 *     the heavy rows (two or more models predict the class), ITEM-major: the heavy rows of item n are
 *     T + heavy_off[n] .. T + heavy_off[n+1] - 1 in ascending class order;
 *   - built for sm_100a only.
 */
#ifndef CODA_B200_H
#define CODA_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CODA_B200_VERSION 202
#define CODA_B200_NODES 256 /* quadrature nodes, coda/coda.py:79 */
#define CODA_B200_MAX_WORLD 16
#define CODA_B200_REC_WORDS 8 /* arg-max record: {bits vA, iA, cntA, bits vB, iB, bits v2A, bits v2B, 0} */

#define CODA_B200_OK 0
#define CODA_B200_EINVAL (-1)
#define CODA_B200_ECUDA (-2)

/* device-side flag bits */
#define CODA_B200_FLAG_NONFINITE_INPUT 0x01u /* NaN/Inf in preds */
#define CODA_B200_FLAG_RANGE_INPUT 0x02u     /* preds outside [0, 1]: not post-softmax scores */
#define CODA_B200_FLAG_NONFINITE_TABLE 0x04u /* util._check(pdf/cdf/integrand), coda.py:96-112 */
#define CODA_B200_FLAG_NONFINITE_PI 0x08u    /* pi_hat_xi row sum not finite */
#define CODA_B200_FLAG_NONFINITE_PBEST 0x10u /* util._check(pbest), coda.py:330 */
#define CODA_B200_FLAG_NONFINITE_EIG 0x20u   /* util._check(Pbest(beta) normalized), coda.py:115 */
#define CODA_B200_FLAG_NO_CANDIDATE 0x40u    /* the host-free loop ran out of unlabeled items */
#define CODA_B200_FLAG_XCHG_TIMEOUT 0x80u    /* a peer never arrived at an exchange (2 s) */
#define CODA_B200_FLAG_NEGATIVE_PROB 0x100u  /* util._check_prob: probability < -1e-12 (util.py:33-35) */
#define CODA_B200_FLAG_ROWSUM_WARN 0x200u    /* util._check_prob: |row sum - 1| > 1e-4 (util.py:37-39), a warning */
#define CODA_B200_FLAG_PIPELINE_TIMEOUT 0x400u /* a TMA / tensor-core pipeline stopped (pi_full_tc); the result is invalid */

typedef void* coda_stream_t;

/* ---- plumbing ---------------------------------------------------------------------- */
const char* coda_b200_last_error(void);
int coda_b200_version(void);
int coda_b200_sm_count(void);
int coda_b200_device_check(void); /* fails loudly when no sm_100 device is present */
/* cudaLimitMaxL2FetchGranularity hint (32/64/128 B) for the sector-gather kernels (per device). */
int coda_b200_set_l2_fetch_granularity(int bytes);

/* ---- N-axis shards: peer-memory exchange (SURVEY.md 8e; no reference counterpart) ------------------
 * Every shard owns a mailbox in its own HBM.  The two per-step exchanges (arg-max record, marginal sums) are
 * done INSIDE the step kernels: a rank stores its contribution straight into every peer's mailbox over
 * NVLink (P2P stores), releases a flag with system scope, and spins on its own mailbox until every peer's
 * contribution of the same epoch has landed.  Slots are double-buffered by epoch parity.  The mailbox is
 * reached through CUDA IPC (one process per GPU, torchrun) or plain peer access (one process driving all GPUs). */
typedef struct coda_xchg { /* host struct */
  int world, rank;
  void* box[CODA_B200_MAX_WORLD]; /* mailbox of every rank as addressable from THIS rank's device; box[rank] is local */
  uint64_t* epoch;                /* local, [8], zero-initialised: per-channel epoch counters [0..4) and the nanoseconds
                                     spent waiting for peers per channel [4..8) (latency + skew; bench.py prints them) */
  int H, C, rep_words;            /* fix the slot sizes (same on every rank); rep_words: int64 words of a report block */
} coda_xchg_t;
size_t coda_b200_xchg_box_bytes(int world, int H, int C, int rep_words);
int coda_b200_xchg_alloc(size_t bytes, void** box_out); /* cudaMalloc + zero fill on the current device */
int coda_b200_xchg_free(void* box);
int coda_b200_ipc_export(const void* box, void* handle64_host);
int coda_b200_ipc_open(const void* handle64_host, void** box_out);
int coda_b200_ipc_close(void* box);
int coda_b200_peer_enable(int peer_device); /* current device may load/store peer_device's memory */

/* ---- construction (coda/coda.py:172-203) --------------------------------------------- */

/* One pass over the slab: per-model argmax (coda.py:217, 263, 316), ensemble-mean pseudo
 * label (coda/util.py:13-14 + coda.py:193-194), unanimity bit (coda.py:215-219).
 * ens_out (optional) [N][C]: E[n][c] = sum_h preds[h][n][c], the un-normalised ensemble of coda/util.py:13-14.
 * Also util._check_prob (util.py:28-39) on the input: negatives, non-finite values, row sums. */
int coda_b200_scan_slab(const float* preds, int64_t model_stride, int H, int64_t N, int C, uint16_t* hard,
                        int32_t* pseudo, uint8_t* disagree, float* ens_out, uint32_t* flags, coda_stream_t stream);
int coda_b200_scan_slab_f16(const uint16_t* preds, int64_t model_stride, int H, int64_t N, int C, uint16_t* hard,
                            int32_t* pseudo, uint8_t* disagree, float* ens_out, uint32_t* flags, coda_stream_t stream);

/* Soft confusion sums, coda.py:42 einsum('nc,hnj->hcj').  conf_fx [H][C][C] int64 fixed point
 * (value * 2^fx_shift), ACCUMULATED into; exact and order-independent so shards can be summed. */
int coda_b200_confusion_accum(const float* preds, int64_t model_stride, const int32_t* pseudo, int H, int64_t N,
                              int C, int fx_shift, int64_t* conf_fx, coda_stream_t stream);
int coda_b200_confusion_accum_f16(const uint16_t* preds, int64_t model_stride, const int32_t* pseudo, int H, int64_t N,
                                  int C, int fx_shift, int64_t* conf_fx, coda_stream_t stream);

/* Same sums with the items visited in pseudo-label order (`order` = any permutation that groups equal
 * pseudo labels; C <= 128): register accumulation, no shared-memory atomics.  Bit-identical result. */
int coda_b200_confusion_sorted(const float* preds, int64_t model_stride, const int32_t* pseudo,
                               const int32_t* order, int H, int64_t N, int C, int fx_shift, int64_t* conf_fx,
                               coda_stream_t stream);
int coda_b200_confusion_sorted_f16(const uint16_t* preds, int64_t model_stride, const int32_t* pseudo,
                                   const int32_t* order, int H, int64_t N, int C, int fx_shift, int64_t* conf_fx,
                                   coda_stream_t stream);

/* Row-normalise (coda.py:43) and build the Dirichlet prior (coda.py:46-63, 196). */
/* conf_rest (optional, compact slab): [H][C] sums every column of row (h, c) carries in addition (see below). */
int coda_b200_init_dirichlets(const int64_t* conf_fx, const int64_t* conf_rest, int H, int C, int fx_shift,
                              double prior_strength, double multiplier, int uniform_prior, float* D,
                              coda_stream_t stream);

/* ---- consensus marginals (CODA.update_pi_hat, coda.py:226-233) ------------------------ */

/* U[n][c] = sum_h sum_s D[h][c][s] preds[h][n][s]  (coda.py:227-229, `adjusted` never stored). */
int coda_b200_pi_full(const float* preds, int64_t model_stride, const float* D, int H, int64_t N, int C, float* U,
                      coda_stream_t stream);
int coda_b200_pi_full_f16(const uint16_t* preds, int64_t model_stride, const float* D, int H, int64_t N, int C, float* U,
                          coda_stream_t stream);

/* The same contraction on the tensor cores (tcgen05, TMEM accumulators, bulk-TMA slab stream): both operands are cut
 * into two bf16 limbs, 4 MMAs per K = 16 chunk, accumulators drained to fp32 registers every 4 models (pi_tc.cu).
 * Usable when pi_full_tc_ok(...) != 0 (16 <= C <= 128, C % 4 == 0, model_stride % 4 == 0); `scratch` =
 * pi_full_tc_scratch_bytes(H, C) bytes (the D limbs).  A stopped pipeline sets CODA_B200_FLAG_PIPELINE_TIMEOUT. */
int coda_b200_pi_full_tc_ok(int H, int64_t N, int C, int64_t model_stride);
size_t coda_b200_pi_full_tc_scratch_bytes(int H, int C);
int coda_b200_pi_full_tc(const float* preds, int64_t model_stride, const float* D, int H, int64_t N, int C, float* U,
                         void* scratch, uint32_t* flags, coda_stream_t stream);
/* fp16: eligible for exactly the shapes of the fp32 pass; preds needs 8-byte alignment (fp32: 16). */
int coda_b200_pi_full_tc_ok_f16(int H, int64_t N, int C, int64_t model_stride);
int coda_b200_pi_full_tc_f16(const uint16_t* preds, int64_t model_stride, const float* D, int H, int64_t N, int C,
                             float* U, void* scratch, uint32_t* flags, coda_stream_t stream);

/* Row-normalise with the 1e-12 clamp (coda.py:230) and accumulate sum_n pi_hat_xi[n][:]
 * (coda.py:232) into pisum_fx [C] (int64 fixed point, ACCUMULATED).  xi_out may be NULL. */
int coda_b200_pi_reduce(float* U, int64_t N, int C, int fx_shift, float* xi_out, int64_t* pisum_fx, uint32_t* flags,
                        coda_stream_t stream);

/* Optional class-major shadow copy T[s][c][n] = preds[model_of_slot[s]][n][c] for S of the H models (no
 * reference counterpart: a layout for the one-float-per-(model, item) gather of the rank-1 refresh).
 * Columns are `col_stride` floats apart (>= N, a multiple of 4 so that every column is 16-byte aligned). */
int coda_b200_shadow_build(const float* preds, int64_t model_stride, int H, int64_t N, int C,
                           const int32_t* model_of_slot, int S, int64_t col_stride, float* T, coda_stream_t stream);
/* fp16 shadow of an fp16 slab: col_stride a multiple of 8 (16-byte aligned columns); the step kernels' shadow_off
 * counts slab ELEMENTS (halves) from preds to T. */
int coda_b200_shadow_build_f16(const uint16_t* preds, int64_t model_stride, int H, int64_t N, int C,
                               const int32_t* model_of_slot, int S, int64_t col_stride, uint16_t* T,
                               coda_stream_t stream);

/* update_pi_hat after the rank-1 change of D (coda.py:319): U[n][t] += lr * sum_h preds[h][n][jvec[h]],
 * then the same normalise + column sums as pi_reduce.  The gather list (`terms`, written by the step kernels
 * below) is {nterms, majority class t' or -1} followed by nterms x {element offset, sign, item stride}: with the
 * ensemble sums E the sum over models is taken as E[n][t'] + corrections for the models that disagree with the
 * majority class t' of jvec (exact algebra, fewer gathers); models with a shadow slot are read from the shadow.
 * pisum_fx was zeroed by the step kernel and is accumulated into (this shard's sums).  ctas_per_sm (1..8)
 * bounds the grid so a concurrent stream keeps SM resources.  U must be 16-byte aligned and followed by 16
 * readable bytes (C <= 128 takes a bulk-TMA pipeline that rounds the last tile's copy up). */
/* const_slot: >= 0 = the caller owns that slot of the per-device constant-memory term table (slots hold 2H terms
 * rounded up to 64; floor(3584 / that) slots exist; no two streams of one process may use the same slot of the same
 * device concurrently) -- the gather list is then read through the constant cache; -1 = shared-memory copy. */
int coda_b200_pi_rank1(const float* preds, const float* ens, int H, int64_t N, int C, const int64_t* sel, double lr,
                       int fx_shift, const int32_t* terms, float* U, int64_t* pisum_fx, uint32_t* flags,
                       int ctas_per_sm, int const_slot, coda_stream_t stream);
/* fp16 slab (and shadow): the gather list holds element offsets from preds.  The opt-in variants that read the slab as
 * fp32 words (CODA_B200_R1=tma|v4) return CODA_B200_EINVAL; v1 (default) and v1d are available. */
int coda_b200_pi_rank1_f16(const uint16_t* preds, const float* ens, int H, int64_t N, int C, const int64_t* sel,
                           double lr, int fx_shift, const int32_t* terms, float* U, int64_t* pisum_fx, uint32_t* flags,
                           int ctas_per_sm, int const_slot, coda_stream_t stream);

/* ---- compact slab (BASELINE.json configs[4]: M=1024, N=4e6, C=1000 is 16.4 TB dense; no reference counterpart --
 *      the reference cannot run there, coda.py:227 materialises a second slab) ----------------------------------
 * For every (h, n) the K <= 8 highest-scoring classes: ids [H][N][K] u16 (descending score) and probs [H][N][K] f32;
 * every other class gets rest = (1 - sum_j probs) / (C - K).  Models are model_stride ELEMENTS apart in both
 * arrays.  Each stage below produces what its dense twin produces on the densified slab. */
int coda_b200_scan_compact(const uint16_t* ids, const float* probs, int64_t model_stride, int H, int64_t N, int C,
                           int K, uint16_t* hard, int32_t* pseudo, uint8_t* disagree, float* ens_out, uint32_t* flags,
                           coda_stream_t stream);
/* coda.py:42: conf[h][y][j] == conf_fx[h][y][j] + conf_rest[h][y] (both ACCUMULATED into, int64 fixed point). */
int coda_b200_confusion_compact(const uint16_t* ids, const float* probs, int64_t model_stride, const int32_t* pseudo,
                                int H, int64_t N, int C, int K, int fx_shift, int64_t* conf_fx, int64_t* conf_rest,
                                coda_stream_t stream);
/* coda.py:227-229.  DT_scratch [H][C][C] and RS_scratch [H][C] floats are overwritten (D transposed, row sums). */
int coda_b200_pi_full_compact(const uint16_t* ids, const float* probs, int64_t model_stride, const float* D, int H,
                              int64_t N, int C, int K, float* DT_scratch, float* RS_scratch, float* U,
                              coda_stream_t stream);
/* coda.py:319 (see coda_b200_pi_rank1); the gather list was built with coda_step_t.compact_k = K. */
int coda_b200_pi_rank1_compact(const uint16_t* ids, const float* probs, int64_t model_stride, const float* ens, int H,
                               int64_t N, int C, int K, const int64_t* sel, double lr, int fx_shift,
                               const int32_t* terms, float* U, int64_t* pisum_fx, uint32_t* flags,
                               coda_stream_t stream);

/* Inverted index of the compact slab: for every (model, class) the items whose top-K list holds the class, as
 * {item u32, float bits of (probs - rest)} pairs.  count: counts[h][c] (ACCUMULATED into, int64); the caller turns
 * them into offsets [H*C + 1] (exclusive prefix sums) and a cursor copy; fill: places the 8-byte entries (order
 * inside a list is not defined) and writes rest_sum[n] = sum_h rest(h, n).  N < 2^32 per shard. */
int coda_b200_compact_index_count(const uint16_t* ids, int64_t model_stride, int H, int64_t N, int C, int K,
                                  int64_t* counts, coda_stream_t stream);
int coda_b200_compact_index_fill(const uint16_t* ids, const float* probs, int64_t model_stride, int H, int64_t N, int C,
                                 int K, int64_t* cursor, void* entries, float* rest_sum, coda_stream_t stream);
/* coda.py:319 from the index:  sum_h preds[h][n][jvec[h]] = rest_sum[n] + sum over the H lists (h, jvec[h]) of
 * (probs - rest), scattered into delta [N] (int64 fixed point, zero on entry and on exit: order-independent sums),
 * then the U row pass of coda_b200_pi_rank1.  Reads H lists of about N K / C entries instead of the whole slab.
 * `terms` is only consulted for "no label applied in this step" ({0, -1}). */
int coda_b200_pi_rank1_index(const int64_t* offsets, const void* entries, const float* rest_sum, const int32_t* jvec,
                             int H, int64_t N, int C, const int64_t* sel, double lr, int fx_shift, const int32_t* terms,
                             int64_t* delta, float* U, int64_t* pisum_fx, uint32_t* flags, coda_stream_t stream);

/* ---- Beta quadrature tables (dirichlet_to_beta coda.py:14-25, compute_pbest_beta_batched
 *      coda.py:77-119, batch_update_beta coda.py:150-168) for classes [cls_lo, cls_hi) ------- */
size_t coda_b200_tables_scratch_bytes(int H, int ncls);
/* sel (optional, device): {idx, class}; when non-NULL exactly one class, sel[1], is rebuilt (host-free loop). */
/* dLb / Gb (optional, both or neither): the same tables as bf16 limbs in tensor-core operand order for
 * coda_b200_pair_rows_tc: dLb [C][Hp/32][3][256*32], Gb [C][16][4][Hp*16] bf16, zero-initialised by the caller. */
int coda_b200_beta_tables(const float* D, const float* grid_x, int H, int C, int P, double hyp_w, int cls_lo,
                          int cls_hi, const int64_t* sel, void* scratch, float* dL /*[C][H][P]*/,
                          float* G0T /*[C][P][Hp]*/, float* G1T /*[C][P][Hp]*/, float* PB /*[C][Hp]*/, void* dLb,
                          void* Gb, uint32_t* flags, coda_stream_t stream);

/* ---- hypothetical-update rows (eig_batched inner loop, coda.py:261-279) ---------------- */
/* ent_cnt[n] = distinct predicted classes of item n, heavy_cnt[n] = how many of them two or more models predict,
 * cls_heavy[c] (accumulated) = heavy rows of class c. */
int coda_b200_pair_count(const uint16_t* hard, int H, int64_t N, int C, int32_t* ent_cnt /*[N]*/,
                         int32_t* heavy_cnt /*[N]*/, int32_t* cls_heavy /*[C]*/, coda_stream_t stream);
/* Fills, per item, the entry list (ent_row / ent_cls at ent_off[n]..) and, per class, the class-major work list the
 * row kernels tile over: position q in [cls_base[c], cls_base[c+1]) = {template rows of c, heavy rows of c} with
 * zmask[q] (H-bit set of the models that predict c) and row_of[q] (the row it describes). */
int coda_b200_pair_fill(const uint16_t* hard, int H, int64_t N, int C, const int32_t* ent_off /*[N+1]*/,
                        const int32_t* heavy_off /*[N+1]*/, const int64_t* cls_base /*[C+1]*/,
                        int32_t* cls_cursor /*[C] zeroed*/, int32_t* ent_row, uint16_t* ent_cls,
                        uint32_t* zmask /*[npairs][Hp/32]*/, int32_t* row_of /*[npairs]*/,
                        uint16_t* row_cls /*[n_heavy] class of every heavy row*/, coda_stream_t stream);
/* tiles [ntiles][4] int32 = {class, first work-list position, count <= 32, 0}; processes tiles [tile_lo, tile_hi).
 * Writes gain[row] = H_before - H_after (coda.py:274-276) and, if ph_cache != NULL, the normalised
 * P(best | hypothetical) row (coda.py:271-273), row = row_of[position].  With sel != NULL the launch covers
 * [0, tile_hi - tile_lo) tiles of class sel[1] (pass the largest per-class tile count). */
int coda_b200_pair_rows(const int32_t* tiles, int tile_lo, int tile_hi, const uint32_t* zmask, const int32_t* row_of,
                        const float* dL, const float* G0T, const float* G1T, const float* PB, const float* m0,
                        const float* pi_hat, int H, float* ph_cache, float* gain, const int64_t* sel /*optional*/,
                        const int64_t* tile_off /*[C+1], with sel*/, uint32_t* flags, coda_stream_t stream);
/* The same computation on the tcgen05 tensor cores (Hp <= 256): tiles128 are tiles of <= 128 same-class positions,
 * operands come from the bf16 limb tables of coda_b200_beta_tables. */
int coda_b200_pair_rows_tc(const int32_t* tiles128, int tile_lo, int tile_hi, const uint32_t* zmask,
                           const int32_t* row_of, const void* dLb, const void* Gb, const float* PB, const float* m0,
                           const float* pi_hat, int H, float* ph_cache, float* gain, const int64_t* sel,
                           const int64_t* tile_off, uint32_t* flags, coda_stream_t stream);
/* gain[r] (coda.py:274-276) of the T = C*(1+H) template rows from their cached P(best | hypothetical) rows. */
int coda_b200_template_gains(const float* ph_cache, int H, int C, const float* PB, const float* m0,
                             const float* pi_hat, float* gain /*[T]*/, coda_stream_t stream);

/* ---- the per-step scoring pass (eig_batched coda.py:253-278 + _prefilter coda.py:215-219 + the arg-max of
 *      get_next_item_to_label coda.py:306/309), one kernel, item-major ---------------------------------
 * For every item: information gain of each of its heavy rows straight from the cached row (ph_cache != NULL) or
 * from gain[row] (ph_cache == NULL: the row kernels just wrote it), template gains from gain[0..T), then
 * eig[n] = sum_c pi_hat_xi[n][c] * gain(n, c)  (== H_before - sum_c xi * H_after because sum_c xi = 1), the
 * candidate arg-max (first index wins) and runner-up value per block -> partials [blocks][REC_WORDS]. */
int coda_b200_eig_blocks(int64_t N, int H, int C); /* number of partial records gain_eig writes */
/* max_entries: the longest entry list (or -1 if unknown); short lists and C <= 128 take an 8-lanes-per-item kernel,
 * which reads the lists from the optional ELL copy (coda_b200_ell_build; ell_k = padded list length <= 32). */
int coda_b200_gain_eig(const float* U, int64_t N, int C, int H, const int32_t* ent_off, const int32_t* heavy_off,
                       const int32_t* ent_row, const uint16_t* ent_cls, const float* ph_cache, const float* gain,
                       const float* PB, const float* m0, const float* pi_hat, const uint8_t* labeled,
                       const uint8_t* disagree, int64_t n_offset, int max_entries, const int32_t* ell_row,
                       const uint16_t* ell_cls, int ell_k, float* eig, int64_t* partials, uint32_t* flags,
                       coda_stream_t stream);
int coda_b200_ell_build(const int32_t* ent_off, const int32_t* ent_row, const uint16_t* ent_cls, int64_t N, int K,
                        int32_t* ell_row /*[N][K], -1 = empty*/, uint16_t* ell_cls /*[N][K]*/, coda_stream_t stream);
/* gain[r] (coda.py:274-276) of ALL T + n_heavy rows from their cached rows -- the template rows (class = r / (1+H))
 * and the heavy rows (class = row_cls[r - T]) in one stream: the HBM-bound kernel of the two-kernel scoring pass
 * (row_gains, then gain_eig with ph_cache == NULL).  Item-major heavy rows make the per-item gains contiguous for the
 * assembly that follows. */
int coda_b200_row_gains(const float* ph_cache, const uint16_t* row_cls, int64_t n_heavy, int H, int C,
                        const float* PB, const float* m0, const float* pi_hat, float* gain, coda_stream_t stream);

/* ---- fused single-CTA step kernels: selection, label, posterior update, mixture --------------------------- */
typedef struct coda_step { /* host struct: this shard's device state */
  int H, C;
  int64_t N, n_offset;
  int fx_shift;
  float lr;
  const uint16_t* hard; /* [N][H] */
  uint8_t* labeled;     /* [N] */
  float* D;             /* [H][C][C] */
  int32_t* jvec;        /* [H] p_h(idx) of the labeled item */
  int64_t* sel;         /* {local index or -1, class} */
  /* rank-1 gather list (see coda_b200_pi_rank1) */
  int32_t* terms; /* [2 + 8H] */
  const int32_t* slot_of_model;
  int64_t shadow_off, shadow_col_stride, model_stride;
  int have_ens;
  int compact_k; /* > 0: the slab is in the compact top-K form, the gather list names (model, class) pairs */
  /* marginals / mixture */
  int64_t* pisum_fx;   /* [C] local sums */
  const float* PB;     /* [C][Hp] */
  float* pi_hat;       /* [C] */
  float* m0;           /* [Hp] */
  float* h_before;     /* [1] */
  int64_t* best_model; /* [1] */
  /* selection */
  const int64_t* partials; /* [nblocks][REC_WORDS] */
  int nblocks;
  const float* eig;
  int64_t* bestrec; /* [REC_WORDS] merged (global) record */
  /* host-free loop */
  const int64_t* labels_global;
  int64_t* hist_idx;
  float* hist_q;
  int32_t* hist_tie;
  int64_t hist_cap;
  int64_t* step_ctr; /* [1] */
  uint32_t* flags;
} coda_step_t;

/* coda.py:306/309 + oracle(idx) + coda.py:316-317 with no host in the loop: merge the block records, exchange
 * {record, p_h(candidate)} with every peer, take the global arg-max (first index; an isclose tie -- coda.py:307 --
 * is recorded in hist_tie), look the label up in labels_global, mark the item labeled, D[h][t][p_h(idx)] += lr,
 * build the rank-1 gather list, zero pisum. */
int coda_b200_step_select(const coda_step_t* st, const coda_xchg_t* x, coda_stream_t stream);
/* API path, get_next_item_to_label: merge + exchange only -> bestrec. */
int coda_b200_step_merge(const coda_step_t* st, const coda_xchg_t* x, coda_stream_t stream);
/* API path, add_label (coda.py:315-317): sel = {local idx or -1, class} given; the owner shares p_h(idx). */
int coda_b200_step_label(const coda_step_t* st, const coda_xchg_t* x, coda_stream_t stream);
/* pi_hat (coda.py:232-233; the shards' sums are exchanged and added here), P(best) vector m0 == get_pbest()
 * (coda.py:253, 325-332), H_before (coda.py:254) and argmax (coda.py:346). */
int coda_b200_step_mixture(const coda_step_t* st, const coda_xchg_t* x, coda_stream_t stream);

/* tie scan (coda.py:307 torch.isclose(q, best, rtol=1e-8[, atol=1e-8]) in fp32) against the global record. */
int coda_b200_ties(const float* eig, int64_t N, const uint8_t* labeled, const uint8_t* disagree, int64_t n_offset,
                   const int64_t* best /*[REC_WORDS]*/, int cap, int64_t* tie_hdr /*[2]*/, int64_t* tie_idx,
                   float* tie_val, coda_stream_t stream);
/* every shard's report block (flags, record, tie list: rep_words int64) -> rep_all [world][rep_words] on every shard */
int coda_b200_report_gather(const int64_t* rep, int rep_words, int64_t* rep_all, const coda_xchg_t* x,
                            uint32_t* flags, coda_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* CODA_B200_H */
