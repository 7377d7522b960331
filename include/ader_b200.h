/* ader_b200.h -- C ABI of the B200-native ADER hot path (libader_b200.so).
 *
 * The reference (doublemul/ADER) has no FFI layer: its seam is the TF1 feed/fetch contract of
 * the `Ader` / `Ewc` model objects (ADER.py:16-23, ADER.py:85-150, EWC.py:115-177).  Each entry
 * point below replaces the device work behind one group of those fetches; the Python host
 * (`ader_b200/model.py`) keeps the reference's method surface on top of them.
 *
 * Conventions (SURVEY.md 8b):
 *   - plain C, POD structs, raw DEVICE pointers + sizes, `void* stream` is a cudaStream_t;
 *   - the caller owns every buffer (incl. workspaces; sizes from the *_bytes queries);
 *   - functions never allocate, never synchronise, are stream-ordered and re-entrant;
 *   - return 0 on success, <0 on error (-1 bad argument, -2 bad alignment/size, -3 launch error);
 *     `ader_last_error()` returns a thread-local message;
 *   - no C++ exception crosses the boundary.  There is no CPU fallback.
 *
 * Data layout.  All trainable state lives in ONE flat fp32 vector `theta` (and twins m, v, grad,
 * fisher, theta_star) in the creation order of EWC.py:90 / SURVEY A.2:
 *   [ item_table (v_tab x d) | pos_table (maxlen x d) | block 0 | ... | block NB-1 | lnf.beta | lnf.gamma ]
 *   block = [ln1.beta, ln1.gamma, wq (d x d, in-major), bq, wk, bk, wv, bv, ln2.beta, ln2.gamma, w1, b1, w2, b2]
 * Sessions are packed: only real (non-zero) tokens are stored, T = sum of row lengths.
 */
#ifndef ADER_B200_H
#define ADER_B200_H

#include <stdint.h>
#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

#define ADER_ABI_VERSION 2

typedef struct AderModel {
  int32_t v_tab;       /* rows of the item table = item_num + 1   (ADER.py:29-38)           */
  int32_t d;           /* hidden_units                            (main.py:103)             */
  int32_t maxlen;      /* L                                       (main.py:104)             */
  int32_t num_blocks;  /* (main.py:99)                                                       */
  int32_t num_heads;   /* (main.py:100), must divide d                                      */
} AderModel;

/* ---- introspection ------------------------------------------------------------------- */
int32_t     ader_abi_version(void);
const char* ader_last_error(void);
/* number of fp32 elements in theta; offset (in elements) of tensor `idx` (0..2+14*NB+1). */
int64_t     ader_param_count(const AderModel* m);
int64_t     ader_param_offset(const AderModel* m, int32_t idx);
int64_t     ader_dense_count(const AderModel* m);      /* everything after the item table */

/* ---- encoder: modules.py:23-271 + ADER.py:25-85 (subsystem 1) ------------------------- */
/* Activation workspace (saved for backward) for M rows and a capacity of Tcap real tokens
 * (Tcap <= M * maxlen; the exact token count is computed on the device, overflow is flagged
 * in the workspace's flags slot and clamped). */
size_t  ader_encoder_ws_bytes(const AderModel* m, int32_t M, int32_t Tcap);
/* Backward scratch + split-K partial-gradient workspace. */
size_t  ader_encoder_bwd_ws_bytes(const AderModel* m, int32_t M, int32_t Tcap);
/* byte offset of a named activation slot inside the encoder workspace (tests / debugging).
 * slot: 0 x_in(block), 1 q=LN1(x), 2 Q, 3 K, 4 V, 5 y=attn+q, 6 z=LN2(y), 7 h=relu(.), 8 x_out(last block),
 *       9 probs(block) ; -1 row_len, -2 row_off, -3 tok_row, -4 flags (flags[0] != 0: token overflow) */
int64_t ader_encoder_ws_slot(const AderModel* m, int32_t M, int32_t Tcap, int32_t slot, int32_t block);

/* ids [M, maxlen] int32 left-zero-padded (util.py:151-171) -> rep [M, d] fp32 (ADER.py:85).
 * dropout_rate > 0 applies tf.layers.dropout at the 1+3*NB reference sites (ADER.py:55,
 * modules.py:214,257,262) with a counter-based generator keyed by (seed, step). */
int32_t ader_encoder_fwd(const AderModel* m, const float* theta, const int32_t* ids, int32_t M,
                         int32_t Tcap, void* ws, float* rep, float dropout_rate, uint64_t seed, void* stream);
/* d_rep [M, d] -> grad (flat, same layout as theta): writes the pos_table and all block / lnf
 * gradients, and ADDS the input-lookup scatter (ADER.py:29-38, sqrt(d)-scaled) into the item
 * table rows of `grad` (which must already hold the output-projection gradient, or zeros).
 * The scatter is a stable radix sort by item id + windowed segmented reduction: deterministic (every row is a fixed
 * function of the sorted order; float reductions to memory have exactly one contributor per address). */
int32_t ader_encoder_bwd(const AderModel* m, const float* theta, const int32_t* ids, int32_t M,
                         int32_t Tcap, const void* ws, void* bwd_ws, const float* d_rep, float* grad,
                         float dropout_rate, uint64_t seed, void* stream);

/* Same two contracts on the tensor cores: fused sub-layer kernels ([embed] + LN + Q/K/V, attention + LN, FFN and
 * their backward twins) with row-scaled fp16 operands / fp32 accumulation, weights staged by bulk async copies;
 * weight / bias / LayerNorm-parameter gradients on TF32 tensor cores with fp32 accumulation in a fixed order
 * (deterministic).  Workspaces and slots are identical to the exact path (same *_ws_bytes queries).  Needs
 * hidden_units <= 160.  Results agree with the exact path to the tolerances stated in
 * tests/test_gpu_encoder_fused.py (activations 1e-2, gradients 3e-2 rel-L2 per tensor).
 * d_step (device int32, may be NULL): added to `seed` on the device, so a captured CUDA graph draws fresh dropout
 * masks on every replay (pass the Adam state pointer: state[0] is the step counter). */
int32_t ader_encoder_fwd_tc(const AderModel* m, const float* theta, const int32_t* ids, int32_t M,
                            int32_t Tcap, void* ws, float* rep, float dropout_rate, uint64_t seed,
                            const int32_t* d_step, void* stream);
int32_t ader_encoder_bwd_tc(const AderModel* m, const float* theta, const int32_t* ids, int32_t M,
                            int32_t Tcap, const void* ws, void* bwd_ws, const float* d_rep, float* grad,
                            float dropout_rate, uint64_t seed, const int32_t* d_step, void* stream);

/* ---- logits + CE + distillation: ADER.py:88-93, ADER.py:108-138 (subsystem 2) ---------- */
typedef struct AderLossArgs {
  int32_t M;               /* rows of rep = n_train + n_ex (exemplar rows LAST, main.py:229)   */
  int32_t n_train;         /* rows with one-hot labels `pos`                                   */
  int32_t n_ex;            /* exemplar rows                                                    */
  int32_t V;               /* max_item: logits columns are items 1..V (ADER.py:90-92)          */
  int32_t V_prev;          /* teacher width (columns 1..V_prev), 0 when mode != KD             */
  int32_t mode;            /* 0 vanilla (ADER.py:93), 1 KD (ADER.py:133-137), 2 ER one-hot (ADER.py:126-131) */
  float   lambda_;         /* main.py:196-200                                                  */
  const int32_t* pos;      /* [n_train] labels 1..V                                            */
  const int32_t* ex_pos;   /* [n_ex] labels (mode 2)                                           */
  const float*   teacher;  /* [*, V_prev] fp32 stored exemplar logits (mode 1), or NULL with teacher_rep */
  const int32_t* teacher_row; /* [n_ex] row of `teacher` (or `teacher_rep`) per exemplar row, or NULL = identity */
  int64_t teacher_ld;      /* row stride of `teacher` in elements (>= V_prev)                  */
  int32_t n_train_global;  /* data parallel: denominators of the two means over ALL ranks (0 = local   */
  int32_t n_ex_global;     /* counts); gradients and loss are then summed, not averaged, across ranks  */
  /* Frozen teacher (mode 1, instead of `teacher`): a snapshot of the previous model.  Teacher logits are recomputed per
   * step as teacher_rep[teacher_row[e]] . table^T over items 1..V_prev, so the library never holds an [E, V_prev] matrix.
   * Exactly one of `teacher` / `teacher_rep` is set in mode 1. */
  const float* teacher_rep;      /* [*, d] fp32 exemplar representations (exact encoder, taken at selection time) */
  const float* teacher_table;    /* fp32 rows of items 1..V_prev of the frozen item table, row stride d (exact entry) */
  const void*  teacher_table16;  /* bf16 [ceil(V_prev/128)*128][160] shadow of the same rows (ader_pack_table16;
                                    tcgen05 entries) */
} AderLossArgs;

size_t  ader_loss_ws_bytes(const AderModel* m, const AderLossArgs* a);
/* rep [M,d] -> loss[0] (scalar), row_loss [M], d_rep [M,d]; writes the dense output-projection
 * gradient into grad rows 1..V of the item table (rows 0 and >V untouched). */
int32_t ader_loss_fwd_bwd(const AderModel* m, const float* theta, const float* rep,
                          const AderLossArgs* a, void* ws, float* loss, float* row_loss,
                          float* d_rep, float* grad, void* stream);
/* Same contract on the tcgen05 tensor cores (bf16 operands, fp32 accumulate in TMEM): fused
 * logits + online-softmax CE + distillation, [M, V] logits never materialised in HBM.  Distillation
 * rows enter by linearity: bf16 tiles of coef * softmax(teacher) are MMA operands (uc = Pc.E for the loss and
 * d_rep, dE -= Pc^T.rep), so the hot kernels never read the fp32 teacher.  Results agree with
 * ader_loss_fwd_bwd to bf16 operand rounding (tests state the tolerance).
 * With a frozen teacher (teacher_rep + teacher_table16) two more tcgen05 passes over the snapshot give the teacher's
 * log-sum-exp and then the same bf16 Pc tiles, on the side of the step that does not depend on `rep`. */
size_t  ader_loss_tc_ws_bytes(const AderModel* m, const AderLossArgs* a);
int32_t ader_loss_fwd_bwd_tc(const AderModel* m, const float* theta, const float* rep,
                             const AderLossArgs* a, void* ws, float* loss, float* row_loss,
                             float* d_rep, float* grad, void* stream);
/* Measurement hook: launches only the three tcgen05 kernels (forward statistics, d_rep partials, dE) on a workspace
 * prepared by a preceding ader_loss_fwd_bwd_tc call with the same arguments (bench.py times them with CUDA events). */
int32_t ader_debug_loss_tc_kernels(const AderModel* m, const float* theta, const AderLossArgs* a, void* ws,
                                   float* grad, void* stream);
/* Vocab-parallel form of the same kernels (one rank owns logits columns [v_lo, v_hi), v_lo % 128 == 0):
 *   fwd  -> stats [M,4] = this shard's per-row (max, sum exp(s - max), label logit or 0, KD dot);
 *           the caller all-reduces them (max; rescaled sum; sums) into lse [M];
 *   bwd  -> d_rep_partial [M,d] (to be all-reduce-summed) and grad rows v_lo+1 .. v_hi of the item table.
 * `a->V` stays the GLOBAL max_item.  The workspace must persist between the two calls.  Stored teacher logits only
 * (a frozen teacher is rejected). */
size_t  ader_loss_tc_vp_ws_bytes(const AderModel* m, const AderLossArgs* a, int32_t v_lo, int32_t v_hi);
int32_t ader_loss_tc_vp_fwd(const AderModel* m, const float* theta, const float* rep, const AderLossArgs* a,
                            int32_t v_lo, int32_t v_hi, void* ws, float* stats, void* stream);
int32_t ader_loss_tc_vp_bwd(const AderModel* m, const float* theta, const float* rep, const AderLossArgs* a,
                            int32_t v_lo, int32_t v_hi, void* ws, const float* lse, float* d_rep_partial,
                            float* grad, void* stream);
/* ---- one training pass: sess.run(train_op) minus the optimiser (main.py:233-256) ------------ */
/* encoder forward -> logits + CE + distillation forward/backward -> encoder backward + scatter, i.e. exactly
 *   ader_encoder_fwd_tc(.., enc_ws, rep, ..) ; ader_loss_fwd_bwd_tc(.., rep, a, loss_ws, loss, row_loss, d_rep, grad) ;
 *   ader_encoder_bwd_tc(.., enc_ws, bwd_ws, d_rep, grad, ..)
 * with the same arguments and bit-identical results, issued as a fork/join DAG: launches that are off the critical
 * chain (table-tile packing, teacher products, dE, weight-shadow packing, weight / LayerNorm / position gradients,
 * partial reductions, the scalar loss) go to five library-owned side streams ordered against `stream` by events, and
 * the kernel-to-kernel links of the chain are programmatic dependent launches (the next kernel's prologue overlaps the
 * previous kernel's drain);
 * everything is joined back into `stream` before the call returns, so the function stays stream-ordered for the
 * caller, and under stream capture the side streams become parallel branches of the captured graph.  The side
 * streams/events are created once per host thread and device on first use (the only allocation in the library:
 * call once outside capture first).  serial != 0 issues the same launches on `stream` only. */
int32_t ader_train_fwd_bwd_tc(const AderModel* m, const float* theta, const int32_t* ids, int32_t M, int32_t Tcap,
                              const AderLossArgs* a, void* enc_ws, void* bwd_ws, void* loss_ws, float* rep,
                              float* loss, float* row_loss, float* d_rep, float* grad, float dropout_rate,
                              uint64_t seed, const int32_t* d_step, int32_t serial, void* stream);

/* bf16 shadow of table rows for the tcgen05 entries: `rows` = fp32 rows of items 1..V, row stride d (theta + d for the
 * live table, or a frozen AderLossArgs.teacher_table) -> out bf16 [ceil(V/128)*128][160], rows >= V and columns >= d zero
 * (the operand layout of the tcgen05 loss kernels).  ader_table16_ws_bytes = bytes of `out`.  Needs hidden_units <= 160. */
size_t  ader_table16_ws_bytes(const AderModel* m, int32_t V);
int32_t ader_pack_table16(const AderModel* m, const float* rows, int32_t V, void* out, void* stream);

/* logits [M, V] fp32 = rep . E[1..V]^T  (fetch `logits`, util.py:452,482,514). ld = row stride. */
int32_t ader_logits(const AderModel* m, const float* theta, const float* rep, int32_t M, int32_t V,
                    float* logits, int64_t ld, void* stream);

/* ---- optimiser: tf.train.AdamOptimizer (ADER.py:96) + EWC penalty (EWC.py:115-124) ------ */
typedef struct AderAdamArgs {
  float lr, beta1, beta2, eps;
  int32_t V;               /* table rows 1..V are updated (rows > V have m = v = g = 0 forever) */
  float ewc_lambda;        /* 0 = off; else grad += lambda * F * (theta - theta_star)          */
  const float* fisher;     /* flat, same layout as theta (or NULL)                              */
  const float* theta_star; /* flat (or NULL)                                                    */
} AderAdamArgs;
/* state: device int32[2]; state[0] = step t, incremented by this call (the update uses the value
 * after the increment); state[1] is scratch (bits of the bias-corrected step size). */
int32_t ader_adam_step(const AderModel* m, float* theta, float* adam_m, float* adam_v,
                       const float* grad, int32_t* state, const AderAdamArgs* a, void* stream);

/* The same pass with the optimiser folded in (one GPU: nothing sits between backward and Adam): identical to
 * ader_train_fwd_bwd_tc followed by ader_adam_step(theta, adam_m, adam_v, grad, state, opt), bit for bit, but the
 * step size is prepared at the start of the DAG, the item-table rows are updated as soon as the scatter has added
 * into them and the dense parameters as soon as their split partials are reduced (the weight-gradient tail and the
 * table update overlap).  state[0] is incremented by the dense update, after the last reader of the dropout counter. */
int32_t ader_train_step_tc(const AderModel* m, float* theta, const int32_t* ids, int32_t M, int32_t Tcap,
                           const AderLossArgs* a, void* enc_ws, void* bwd_ws, void* loss_ws, float* rep,
                           float* loss, float* row_loss, float* d_rep, float* grad, float dropout_rate,
                           uint64_t seed, const int32_t* d_step, float* adam_m, float* adam_v, int32_t* state,
                           const AderAdamArgs* opt, int32_t serial, void* stream);

/* ---- evaluation: ADER.py:99-103, util.py:309-339 (subsystem 5) -------------------------- */
size_t  ader_eval_ws_bytes(const AderModel* m, int32_t M, int32_t V);
/* rep [M,d], gt [M] (1..V) -> rank [M] (0-based rank of gt, ties -> lower index first),
 * topk_item [M,k] (1-based ids, best first), topk_score [M,k]; k <= 32. */
int32_t ader_eval_rank_topk(const AderModel* m, const float* theta, const float* rep, const int32_t* gt,
                            int32_t M, int32_t V, int32_t k, void* ws, int32_t* rank,
                            int32_t* topk_item, float* topk_score, void* stream);

/* The same ranks on the tcgen05 tensor cores, the [R, V] score matrix never written (the metrics of util.py:329-339 only
 * read rank(gt)).  Filter and refine: the exact fp32 score of the ground-truth item anchors a certainty band
 * s_gt +- eps_i, eps_i = 2^-12 ||rep_i|| max_j ||E_j||; approximate scores from a two-term bf16 split of both operands
 * (three products hi.hi + hi.lo + lo.hi accumulated in TMEM) are counted when certainly above, and the few columns inside
 * the band are re-scored with the exact fmaf chain of ader_eval_rank_topk -- ranks are identical to that entry, ties
 * included.  overflow[0] (device int) != 0: a row had more than ADER_EVAL_CAND_CAP columns inside its band; the caller
 * must then use ader_eval_rank_topk for this batch.  Needs hidden_units <= 160. */
#define ADER_EVAL_CAND_CAP 256
size_t  ader_eval_rank_tc_ws_bytes(const AderModel* m, int32_t R, int32_t V);
int32_t ader_eval_rank_tc(const AderModel* m, const float* theta, const float* rep, const int32_t* gt, int32_t R,
                          int32_t V, void* ws, int32_t* rank, int32_t* overflow, void* stream);
/* ... plus the top-k items of every row (ids 1-based, best first, ties -> lower id; exact fp32 scores), identical to
 * ader_eval_rank_topk: a first tensor-core pass keeps the largest approximate score of every (vocabulary chunk, column
 * half) of a row -- each belongs to a different item, so the k-th largest of them, minus 2 eps, bounds the approximate
 * score of every top-k item from below; a second pass collects the columns above that bound (and does the rank counting
 * of ader_eval_rank_tc), and the candidates are re-scored exactly and sorted.  Needs 2 * ader_eval_topk_chunks(R, V) >= k
 * (enough distinct local maxima; small vocabularies use ader_eval_rank_topk).  Same workspace query, same overflow flag. */
int32_t ader_eval_topk_chunks(const AderModel* m, int32_t R, int32_t V);
int32_t ader_eval_rank_topk_tc(const AderModel* m, const float* theta, const float* rep, const int32_t* gt, int32_t R,
                               int32_t V, int32_t k, void* ws, int32_t* rank, int32_t* topk_item, float* topk_score,
                               int32_t* overflow, void* stream);

/* ---- exemplar selection: util.py:401-461 (subsystem 4) ---------------------------------- */
/* Segmented herding.  rep [N,d]; segment s owns candidate rows cand[seg_off[s] .. seg_off[s+1])
 * (indices into rep, in the reference's sess_by_item order); quota[s] = min(m, n_s);
 * max_steps[s] = ceil(1.1*m) evaluated in float64 on the host (util.py:425).
 * Output picks[seg_off[s] + k] = k-th selected LOCAL candidate index, n_picked[s]. */
size_t  ader_herding_ws_bytes(const AderModel* m, int32_t N);
int32_t ader_herding_segmented(const AderModel* m, const float* rep, int32_t N, const int32_t* cand,
                               const int32_t* seg_off, int32_t n_seg, const int32_t* quota,
                               const int32_t* max_steps, void* ws, int32_t* picks, int32_t* n_picked,
                               void* stream);

/* ---- EWC Fisher diagonal: EWC.py:126-164 ------------------------------------------------ */
/* acc (fp64, flat) += square_fp32(grad) over table rows 1..V and all dense params. */
int32_t ader_fisher_accumulate(const AderModel* m, const float* grad, double* acc, int32_t V, void* stream);
/* fisher (fp32, flat) = acc / n_data over the same range; zero elsewhere. */
int32_t ader_fisher_finalize(const AderModel* m, const double* acc, float* fisher, int32_t V,
                             int32_t n_data, void* stream);

/* ---- data parallel over NVLink peer memory (SURVEY 8e) --------------------------------------
 * The reference is single-device (main.py:96,120,143: one CUDA_VISIBLE_DEVICES id, one tf.Session); a rank here is a
 * process that runs `sess.run(train_op)` (main.py:233-256) on its shard of the step's rows with the GLOBAL mean
 * denominators (AderLossArgs.n_*_global).  ader_dp_adam_step then replaces all-reduce(grad) + ader_adam_step by ONE
 * kernel: rank r owns a slice of [table rows 1..V | dense parameters]; it loads that slice of every rank's gradient
 * through peer pointers, sums in rank order, applies the TF1-Adam expression of ader_adam_step with its local m / v,
 * and stores the new theta slice into every replica.  Cross-rank ordering uses epoch flags in peer memory (no host,
 * graph-capturable); a wait that sees no progress for ~20 s marks the error word instead of hanging the GPU.
 *   flags[r]: ADER_DP_FLAG_WORDS zero-initialised uint32 of rank r, mapped into every rank.
 * ader_dp_wait must be the first launch of a step (before anything rewrites grad or reads theta): it waits until every
 * rank has finished the previous ader_dp_adam_step.  Pointers of other processes come from ader_ipc_export/open. */
#define ADER_DP_MAX_RANKS 16
#define ADER_DP_FLAG_WORDS 64
typedef struct AderDpComm {
  int32_t   rank, world;
  int32_t   separate_arrive;            /* kept for layout compatibility, ignored: the "gradients complete" barrier always runs
                                           as its own single-warp kernel (k_dp_arrive) ahead of the full-occupancy update */
  int32_t   reserved;
  float*    theta[ADER_DP_MAX_RANKS];
  float*    grad[ADER_DP_MAX_RANKS];
  uint32_t* flags[ADER_DP_MAX_RANKS];
  /* optional NVLS multicast views of the SAME buffers (NVSwitch multicast object bound to every rank's theta / grad,
     e.g. torch symmetric memory): when both are set the update kernel sums the gradient inside the switch
     (multimem.ld_reduce: each rank loads its slice once instead of once per peer) and broadcasts the new parameters with
     one multimem.st per quad; NULL = peer loads / stores through theta[] / grad[]. */
  float*    mc_theta;
  float*    mc_grad;
} AderDpComm;
int32_t ader_dp_wait(const AderDpComm* c, void* stream);
int32_t ader_dp_adam_step(const AderModel* m, const AderDpComm* c, float* adam_m, float* adam_v, int32_t* state,
                          const AderAdamArgs* a, void* stream);
/* synchronous read of this rank's flag block: err != 0 after a timed-out wait; epoch = 2 x completed steps */
int32_t ader_dp_status(const AderDpComm* c, int32_t* err_out, uint32_t* epoch_out);
/* CUDA IPC: 64-byte handle of the allocation that holds dev_ptr + the byte offset of dev_ptr inside it (exporter);
 * ader_ipc_open maps that allocation into this process and returns its base (importer adds the offset). */
int32_t ader_ipc_export(const void* dev_ptr, void* handle64, int64_t* offset);
int32_t ader_ipc_open(const void* handle64, void** base_ptr);
int32_t ader_ipc_close(void* base_ptr);

/* The same statistic for S samples in ONE batched pass (Ewc.compute_fisher's loop over `sess.run(self.gradient)` at batch 1,
 * EWC.py:142-161): acc (fp64, flat) += sum_s (d CE_s / d theta)^2 over table rows 1..V and all dense parameters, with
 * per-sample (batch-of-one, eval mode) semantics.  One exact forward + data-gradient backward over all samples; the
 * per-sample weight gradients are formed where the ordinary backward would sum over the batch (outer products over the
 * tokens of one sample), squared in fp32 and accumulated in fp64; the item-table part is the product of squares
 * (softmax - onehot)^2 x rep^2 over row chunks plus an exact correction of the (sample, item) pairs that also receive
 * the input-lookup scatter.  ids [S, maxlen] left-padded, every row with >= 1 token; pos [S] labels.  enc_ws / bwd_ws
 * sized for (S, Tcap) by the encoder queries.  Follow with ader_fisher_finalize. */
size_t  ader_fisher_batched_ws_bytes(const AderModel* m, int32_t S, int32_t V);
int32_t ader_fisher_batched(const AderModel* m, const float* theta, const int32_t* ids, const int32_t* pos, int32_t S,
                            int32_t Tcap, int32_t V, void* enc_ws, void* bwd_ws, void* ws, double* acc, void* stream);

/* ---- helpers ---------------------------------------------------------------------------- */
/* out[i, :] = src[idx[i], :] for int32 rows (batch assembly from the GPU-resident row matrix). */
int32_t ader_gather_rows_i32(const int32_t* src, const int32_t* idx, int32_t n, int32_t width,
                             int32_t* out, void* stream);

/* the whole batch of a step in one launch (Sampler.sampler + exemplar_sampler, util.py:151-263, on GPU-resident row
 * matrices): ids [n_train + n_ex, width] = t_ids[ti[.]] then e_ids[ei[.]]; pos [n_train] = t_lab[ti[.]];
 * aux [n_ex] = e_aux[ei[.]] (teacher row or one-hot label of each exemplar; aux / e_aux may be NULL). */
int32_t ader_gather_batch(const int32_t* t_ids, const int32_t* t_lab, const int32_t* ti, int32_t n_train,
                          const int32_t* e_ids, const int32_t* e_aux, const int32_t* ei, int32_t n_ex,
                          int32_t width, int32_t* ids, int32_t* pos, int32_t* aux, void* stream);

/* the same assembly fed from an epoch-resident index queue: q = the row indices of every step of the epoch back to back
 * ([n_train train indices | n_ex exemplar indices] per step), q_off[s] = start of step s, *counter = running step.  A captured
 * step replays without any host-to-device copy; ader_queue_advance (stream-ordered) moves to the next step. */
int32_t ader_gather_batch_q(const int32_t* t_ids, const int32_t* t_lab, int32_t n_train, const int32_t* e_ids,
                            const int32_t* e_aux, int32_t n_ex, const int32_t* q, const int64_t* q_off,
                            const int32_t* counter, int32_t width, int32_t* ids, int32_t* pos, int32_t* aux, void* stream);
int32_t ader_queue_advance(int32_t* counter, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* ADER_B200_H */
