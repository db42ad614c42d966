/* tcar_b200.h -- C ABI of libtcar_b200.so: the B200 (sm_100a) replacement for the TensorFlow kernels that the
 * reference's TCAR train / full-catalog-eval hot path executes inside `sess.run`
 * (summmeer/session-based-news-recommendation: model_combine.py:231-234 train, :283-286 eval).
 *
 * Conventions (SURVEY.md 8b):
 *   - every function returns 0 on success, a cudaError_t (>0) or a TCAR_ERR_* code (<0); nothing throws;
 *   - all pointers are DEVICE pointers owned by the caller; no function allocates or frees device memory;
 *   - every function is asynchronous on the caller-supplied stream (`void* stream` is a cudaStream_t) and
 *     keeps no global mutable state besides cached immutable driver/device queries;
 *   - index arrays are int32, tables / activations fp32 unless a name says bf16.
 *
 * Shapes: B <= 512 sessions per call, T <= 40 clicks, H = 250, Th = 64, N items, Nn negatives.
 * Trainable / frozen item tables use a 256-float row pitch (TCAR_HP) so rows are 128-bit aligned.
 */
#ifndef TCAR_B200_H_
#define TCAR_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define TCAR_H 250        /* hidden_size == content width   (model_combine.py:45, main.py:109)        */
#define TCAR_HP 256       /* row pitch of item/content tables in floats                                 */
#define TCAR_TH 64        /* time_hidden_size               (model_combine.py:46, modules.py:138)     */
#define TCAR_XW 500       /* [item+pos | content]           (model_combine.py:111)                    */
#define TCAR_PW 320       /* 5 publish-time embeddings      (model_combine.py:84)                     */
#define TCAR_NBINS 139    /* 13 + 32 + 8 + 25 + 61 rows of the month/day/week/hour/minute tables      */
#define TCAR_KEXT 640     /* scoring K: 500 + 139 one-hot time bins + 1 zero pad                        */
#define TCAR_QROWS 512    /* max sessions per scoring call (main.py:101 batch_size default)            */
#define TCAR_MAXT 40      /* position table rows            (model_combine.py:57)                     */
#define TCAR_TOPK 20      /* cutoff                          (model_combine.py:296,301)                */
#define TCAR_CHUNK 8      /* items per eval chunk-max                                                   */
#define TCAR_NCAND_CHUNKS 32 /* chunks re-scored per query (256 candidate items)                        */
#define TCAR_MAX_EVAL_TILES 32768 /* 128-item tiles per catalog (shard) the top-20 selection handles: 4.2 M items */
/* One shard's evaluation results for <= 512 queries, as ONE contiguous block of 32-bit words (what a rank sends in the
 * single exchange of the catalog-sharded evaluation): planes at fixed offsets, each in the layout the kernels write. */
#define TCAR_EVAL_OFF_SCORES 0                          /* float [512][20]  top-20 scores                           */
#define TCAR_EVAL_OFF_IDS (TCAR_QROWS * TCAR_TOPK)      /* int32 [512][20]  top-20 global item ids (-1 = empty)      */
#define TCAR_EVAL_OFF_NGT (2 * TCAR_QROWS * TCAR_TOPK)  /* int32 [512]      #(S > S[label]) among the shard's items  */
#define TCAR_EVAL_OFF_SUMEXP (TCAR_EVAL_OFF_NGT + TCAR_QROWS)   /* float [512] softmax partial sum                   */
#define TCAR_EVAL_OFF_ROWMAX (TCAR_EVAL_OFF_SUMEXP + TCAR_QROWS) /* float [512] largest exponent argument (guard)    */
#define TCAR_EVAL_BLOCK_WORDS (TCAR_EVAL_OFF_ROWMAX + TCAR_QROWS)
#define TCAR_EVAL_NSEL 33         /* entries of a (query, item range) candidate list: 32 chunks + 1 bound carrier     */
#define TCAR_WIDEN_SPLITS 16      /* CTAs sharing one flagged query in tcar_eval_topk_widen                       */
#define TCAR_NORM_SPLIT 8    /* partial sums per tensor written by tcar_sqnorm_segments                     */
#define TCAR_TABLE_GRAD_CHUNKS 148   /* max click chunks (CTAs) of tcar_small_table_grads pass 1               */
#define TCAR_TABLE_GRAD_PART 19600   /* floats of partial sums per chunk: 139x64 + 11x64 + 40x250              */

#define TCAR_CLUSTER_PAIR (-2) /* tcar_score_fwd `cluster` value: CTA pair, tcgen05.mma.cta_group::2 (M = 256)   */

/* Overflow guard of the full-catalog softmax: the scoring kernel shifts the exponent by the label score c_b; a row
 * whose largest argument (S - c_b) log2(e) exceeds this limit (55 nats) is re-run shifted by its maximum, which is what
 * TF's sparse_softmax_cross_entropy_with_logits (model_combine.py:145) always does.  Below the limit the sums of up to
 * 2^19 terms <= 2^80 and everything the backward GEMMs derive from them stay far inside fp32 / bf16 range. */
#define TCAR_EXP_LIMIT2 80.0f

#define TCAR_ERR_ARG (-1)
#define TCAR_ERR_DRIVER (-2)
#define TCAR_ERR_TENSORMAP (-3)

/* ------------------------------------------------------------------------------------------------------------
 * (1) fused gather -- replaces the ten `embedding_lookup(..., max_norm=1)` call sites of model_combine.py:54-107
 *     (modules.py:36): clip(x) = x / max(||x||_2, 1) per gathered row.
 *   idx   [7][B*T] : seq (1-based item id), month, day, week, hour, minute, gap      (sampler.py:68-87)
 *   ctx   [2][B]   : click week, click hour                                          (sampler.py:106-107)
 *   X [B*T,500] = [clip(item[seq]) + clip(pos[t]) | clip(content[seq])]; P [B*T,320]; D [B*T,64]; CT [B,128]
 */
int tcar_gather_fwd(const int32_t* idx, const int32_t* ctx, const float* item, const float* content,
                    const float* pos, const float* month, const float* day, const float* week, const float* hour,
                    const float* minute, const float* dur, float* X, float* P, float* D, float* CT, int B, int T,
                    void* stream);

/* (2) attention pooling forward -- modules.py:72-152 (count_alpha_m / count_alpha_s / *_attention_layer) after
 *     the linear_3d projections.  U1/U2 [B*T, 256-float pitch] hold the pre-activation sums on entry and
 *     sigmoid(.) on exit (S1/S2/dU1/dU2 of the backward use the same pitch).
 *     alpha [3][B*T] = nrm(e1), nrm(e2), nrm(e_t) with nrm(x) = exp(x)/(sum exp(x) + 1e-9)  (util.py:92-100). */
int tcar_pool_fwd(const float* X, const float* P, float* U1, float* U2, const float* q, const float* w_r,
                  const float* w_t, float* alpha, float* pooled, float* pooled_t, int B, int T, void* stream);

/* (2b) attention pooling backward (gradient of (2) that tf.gradients derives, model_combine.py:156).
 *      Outputs dU1/dU2 (pre-activation grads), dXi [B*T, 256-float pitch] (item half of dX only -- content is frozen),
 *      dP [B*T,320], dq [B,500], de [3][B*T]. */
int tcar_pool_bwd(const float* X, const float* P, const float* S1, const float* S2, const float* q,
                  const float* w_r, const float* w_t, const float* alpha, const float* dpooled,
                  const float* dpooled_t, float* dU1, float* dU2, float* dXi, float* dP, float* dq, float* de,
                  int B, int T, void* stream);

/* (3a) candidate matrix -- model_combine.py:86-92,135-136 restated as Iext [Npad,640] bf16 =
 *      [item[1:] | content[1:] | one-hot(month,day,week,hour,minute bins) | 0]; rows >= N are zero. */
int tcar_build_iext(const float* item, const float* content, const int32_t* mwdhm, void* iext_bf16, int N,
                    int n_pad, void* stream);

/* clip() of the 139 month/day/week/hour/minute rows: CT [139,64] and 1/max(norm,1) [139]. */
int tcar_clip_time_tables(const float* month, const float* day, const float* week, const float* hour,
                          const float* minute, float* ct_tab, float* ct_scale, void* stream);

/* (3b) query operand: Tq [B,139] = a_pt . clip(tables)^T (fp32), Q [512,640] bf16 = [a_ic | Tq | 0] (rows >= B
 *      zero), c_ref [B] = fp32 score of the label item = S[b, label[b]] (model_combine.py:138,145). */
int tcar_build_query(const float* a_ic, const float* a_pt, const float* ct_tab, const float* item,
                     const float* content, const int32_t* mwdhm, const int32_t* label, float* Tq, void* q_bf16,
                     float* c_ref, int B, void* stream);

/* (0) GPU-resident sampler (sampler.py:52-113; SURVEY 8f-2): assemble the packed batch [7*B*T idx | 2*B ctx | B label
 *     | B*Nn neg] on the device from the columnar cache of one session-length bucket (seq [n,T+1], feats [6,n,T],
 *     ctx [2,n], all int32) and the batch's bucket rows [B].  neg_in != NULL: negatives copied from it (host-drawn,
 *     the reference's NumPy stream); neg_in == NULL: negative e = (philox4x32_10(key = seed, counter = offset + e/4)
 *     [e % 4] * item_num) >> 32, uniform in [0, item_num). */
int tcar_assemble_batch(const int32_t* rows, const int32_t* seq, const int32_t* feats, const int32_t* ctx,
                        int n_bucket, int B, int T, int Nn, const int32_t* neg_in, int item_num,
                        unsigned long long seed, unsigned long long offset, int32_t* out, void* stream);

/* Impression-list negatives on the device (sampler.py:118-131, the MIND configuration): for session b (bucket row
 * rows[b]) up to 21 uniform draws from its impression list impr_ids[impr_off[row] .. impr_off[row + 1]) -- entries are
 * 0-based item ids, -1 for an article that is not in item_dict -- the first Nn hits are kept, the remaining slots are
 * filled with uniform draws from [0, item_num).  Philox4x32-10 keyed by `seed`; session b owns TCAR_IMPR_BLOCKS(Nn)
 * counters from offset + b * TCAR_IMPR_BLOCKS(Nn): word j < 21 = try j, word 21 + k = fill of slot k.
 * neg_out [B, Nn] is then passed to tcar_assemble_batch as neg_in. */
#define TCAR_IMPR_BLOCKS(Nn) ((21 + (Nn) + 3) / 4)
int tcar_impression_negatives(const int32_t* rows, const int32_t* impr_off, const int32_t* impr_ids, int B, int Nn,
                              int item_num, unsigned long long seed, unsigned long long offset, int32_t* neg_out,
                              void* stream);

/* (3c) full-catalog scoring S = Q . Iext^T on tcgen05 (model_combine.py:138), never materialising S.
 *   mode 0 (train): E = exp(S - c_ref) in bf16, logically [512, n_pad], stored in blocks of 8 items:
 *                   E[b, n] at element ((n / 8) * 512 + b) * 8 + n % 8 (coalesced epilogue stores; the backward
 *                   kernels read it through a 3-D tensor map); rowsum_part [n_pad/128][512]
 *   mode 1 (eval) : chunkmax [512, n_pad/8] fp32 = max of S over 8 consecutive items, tilemax [512, n_pad/128]
 *                   fp32 = max over 128 consecutive items (first selection level of tcar_eval_topk_certified),
 *                   rowsum_part as above
 *   cluster in {1,2,4}: CTAs per cluster sharing each item tile by TMA multicast (one 128x128 UMMA per CTA);
 *   cluster == TCAR_CLUSTER_PAIR: CTA pairs issuing 256x256 cta_group::2 UMMAs, each CTA streaming half of every
 *   item tile (the production configuration: twice the pipeline depth per byte of shared memory). */
int tcar_score_fwd(const void* q_bf16, const void* iext_bf16, const float* c_ref, void* e_out, float* rowsum_part,
                   float* chunkmax, float* tilemax, int n_rows, int n_items, int n_pad, int mode, int cluster,
                   void* stream);
/* The same with the softmax overflow guard (TCAR_EXP_LIMIT2), run as two passes around tcar_ce_finish_guarded:
 *   pass 1  rowmax_part [n_pad/128][512] != NULL, rowmax == NULL: also leaves the largest exponent argument
 *           (S - c_ref) log2(e) of every (128-item block, session) pair;
 *   pass 2  rowmax [512] != NULL (what tcar_ce_finish_guarded pass 1 reduced, or its maximum over the ranks of a
 *           catalog-sharded step): rows above the limit are shifted by rowmax[b] on top of c_ref[b], so their largest
 *           term is 2^0.  CTAs none of whose 256 session rows need it return immediately (the common case costs one
 *           empty launch); the others rewrite E / rowsum_part / chunkmax -- identical values for the quiet rows. */
int tcar_score_fwd_guarded(const void* q_bf16, const void* iext_bf16, const float* c_ref, void* e_out,
                           float* rowsum_part, float* chunkmax, float* tilemax, float* rowmax_part, const float* rowmax,
                           int n_rows, int n_items, int n_pad, int mode, int cluster, void* stream);
int tcar_score_fwd_tiles(int n_pad);
/* Eval mode with a publish-time window per session row: item n is in the window of row b when
 * win_lo[b] <= item_time[n] <= win_hi[b] (int32, any clock unit the caller uses for both; win_lo[b] > win_hi[b] is an
 * empty window).  chunkmax / tilemax / rowsum_part as mode 1, except that an item outside the row's window counts as
 * -inf, exactly as items >= n_items do: a chunk or tile without an in-window item has the maximum -inf, and an
 * in-window chunk keeps the bit-exact mode-1 value.  item_time holds n_pad entries (those past n_items are not read as
 * scores).  Always the CTA-pair kernel (score_fwd_pair_kernel<2>); tilemax is nullable.  The inputs of
 * tcar_recommend_window. */
int tcar_score_fwd_window(const void* q_bf16, const void* iext_bf16, const float* c_ref, float* rowsum_part,
                          float* chunkmax, float* tilemax, const int32_t* item_time, const int32_t* win_lo,
                          const int32_t* win_hi, int n_rows, int n_items, int n_pad, void* stream);
/* Eval mode with a freshness decay per session row (DESIGN §4.10): chunkmax / tilemax as mode 1, but of the decayed
 * score r = s - p instead of s, with
 *   age = min(max(t_ref[b] - item_time[n], 0), TCAR_DECAY_MAX_AGE)   (exact, then exact in fp32)
 *   p   = rate[b] * age                                              (one fp32 multiply)
 *   r   = s - p                                                      (one fp32 subtract)
 * (item_time / t_ref int32 in one clock unit, rate[b] >= 0 and finite in score units per clock unit; items published
 * after t_ref[b] get age 0).  Items >= n_items, and with win_lo / win_hi (both given, or both NULL for no window)
 * items outside [win_lo[b], win_hi[b]], count as -inf as in tcar_score_fwd_window.  No softmax partial sums: only the
 * maxima are written.  item_time holds n_pad entries.  Always the CTA-pair kernel (score_fwd_pair_kernel<3>); tilemax
 * is nullable.  The inputs of tcar_recommend_decay. */
#define TCAR_DECAY_MAX_AGE 8388607   /* 2^23 - 1: ages saturate here (about 16 years in minutes) */
int tcar_score_fwd_decay(const void* q_bf16, const void* iext_bf16, float* chunkmax, float* tilemax,
                         const int32_t* item_time, const int32_t* t_ref, const float* rate, const int32_t* win_lo,
                         const int32_t* win_hi, int n_rows, int n_items, int n_pad, void* stream);

/* (4a) softmax cross-entropy from the partial sums (model_combine.py:145): sumexp[b] = sum_tiles part,
 *      ce[b] = log(sumexp[b]) (because c_ref is the label score). Fixed summation order. */
int tcar_ce_finish(const float* rowsum_part, float* sumexp, float* ce, int n_tiles, int B, void* stream);
/* With the overflow guard.  pass 1: sums + rowmax[b] = max_tiles rowmax_part (log2 units; ce may be inf for a row above
 * TCAR_EXP_LIMIT2 until pass 2).  pass 2 (after tcar_score_fwd_guarded re-ran with `rowmax`): rows above the limit are
 * summed again, ce[b] = log(sumexp[b]) + rowmax[b] ln 2 = logsumexp(S_b) - c_b; other rows keep their pass-1 values.
 * pass 3: rowmax only (the catalog-sharded step reduces it over the ranks first).  pass 0 == tcar_ce_finish. */
int tcar_ce_finish_guarded(const float* rowsum_part, const float* rowmax_part, float* sumexp, float* ce, float* rowmax,
                           int n_tiles, int B, int pass, void* stream);
/* The same fixed-order sum only, stored with a stride: out[b * out_stride] = sum_tiles part[tile][b]. */
int tcar_rowsum_finish(const float* rowsum_part, float* out, int out_stride, int n_tiles, int B, void* stream);

/* (4b) negative-feedback loss (model_combine.py:142-143,147): neg[b] = -log(1 - sigmoid(sum_j I_ic[neg_bj].a_ic[b])
 *      + 1e-24); loss[b] = ce[b] + 0.01 neg[b]; coef[b] = 0.01 d neg/d z; dA_neg[b,500] = coef[b] sum_j I_ic[neg_bj].
 *      ce == NULL: loss is not written (the kernel needs none of the scoring GEMM's results and may run beside it);
 *      tcar_loss_combine writes loss[b] = ce[b] + 0.01 negloss[b] once the cross loss is known. */
int tcar_neg_loss(const float* a_ic, const float* item, const float* content, const int32_t* neg, const float* ce,
                  float* negloss, float* loss, float* coef, float* dA_neg, int B, int Nn, void* stream);
int tcar_loss_combine(const float* ce, const float* negloss, float* loss, int B, void* stream);
/* Catalog-sharded step: sumexp[b] = sums[b * stride] (the softmax sums ride in the pad column of the reduce-scattered
 * dQ), ce[b] = log(sumexp[b]) + (rowmax[b] > TCAR_EXP_LIMIT2 ? rowmax[b] ln 2 : 0); rowmax nullable. */
int tcar_ce_from_sums(const float* sums, int stride, const float* rowmax, float* sumexp, float* ce, int B,
                      void* stream);

/* (3d) scoring backward wrt the query operand: dq_raw [512,640] = E . Iext (split-K partials in `part`,
 *      [tcar_score_bwd_q_splits()][512][640], reduced in fixed order). */
int tcar_score_bwd_q_splits(int n_rows, int n_pad);
int tcar_score_bwd_q(const void* e_bf16, const void* iext_bf16, float* part, float* dq_raw, int n_rows, int n_pad,
                     void* stream);

/* (3e) assemble d a_ic, d a_pt, dTq from dq_raw (softmax part / sumexp, minus the label one-hot in fp32, plus the
 *      negative-feedback part) and emit Qs [512,256] bf16 = a_ic[:, :250] / sumexp for (3f). */
int tcar_score_bwd_finish(const float* dq_raw, const float* sumexp, const float* dA_neg, const float* a_ic,
                          const float* ct_tab, const float* item, const float* content, const int32_t* mwdhm,
                          const int32_t* label, float* d_a_ic, float* d_a_pt, float* dTq, void* qs_bf16, int B,
                          void* stream);

/* (3f) scoring backward wrt the item embeddings: g_item[n+1, :250] = sum_b E[b,n] Qs[b,:] (dense, overwrites).
 *      sq_partial [tcar_score_bwd_i_ctas(n_pad)] (nullable): per-CTA sum of squares of what was written. */
int tcar_score_bwd_i(const void* e_bf16, const void* qs_bf16, float* g_item, float* sq_partial, int n_rows,
                     int n_items, int n_pad, void* stream);
int tcar_score_bwd_i_ctas(int n_pad);
/* Same with accumulate != 0: g_item += result.  A catalog-sharded train step (SURVEY 8e row 2) scores several groups
 * of <= 512 sessions (one per rank) against the rank's item range; groups after the first add to the dense gradient.
 * sq_partial then holds the sums of squares of the ACCUMULATED values written by this call. */
int tcar_score_bwd_i_acc(const void* e_bf16, const void* qs_bf16, float* g_item, float* sq_partial, int n_rows,
                         int n_items, int n_pad, int accumulate, void* stream);
/* dItems of ALL present session groups in one launch (what tcar_score_bwd_i / tcar_score_bwd_i_groups run): the groups
 * (E_g at e_bf16 + g * e_stride, Qs_g at qs_bf16 + g * qs_stride, n_rows[g] sessions, 0 = absent) are concatenated along
 * the reduction dimension, the gradient of the item range is accumulated in TMEM and written ONCE through
 * shared-memory staging + TMA stores (full 128-byte row segments).  groups <= TCAR_MAX_PEERS; sq_partial as above. */
int tcar_score_bwd_i_multi(const void* e_bf16, long long e_stride, const void* qs_bf16, long long qs_stride,
                           float* g_item, float* sq_partial, const int* n_rows, int groups, int n_items, int n_pad,
                           void* stream);

/* (5a) gradients of the seven small embedding tables (pos, month, day, week, hour, minute, duration): sums the
 *      gather-side, click-context-side and scoring-side contributions per table row in a fixed order, applies the
 *      clip Jacobian once per row and writes g_* (same shapes as the tables).  dXi has a 256-float row pitch.
 *      part: scratch of TCAR_TABLE_GRAD_CHUNKS x TCAR_TABLE_GRAD_PART floats (per-chunk partial sums, no initial
 *      state). */
int tcar_small_table_grads(const int32_t* idx, const int32_t* ctx, const float* dXi, const float* dP,
                           const float* dD, const float* dCT, const float* dTq, const float* a_pt,
                           const float* pos, const float* month, const float* day, const float* week,
                           const float* hour, const float* minute, const float* dur, float* g_pos, float* g_month,
                           float* g_day, float* g_week, float* g_hour, float* g_minute, float* g_dur, float* part,
                           int B, int T, void* stream);

/* (5a') backward of an elementwise activation fused with the bias gradient (linear_2d, modules.py:43-55):
 *      dz[r,c] = dy[r,c] * act'(y[r,c]) with act' expressed through the OUTPUT y (mode 0: tanh -> 1 - y^2,
 *      mode 1: relu -> y > 0); gb[c] = sum_r dz[r,c] in a fixed order.  dz may alias dy; `ld` = row pitch of all
 *      three matrices. */
int tcar_act_bwd_colsum(const float* dy, const float* y, float* dz, float* gb, int rows, int cols, int ld, int mode,
                        void* stream);
/* Several such column reductions in ONE launch.  mode 0 / 1 as above (a = dy [rows, ld]); mode 2: the weight-vector
 * gradients of count_alpha_* (modules.py:99,134): out[c] = sum_r y[r,c] * a[r] (a = [rows] vector, dz unused).
 * scratch (optional): TCAR_COL_SCRATCH(cols) floats, ZERO before the first use (the kernel leaves its ticket counters
 * at zero); with it, jobs of more than 1024 rows are split across CTAs and combined in a fixed order. */
#define TCAR_COL_JOBS 4
#define TCAR_COL_MAX_SPLIT 32
#define TCAR_COL_SCRATCH(cols) (TCAR_COL_MAX_SPLIT * (cols) + ((cols) + 31) / 32)
typedef struct tcar_col_job {
    const float* a;
    const float* y;
    float* dz;
    float* out;
    float* scratch;
    int rows, cols, ld, mode;
} tcar_col_job;
int tcar_col_jobs(const tcar_col_job* jobs, int njobs, void* stream);

/* (2c) dense projections on the tensor cores (tcgen05.mma.kind::tf32) -- the matmuls of linear_2d / linear_3d
 *      (modules.py:43-70) and their weight / data gradients:
 *          C[M,N] = act( sum_{s<nseg} A_s[M,K_s] . B_s[K_s,N] + bias )         act: 0 none, 1 relu, 2 tanh
 *      A_s is given K-major (row-major [M,K_s], a_mn_major = 0) or MN-major (row-major [K_s,M], a_mn_major = 1);
 *      B_s K-major (row-major [N,K_s]) or MN-major (row-major [K_s,N]).  Row pitches (lda/ldb, in floats) must be
 *      multiples of 4 and base pointers 16-byte aligned (TMA).  precise = 1: 3xTF32 (fp32-class accuracy), needs
 *      b = tf32(B), b_lo = tf32(B - b) with the same layout (tcar_prep_weights); precise = 0: single-pass TF32.
 *      splits > 1 splits the reduction over CTAs: `part` [tcar_gemm_tf32_part_elems(M,N,splits)] floats, reduced in
 *      a fixed order (no bias / act / accumulate / precise in that mode).  accumulate = 1: C += result. */
typedef struct tcar_gemm_seg {
    const float* a;
    const float* b;
    const float* b_lo;
    int lda, ldb, k, a_mn_major, b_mn_major;
    int a_koff; /* first K index of this segment inside `a` (a column / row offset that keeps `a` 16-byte aligned) */
} tcar_gemm_seg;
int tcar_gemm_tf32(const tcar_gemm_seg* segs, int nseg, int M, int N, const float* bias, int act, float* C, int ldc,
                   int accumulate, int precise, int splits, float* part, void* stream);
/* Several independent problems in ONE launch (each launch costs ~7 us of fixed latency on the GPU): e.g. all weight
 * gradients that consume dU1 / dU2.  Split problems of one group need disjoint `part` buffers. */
#define TCAR_GEMM_MAX_GROUP 8
typedef struct tcar_gemm_problem {
    tcar_gemm_seg segs[3];
    int nseg, M, N;
    const float* bias;
    int act;
    float* C;
    int ldc, accumulate, precise, splits;
    float* part;
    float* C2;      /* optional second destination: rows >= c2_row0 of the result are ALSO written to               */
    int c2_row0;    /* C2[(row - c2_row0) * ldc + col] (W_c's gradient is the bottom half of X^T dU1: no copy kernel) */
} tcar_gemm_problem;
int tcar_gemm_tf32_group(const tcar_gemm_problem* probs, int nprob, void* stream);
int tcar_gemm_tf32_splits(int M, int N, int k_total, int want);
long long tcar_gemm_tf32_part_elems(int M, int N, int splits);
/* hi/lo split of the dense weights into padded layouts: table [ntensors][7] = {src_off, rows, cols, dst_off,
 * dst_pitch, src2_off, src2_row0} (int32, device); w = theta[src] (+ theta[src2] for rows >= src2_row0 when
 * src2_off >= 0 -- folds W_c into the bottom half of W_in); hi = tf32(w) rounded to nearest, lo = tf32(w - hi);
 * pad columns zero. */
int tcar_prep_weights(const float* theta, const int32_t* table, int ntensors, float* hi, float* lo, void* stream);

/* (5b) deterministic scatter-add of the sparse item-row gradients into the dense g_item [N+1,256]:
 *      clicked rows (clip Jacobian of dXi), label rows (-a_ic[:, :250]) and negative rows (coef a_ic[:, :250]).
 *      Three passes: claim a hash slot per row and count its entries; rows with ONE entry are updated in place
 *      (128-bit read-modify-write), rows shared by several entries accumulate in exact int64 fixed point (2^-40),
 *      so the result never depends on the order in which duplicates arrive; finally the shared rows are applied.
 *      Scratch, all restored on exit: hash_keys [hash_size] int32 = -1, hash_cnt [hash_size] int32 = 0, hash_acc
 *      [hash_size][256] int64 = 0; entry_slot [B*T + B + B*Nn] int32 (no initial state).  hash_size: power of two,
 *      >= 2 x entries.  slot_sq [hash_size] (nullable) receives, per slot, the change of ||g_item||^2 caused by the
 *      rows of that slot (0 for empty slots) -- input of tcar_sqnorm_combine. */
int tcar_scatter_add_rows(const int32_t* seq, const int32_t* label, const int32_t* neg, const float* dXi,
                          const float* a_ic, const float* coef, const float* item, float* g_item,
                          int32_t* hash_keys, int32_t* hash_cnt, long long* hash_acc, int32_t* entry_slot,
                          float* slot_sq, int hash_size, int B, int T, int Nn, void* stream);

/* Same, restricted to the table rows [row_lo, row_hi) of one catalog shard: entries whose row lies outside are
 * ignored (the rank that owns them applies them).  Rows are table rows (1-based item ids: seq as is, label + 1,
 * neg + 1).  Called once per source rank with that rank's all-gathered (seq, label, neg, dXi, a_ic, coef). */
int tcar_scatter_add_rows_range(const int32_t* seq, const int32_t* label, const int32_t* neg, const float* dXi,
                                const float* a_ic, const float* coef, const float* item, float* g_item,
                                int32_t* hash_keys, int32_t* hash_cnt, long long* hash_acc, int32_t* entry_slot,
                                float* slot_sq, int hash_size, int B, int T, int Nn, int row_lo, int row_hi,
                                void* stream);

/* (5c) per-tensor squared L2 norms (for tf.clip_by_norm, model_combine.py:158-160). seg_off [nseg+1], every
 *      segment start 16-byte aligned and zero padded to a multiple of 4 floats.  tcar_sqnorm_segments writes
 *      sqnorm [nseg][TCAR_NORM_SPLIT] partial sums (tcar_adam_small adds them in index order). */
int tcar_sqnorm_segments(const float* flat, const int32_t* seg_off, float* sqnorm, int nseg, void* stream);
int tcar_sqnorm_big(const float* x, float* partial, float* sqnorm, long long n, void* stream);
/* squared norm of the item gradient WITHOUT re-reading it: out[0] = sum(a[0..na)) + sum(b[0..nb)) in a fixed order,
 * a = per-CTA sums of squares written by tcar_score_bwd_i, b = slot_sq of tcar_scatter_add_rows. */
int tcar_sqnorm_combine(const float* a, int na, const float* b, int nb, float* out, void* stream);
/* tcar_sqnorm_segments + tcar_sqnorm_combine + `step[0] += 1` in ONE launch (the single-GPU train step): item_part
 * [TCAR_NORM_SPLIT] floats and ticket [1] int32 (zero before the first use, left at zero) are scratch.  The two halves
 * can also be launched separately (they are independent): sqnorm_item == NULL -> small tensors (+ step) only;
 * nseg == 0 -> item norm only (step must be NULL). */
int tcar_update_norms(const float* flat, const int32_t* seg_off, float* sqnorm_small, int nseg, const float* a, int na,
                      const float* b, int nb, float* sqnorm_item, float* item_part, int32_t* ticket, int32_t* step,
                      void* stream);

/* Debug aid (not thread-safe, not used on the product path): when trace_buf != NULL every CTA of the following
 * tcar_gemm_tf32* launches writes 8 clock64() stamps to trace_buf[8 * cta + k]: 0 start, 1 prologue done, 2 last TMA
 * issued, 3 first stage landed, 4 last MMA committed, 5 accumulator ready, 6 epilogue stores issued, 7 end. */
int tcar_debug_gemm_trace(long long* trace_buf);

/* (5d) clip_by_norm + TF-flavoured Adam (model_combine.py:155-163): lr_t = lr sqrt(1-b2^t)/(1-b1^t),
 *      theta -= lr_t m / (sqrt(v) + eps).  `step` [1] int32 on device holds t (already incremented). */
int tcar_adam_small(float* theta, float* m, float* v, const float* g, const int32_t* seg_off, const float* sqnorm,
                    int nseg, const int32_t* step, float lr, float max_grad, void* stream);
/* item table rows [row0, row0 + nrows) of [N+1,256] (the pointers address the first row of the slice; iext is the
 * whole operand): also refreshes the item columns of Iext (bf16) in the same pass.  Whole table: row0 = 0,
 * nrows = N + 1; data-parallel training updates one contiguous slice per rank (parallel.py).
 * iext_bf16 may be NULL (no refresh: a slice that runs past row N, followed by tcar_refresh_iext_items).
 * The six pad columns of the 256-float pitch are not touched.  `row_flags` (optional, [N+1] int32, indexed by
 * absolute row): rows whose flag equals the step number t were already updated by tcar_adam_item_rows and are skipped.
 * `ctas_per_sm`: grid = 148 x ctas_per_sm CTAs of 256 threads (0 = 64).  Many short-lived CTAs measured faster than
 * 16 long ones per SM (445 vs 510 us under ncu), and they let kernels of a higher-priority stream (the next batch's
 * session forward, Seq2SeqAttNN.train_step) into the SM resources retiring CTAs free within a few microseconds. */
int tcar_adam_item(float* item, float* m, float* v, const float* g, const float* sqnorm, const int32_t* step,
                   float lr, float max_grad, void* iext_bf16, int row0, int nrows, const int32_t* row_flags,
                   int ctas_per_sm, void* stream);
/* The same update (same arithmetic, so bit-identical results) for the rows the NEXT batch will gather before the
 * table-wide pass has finished: rows seq[0..n_seq) and label[0..n_label) + 1 of the whole [n_rows,256] table.  Each
 * listed row is claimed once by writing t into row_flags[row]; duplicates and out-of-range ids are ignored. */
int tcar_adam_item_rows(float* item, float* m, float* v, const float* g, const float* sqnorm, const int32_t* step,
                        float lr, float max_grad, void* iext_bf16, const int32_t* seq, int n_seq,
                        const int32_t* label, int n_label, int32_t* row_flags, int n_rows, void* stream);
/* The same for the batches of several ranks (catalog-sharded step with look-ahead): ids = packed batches [7*B*T idx |
 * 2*B ctx | B label | B*Nn neg] of rank g at ids + g * ids_stride with B = n_rows[g] (HOST array); rows seq, label + 1
 * and neg + 1 that fall into the caller's table rows [row_lo, row_hi) are updated (item / m / v / g address row 0 of the
 * whole table), all others are ignored and NOT claimed in row_flags. */
int tcar_adam_item_rows_groups(float* item, float* m, float* v, const float* g, const float* sqnorm,
                               const int32_t* step, float lr, float max_grad, void* iext_bf16, const int32_t* ids,
                               long long ids_stride, const int* n_rows, int groups, int T, int Nn, int32_t* row_flags,
                               int row_lo, int row_hi, void* stream);
/* item columns of Iext from the fp32 item table (after all-gathering slices updated by other ranks). */
int tcar_refresh_iext_items(const float* item, void* iext_bf16, int N, void* stream);

/* (7) peer memory of the catalog-sharded train step (single node, NVLink / NVSwitch; SURVEY 8e row 2, 8f-3).  Every
 *     rank owns the fp32 master copy of a contiguous range of item-table rows; the rows a rank's sessions read are
 *     loaded directly from the owner's HBM.  The three functions below are the only ones of this library that are
 *     synchronous host calls without a stream (they wrap cudaIpc*): export a device allocation (any pointer inside a
 *     cudaMalloc'ed block: `handle` receives the 64-byte IPC handle of the block, `offset` the pointer's offset in
 *     it), open another rank's export, close it again. */
#define TCAR_MAX_PEERS 16
#define TCAR_PEER_HANDLE_BYTES 64
int tcar_peer_export(const void* ptr, unsigned char* handle, long long* offset);
int tcar_peer_open(const unsigned char* handle, long long offset, void** ptr);
int tcar_peer_close(void* ptr, long long offset);
/* table[row] = peers[owner(row)][row] for the table rows one batch reads -- seq[0..B*T) as is, label[0..B) + 1,
 * neg[0..B*Nn) + 1 -- that are owned by OTHER ranks (256-float rows).  peers [G] and row_bounds [G+1] are HOST arrays
 * (rank g owns rows [row_bounds[g], row_bounds[g+1])); seq / label / neg are device arrays.  The caller orders this
 * after the owners' updates (a collective on the same stream). */
int tcar_peer_fetch_rows(const int32_t* seq, const int32_t* label, const int32_t* neg, int B, int T, int Nn,
                         const void* const* peers, const int32_t* row_bounds, int G, int self, float* table,
                         void* stream);

/* (8) session groups of the catalog-sharded step.  Every rank scores the sessions of ALL ranks against its own item
 *     range: group g = rank g's sessions, n_rows[g] <= 512 of them (HOST array; 0 = group absent), operands of
 *     consecutive groups `*_stride` ELEMENTS apart.  Each function is the loop over groups around the single-group entry
 *     point of the same name (one host call per phase).
 *     fwd:   mode 0 of tcar_score_fwd with cluster as given.
 *     bwd_q: tcar_score_bwd_q per group into dq + g * dq_stride; with rowsum_part != NULL the group's softmax partial
 *            sums (fixed-order sum over n_tiles, as tcar_ce_finish) are stored in the zero pad column 639 of its dQ
 *            rows, so that one reduce-scatter delivers dQ and sum exp to the sessions' rank.
 *     bwd_i: one launch over all present groups (tcar_score_bwd_i_multi); sq_partial (nullable) = sums of squares of
 *            the complete dense gradient.  (More than TCAR_MAX_PEERS groups: the first present group overwrites
 *            g_item, later ones accumulate through tcar_score_bwd_i_acc.)
 *     scatter: tcar_scatter_add_rows_range per group; ids = packed batches [7*B*T idx | 2*B ctx | B label | B*Nn neg],
 *            payload = [a_ic 512x500 | coef 512 | dXi B*T x 256] floats; slot_sq (nullable): [groups][hash_size]. */
int tcar_score_fwd_groups(const void* q_bf16, long long q_stride, const float* c_ref, long long c_stride,
                          const void* iext_bf16, void* e_out, long long e_stride, float* rowsum_part,
                          long long part_stride, const int* n_rows, int groups, int n_items, int n_pad, int cluster,
                          void* stream);
/* bwd_q of ALL present groups in one launch (what tcar_score_bwd_q_groups uses when more than one group is present):
 * E_g at e_bf16 + g * e_stride, dq [groups][512][640] back to back, part >= tcar_score_bwd_q_multi_part_elems(groups)
 * floats of scratch.  With R x 4 m-tiles of 128 session rows the reduction over the items needs only 148 / (8 R) splits:
 * long K loops and one small split reduction instead of R short launches. */
long long tcar_score_bwd_q_multi_part_elems(int groups);
int tcar_score_bwd_q_multi(const void* e_bf16, long long e_stride, const void* iext_bf16, float* part, float* dq,
                           const int* n_rows, int groups, int n_pad, void* stream);
int tcar_score_bwd_q_groups(const void* e_bf16, long long e_stride, const void* iext_bf16, float* part, float* dq,
                            long long dq_stride, const float* rowsum_part, long long part_stride, int n_tiles,
                            const int* n_rows, int groups, int n_pad, void* stream);
int tcar_score_bwd_i_groups(const void* e_bf16, long long e_stride, const void* qs_bf16, long long qs_stride,
                            float* g_item, float* sq_partial, const int* n_rows, int groups, int n_items, int n_pad,
                            void* stream);
int tcar_scatter_add_rows_groups(const int32_t* ids, long long ids_stride, const float* payload,
                                 long long payload_stride, const float* item, float* g_item, int32_t* hash_keys,
                                 int32_t* hash_cnt, long long* hash_acc, int32_t* entry_slot, float* slot_sq,
                                 int hash_size, const int* n_rows, int groups, int T, int Nn, int row_lo, int row_hi,
                                 void* stream);
/* The same scatter-add for ALL groups against one hash table in three launches (count over every group first, so
 * "touched once" is a global property; shared rows add up in order-independent fixed point): hash_size >= 2 x the
 * entries of all groups together, entry_slot >= groups x (largest group's entries) words, slot_sq ONE block of
 * hash_size floats (nullable).  Same arguments otherwise; TCAR_ERR_ARG when the table is too small. */
int tcar_scatter_add_rows_multi(const int32_t* ids, long long ids_stride, const float* payload,
                                long long payload_stride, const float* item, float* g_item, int32_t* hash_keys,
                                int32_t* hash_cnt, long long* hash_acc, int32_t* entry_slot, float* slot_sq,
                                int hash_size, const int* n_rows, int groups, int T, int Nn, int row_lo, int row_hi,
                                void* stream);

/* Softmax overflow guard for the session groups of a catalog-sharded step (see tcar_score_fwd_guarded):
 *   tcar_score_fwd_groups_guarded(..., rowmax_part, NULL, ...)     pass 1, also leaves per-block exponent maxima
 *   tcar_rowmax_groups                                             rowmax [groups][512] = max over the blocks (1 launch)
 *   -- across ranks: all-reduce(MAX) of rowmax, every owner must shift a session row by the same amount --
 *   tcar_score_fwd_groups_guarded(..., NULL, rowmax, ...)          pass 2, empty launches unless a row is above the limit
 * and the caller adds rowmax[b] ln 2 to log(sum) for the rows above TCAR_EXP_LIMIT2. */
int tcar_score_fwd_groups_guarded(const void* q_bf16, long long q_stride, const float* c_ref, long long c_stride,
                                  const void* iext_bf16, void* e_out, long long e_stride, float* rowsum_part,
                                  long long part_stride, float* rowmax_part, const float* rowmax, const int* n_rows,
                                  int groups, int n_items, int n_pad, int cluster, void* stream);
/* All groups in ONE launch (what tcar_score_fwd_groups_guarded does for more than one group with CTA pairs): work unit =
 * (256-session row block, 256-item tile), every CTA pair takes a contiguous run of units and swaps its resident session
 * rows when the run crosses into the next row block.  Train mode only. */
int tcar_score_fwd_multi(const void* q_bf16, long long q_stride, const float* c_ref, long long c_stride,
                         const void* iext_bf16, void* e_out, long long e_stride, float* rowsum_part,
                         long long part_stride, float* rowmax_part, const float* rowmax, const int* n_rows, int groups,
                         int n_items, int n_pad, void* stream);
/* The same in eval mode: chunk / tile maxima of group g at chunkmax + g * cm_stride / tilemax + g * tm_stride. */
int tcar_score_fwd_multi_eval(const void* q_bf16, long long q_stride, const float* c_ref, long long c_stride,
                              const void* iext_bf16, float* chunkmax, long long cm_stride, float* tilemax,
                              long long tm_stride, float* rowsum_part, long long part_stride, float* rowmax_part,
                              const float* rowmax, long long rowmax_stride, const int* n_rows, int groups, int n_items,
                              int n_pad, void* stream);
int tcar_rowmax_groups(const float* rowmax_part, long long part_stride, float* rowmax, int n_tiles, const int* n_rows,
                       int groups, void* stream);
/* Pass 1 / 2 of tcar_ce_finish_guarded for several groups in one launch: group g's partials at + g * part_stride, its
 * sumexp / rowmax vectors at + g * out_stride (catalog-sharded evaluation; the queries' owner combines the sums). */
int tcar_ce_finish_groups(const float* rowsum_part, const float* rowmax_part, long long part_stride, float* sumexp,
                          float* rowmax, long long out_stride, int n_tiles, const int* n_rows, int groups, int pass,
                          void* stream);

/* (6) evaluation (model_combine.py:283-306, util.py:8-18): select the 32 best 128-item tiles per query from tilemax,
 *     then the 32 best 8-item chunks among their 512 chunks from chunkmax (exactly the 32 best chunks overall, ties
 *     to the lower index), re-score their 256 items exactly in fp32, return top-20 ids/scores ordered by (score desc, id asc) and
 *     n_greater[b] = #candidates scoring strictly above the label (rank-1 whenever rank <= 20).
 *     chunkmax covers the N local items of this catalog shard; item/content/mwdhm are the GLOBAL fp32 tables,
 *     label holds global 0-based ids and item_offset is the global id of local item 0.
 *     Certification: cat_stats[2] (tcar_catalog_stats over the items this call scores, or any superset) bounds the
 *     bf16-GEMM error of every chunk maximum; a query whose best un-re-scored chunk could still reach its 20th exact
 *     score is flagged in uncertain[b] (1 / 0) with the bound tau[b], and tcar_eval_topk_widen completes it.  Together
 *     the two calls return the exact top-20 (np.argsort(pred)[::-1][:20], model_combine.py:301, ties to the lower id)
 *     and the exact rank whenever rank <= 20 -- not "with high probability".  cat_stats = NULL skips the certification
 *     (uncertain / tau unused). */
int tcar_eval_topk_certified(const float* chunkmax, const float* tilemax, const float* a_ic, const float* Tq,
                             const float* item, const float* content, const int32_t* mwdhm, const int32_t* label,
                             int32_t* top_ids, float* top_scores, int32_t* n_greater, int B, int N, int n_pad,
                             int item_offset, const float* cat_stats, int32_t* uncertain, float* tau, void* stream);
/* The two halves of tcar_eval_topk_certified for the catalog-sharded evaluation, where the chunk maxima of an item
 * range and the queries' owner live on different GPUs (Seq2SeqAttNN.eval_round):
 *   tcar_eval_select   (item range)  sel_vals / sel_ids [B][TCAR_EVAL_NSEL]: the range's 32 best chunks per query as
 *                      (bf16-GEMM chunk maximum, GLOBAL chunk id = (item_offset + local item) / 8; -1 = none), and a
 *                      33rd entry (id -2) whose value bounds every chunk of the range that is NOT listed.  No re-scoring.
 *   tcar_eval_rescore  (query owner) `lists` such lists per query, list_stride words apart: the 32 best entries overall
 *                      are re-scored exactly from the fp32 tables (global ids, N_total items), top-20 / n_greater as in
 *                      tcar_eval_topk_certified; the 33rd best value bounds everything else, queries it cannot
 *                      certify are flagged (uncertain, tau) for tcar_eval_topk_widen on every item range.
 *                      lists * 33 <= 512. */
int tcar_eval_select(const float* chunkmax, const float* tilemax, float* sel_vals, int32_t* sel_ids, int B, int N,
                     int n_pad, int item_offset, void* stream);
int tcar_eval_rescore(const float* sel_vals, const int32_t* sel_ids, int lists, long long list_stride, const float* a_ic,
                      const float* Tq, const float* item, const float* content, const int32_t* mwdhm,
                      const int32_t* label, int32_t* top_ids, float* top_scores, int32_t* n_greater, int B, int N_total,
                      const float* cat_stats, int32_t* uncertain, float* tau, void* stream);
/* Second stage: for every flagged query, re-scores ALL chunks whose maximum reaches tau[b] (any number of them -- in
 * the limit a full exact scan, so the work of one query is spread over TCAR_WIDEN_SPLITS CTAs; the CTA that finishes
 * last merges their partial lists) and rewrites its top_ids / top_scores / n_greater; certified queries are untouched
 * (their CTAs return).  workspace: tcar_eval_topk_widen_ws_bytes(1) bytes (x groups for the _groups form), ZERO before
 * the first call (it ends with one ticket counter per query, which every call leaves at zero again). */
long long tcar_eval_topk_widen_ws_bytes(int groups);
int tcar_eval_topk_widen(const float* chunkmax, const float* tilemax, const float* a_ic, const float* Tq,
                         const float* item, const float* content, const int32_t* mwdhm, const int32_t* label,
                         const int32_t* uncertain, const float* tau, int32_t* top_ids, float* top_scores,
                         int32_t* n_greater, int B, int N, int n_pad, int item_offset, void* workspace, void* stream);
/* tcar_eval_select / tcar_eval_topk_widen for the session groups of a catalog-sharded evaluation round in ONE launch
 * (pair) each: group g has n_rows[g] queries (HOST array); its chunk / tile maxima lie cm_stride / tm_stride floats
 * apart; its a_ic / Tq / label planes q_stride 32-bit words apart (one exchange block per group); its (uncertain, tau)
 * vectors flag_stride words apart; its outputs out_stride words apart. */
int tcar_eval_select_groups(const float* chunkmax, long long cm_stride, const float* tilemax, long long tm_stride,
                            float* sel_vals, int32_t* sel_ids, long long out_stride, const int* n_rows, int groups,
                            int N, int n_pad, int item_offset, void* stream);
int tcar_eval_topk_widen_groups(const float* chunkmax, long long cm_stride, const float* tilemax, long long tm_stride,
                                const float* a_ic, const float* Tq, const int32_t* label, long long q_stride,
                                const float* item, const float* content, const int32_t* mwdhm,
                                const int32_t* uncertain, const float* tau, long long flag_stride, int32_t* top_ids,
                                float* top_scores, int32_t* n_greater, long long out_stride, const int* n_rows,
                                int groups, int N, int n_pad, int item_offset, void* workspace, void* stream);
/* out2[0] = max ||[item | content] row||_2, out2[1] = max ||row - bf16(row)||_2 over table rows [row_lo, row_hi)
 * (row = item id + 1).  Needed again only after the item table changed. */
int tcar_catalog_stats(const float* item, const float* content, int row_lo, int row_hi, float* out2, void* stream);

/* merge G per-shard top-20 lists [G][B][20] into the global top-20 (score desc, id asc). */
int tcar_topk_merge(const int32_t* ids, const float* scores, int32_t* out_ids, float* out_scores, int G, int B,
                    void* stream);
/* The whole reduction of the catalog-sharded evaluation in one launch: `blocks` = G result blocks (layout
 * TCAR_EVAL_OFF_*, `block_words` 32-bit words apart -- the receive buffer of ONE all-gather / all-to-all) ->
 * global top-20 (score desc, id asc), summed rank counts, and ce[b] = logsumexp(S_b) - S_b[label] combined from the
 * shards' partial sums and their own exponent shifts (util.py:14, model_combine.py:145,301). */
int tcar_eval_merge(const void* blocks, long long block_words, int32_t* out_ids, float* out_scores, int32_t* out_ngt,
                    float* out_ce, int G, int B, void* stream);
/* Pieces of the same reduction for the two-stage sharded evaluation: the cross loss from G ranges' (sumexp, rowmax)
 * vectors `gstride` words apart; and the list / rank-count merge restricted to the queries flagged in only_if[b] (the
 * widening pass of every item range), all other queries keep what out_* hold. */
int tcar_eval_ce_combine(const float* sumexp, const float* rowmax, long long gstride, float* out_ce, int G, int B,
                         void* stream);
int tcar_eval_merge_flagged(const void* blocks, long long block_words, const int32_t* only_if, int32_t* out_ids,
                            float* out_scores, int32_t* out_ngt, int G, int B, void* stream);

/* (6b) candidate re-ranking: session b's list is cand_ids[cand_off[b] .. cand_off[b+1]) (0-based item ids, at most
 *      max_len <= TCAR_RERANK_MAXL entries; duplicates allowed).  a_ic / Tq are the session vectors of
 *      tcar_build_query; item / content / mwdhm the fp32 tables of the full-catalog evaluation.
 *        scores [nnz]   exact fp32 score of cand_ids[j], in input order: the arithmetic of the top-20 re-scoring
 *                       (tcar_eval_topk_certified), so a candidate scores bit for bit what the full-catalog top-20
 *                       reports for it (model_combine.py:138);
 *        ranked [nnz]   each list's ids ordered by (score desc, id asc, input position asc);
 *      with label != NULL (label[b] = the positive, every other entry of the list is a negative):
 *        label_rank [B] 1 + #(negatives scoring strictly above the label): the label wins ties (util.py:14);
 *        auc [B]        (#(negatives below) + 1/2 #(negatives equal)) / #negatives, NaN without negatives.
 *      An id outside [0, N) is not read and scores NaN; a label outside [0, N) gives label_rank 0 and auc NaN; a list
 *      longer than max_len is not processed (outputs left as they are).  B = 0 launches nothing. */
#define TCAR_RERANK_MAXL 2048
int tcar_rerank(const float* a_ic, const float* Tq, const float* item, const float* content, const int32_t* mwdhm,
                const int32_t* cand_off, const int32_t* cand_ids, const int32_t* label, int B, int N, int max_len,
                float* scores, int32_t* ranked, int32_t* label_rank, float* auc, void* stream);

/* (6c) top-K recommendation: the exact top-K of the whole catalog per session, without the excluded ids.
 *      chunkmax / tilemax: the eval-mode scoring GEMM (tcar_score_fwd mode 1) over the N items for these B queries;
 *      a_ic / Tq / item / content / mwdhm as for tcar_eval_topk_certified; cat_stats: tcar_catalog_stats over the N
 *      items.
 *      Exclusions of session b (0-based ids; duplicates and ids outside [0, N) allowed): x_ids[x_off[b] .. x_off[b+1])
 *      when x_off != NULL, and clicks[b*T .. b*T+T) - 1 when clicks != NULL (the 1-based click ids of the packed
 *      batch, T clicks per session); at most TCAR_RECOMMEND_MAXX entries in all, a session with more is not processed
 *      (outputs left as they are).
 *        ids [B][K]       item ids ordered by (exact score desc, id asc); -1 past the end of a small catalog
 *        scores [B][K]    their exact fp32 scores (the arithmetic of the top-20 re-scoring, so bit for bit what
 *                         eval_step and tcar_rerank report for the same item); -inf past the end
 *        rescored [B]     (nullable) items re-scored exactly: the width of the band the error bound left open.
 *      1 <= K <= TCAR_RECOMMEND_MAXK.  workspace: tcar_recommend_ws_bytes(B) bytes (a buffer sized for B serves every
 *      smaller B), ZERO before the first call (it starts with TCAR_QROWS ticket counters that every call leaves at
 *      zero again).  Two launches; B = 0 launches nothing. */
#define TCAR_RECOMMEND_MAXK 256
#define TCAR_RECOMMEND_MAXX 1024
long long tcar_recommend_ws_bytes(int B);
int tcar_recommend(const float* chunkmax, const float* tilemax, const float* a_ic, const float* Tq, const float* item,
                   const float* content, const int32_t* mwdhm, const float* cat_stats, const int32_t* x_off,
                   const int32_t* x_ids, const int32_t* clicks, int T, int B, int N, int n_pad, int K, void* workspace,
                   int32_t* ids, float* scores, int32_t* rescored, void* stream);
/* The same restricted to a publish-time window per session: the exact top-K, by (score desc, id asc), of the items
 * with win_lo[b] <= item_time[n] <= win_hi[b] that are not excluded.  chunkmax / tilemax must come from
 * tcar_score_fwd_window with the same item_time / win_lo / win_hi (the masked maxima keep the selection exact); the
 * scores are the same exact fp32 scores as tcar_recommend's.  A window with fewer than K eligible items pads with
 * -1 / -inf; rescored counts in-window items only.  Same workspace, limits and launches as tcar_recommend. */
int tcar_recommend_window(const float* chunkmax, const float* tilemax, const float* a_ic, const float* Tq,
                          const float* item, const float* content, const int32_t* mwdhm, const float* cat_stats,
                          const int32_t* x_off, const int32_t* x_ids, const int32_t* clicks, int T, int B, int N,
                          int n_pad, int K, void* workspace, int32_t* ids, float* scores, int32_t* rescored,
                          const int32_t* item_time, const int32_t* win_lo, const int32_t* win_hi, void* stream);
/* The same ranked by the decayed score r = s - rate[b] * age of tcar_score_fwd_decay: the exact top-K, by (r desc,
 * id asc), of the non-excluded items (and with win_lo / win_hi, both given or both NULL, of the in-window ones);
 * scores holds r, from the exact fp32 score s of tcar_recommend and the same p as the GEMM epilogue.  chunkmax /
 * tilemax must come from tcar_score_fwd_decay with the same item_time / t_ref / rate / window.  Padding and rescored
 * as tcar_recommend_window.  Same workspace, limits and launches as tcar_recommend. */
int tcar_recommend_decay(const float* chunkmax, const float* tilemax, const float* a_ic, const float* Tq,
                         const float* item, const float* content, const int32_t* mwdhm, const float* cat_stats,
                         const int32_t* x_off, const int32_t* x_ids, const int32_t* clicks, int T, int B, int N,
                         int n_pad, int K, void* workspace, int32_t* ids, float* scores, int32_t* rescored,
                         const int32_t* item_time, const int32_t* t_ref, const float* rate, const int32_t* win_lo,
                         const int32_t* win_hi, void* stream);
/* The same with at most C items of one category and a per-session set of allowed categories: the exact top-K, by
 * (score desc, id asc), of the non-excluded items of the allowed categories, in which an item that has C better items
 * of its category in the list is left out (C >= K: no cap).  G <= TCAR_RECOMMEND_MAXG categories, item_cat [N] the
 * code in [0, G) of every (original) item id.  The catalog in category order: perm [N'] the original id at position p
 * (-1 on a pad), every category padded to whole TCAR_CHUNK chunks by repeating its last item; category g owns the
 * chunks cat_chunk_off[g] .. cat_chunk_off[g + 1] (cat_chunk_off [G + 1], cat_chunk_off[G] = N' / TCAR_CHUNK).
 * chunkmax: tcar_score_fwd mode 1 over iext_cat (row p = the iext row of perm[p], a pad's that of the item it repeats)
 * with n_items = N' and this n_pad.  Allowed codes of session b: a_codes[a_off[b] .. a_off[b + 1]) (in [0, G),
 * duplicates allowed; an empty list returns -1 / -inf throughout); a_off == NULL allows every category.  Exclusions,
 * outputs and limits as tcar_recommend (ids are original ids; rescored counts items scored exactly).  workspace:
 * tcar_recommend_category_ws_bytes(B) bytes, ZERO before the first call (tcar_recommend's layout, then per-category
 * thresholds).  Two launches; B = 0 launches nothing. */
#define TCAR_RECOMMEND_MAXG 1024
long long tcar_recommend_category_ws_bytes(int B);
int tcar_recommend_category(const float* chunkmax, const float* a_ic, const float* Tq, const float* item,
                            const float* content, const int32_t* mwdhm, const float* cat_stats, const int32_t* x_off,
                            const int32_t* x_ids, const int32_t* clicks, int T, int B, int n_pad, int K,
                            const int32_t* perm, const int32_t* item_cat, const int32_t* cat_chunk_off, int G,
                            const int32_t* a_off, const int32_t* a_codes, int C, void* workspace, int32_t* ids,
                            float* scores, int32_t* rescored, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* TCAR_B200_H_ */
