/*
 * e2e_asr_b200.h — C ABI of the B200-native joint CTC/attention(+RNNLM)
 * beam-search decode path (libe2e_asr_b200.so).
 *
 * The reference (DanielLin94144/E2E-ASR-Pytorch) is pure Python: it has no FFI
 * of its own, so each entry point below names the reference code it replaces
 * (paths relative to the reference root) and INTEGRATION.md shows the ctypes
 * binding a maintainer would add.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless its name ends in _host;
 *   - the caller owns every buffer; the library allocates nothing, keeps no
 *     state between calls except the per-thread error string, and never
 *     synchronises: all work is enqueued on `stream` (a cudaStream_t);
 *   - return value: 0 on success, a negative E2E_ERR_* code otherwise
 *     (e2e_last_error() then describes it).  Nothing throws across the ABI;
 *   - data-dependent failures of the reference (IndexError / ValueError) are
 *     reported asynchronously through the `status` words (E2E_STATUS_* bits),
 *     which the host reads back when it needs the result;
 *   - "utterance" u in [0,U), beam "slot" b in [0,B), "hypothesis" n = u*B+b,
 *     "candidate" j in [0,C), prefix-state "lane" l = b*C+j inside an utterance.
 *
 * Layouts (all fp32 unless noted)
 *   x        [Tmax][U][Vp]        frame-major CTC log-posteriors, Vp = e2e_padded_vocab(V)
 *   r        [U][Tmax][lanes][2]  prefix states: [..][0] non-blank-ending, [..][1] blank-ending
 *   history  [Smax][U][B]         back-pointers / tokens / per-token scores of every step
 */
#ifndef E2E_ASR_B200_H
#define E2E_ASR_B200_H

#ifdef __cplusplus
extern "C" {
#endif

#define E2E_ABI_VERSION 1

/* constants of the reference that are part of parity */
#define E2E_CTC_LOGZERO   (-100000000.0f) /* src/ctc.py:12   */
#define E2E_CTC_BLANK     0               /* src/ctc.py:13   */
#define E2E_CTC_EOS       1               /* src/ctc.py:14   */
#define E2E_DEC_LOG_ZERO  (-10000000.0f)  /* src/decode.py:11 */

/* return codes */
#define E2E_OK              0
#define E2E_ERR_ARG        (-1)  /* invalid argument (null pointer, size <= 0, bad alignment, ...) */
#define E2E_ERR_LAUNCH     (-2)  /* CUDA launch / runtime error (message has the CUDA string)     */
#define E2E_ERR_UNSUPPORTED (-3) /* size outside what the kernels are built for                   */

/* bits of the per-utterance status words */
#define E2E_STATUS_PREFIX_TOO_LONG   1 /* len(prefix) > T: reference raises IndexError, src/ctc.py:85          */
#define E2E_STATUS_TOKEN_NOT_CAND    2 /* beam winner outside the CTC candidates: ValueError, src/decode.py:252 */

/* flags of e2e_ctc_prefix_score */
#define E2E_PREFIX_FULL           1 /* full_compute semantics (src/ctc.py:29-66): candidates are 0..V-1 */
#define E2E_PREFIX_SKIP_DEAD_ROWS 2 /* do not write state rows t < start (they are never read back by
                                       the batched beam search; the drop-in scorer always writes them) */
#define E2E_PREFIX_FAST_MATH      4 /* MUFU ex2/lg2 log-add-exp (abs. error ~3e-7) instead of the default
                                       table-based one (within one fp32 rounding of exact)              */
#define E2E_PREFIX_LIBM_MATH      8 /* CUDA expf/log1pf log-add-exp: slow cross-check of the default     */
#define E2E_PREFIX_ROW_COPIES    16 /* stage posterior tiles with one bulk copy per row instead of one
                                       tensor-map box copy per tile (cross-check of the TMA path)       */
#define E2E_PREFIX_POLY_MATH     32 /* MUFU ex2 + degree-8 polynomial log-add-exp (no table; polynomial error
                                       3.3e-8; what BeamDecoder passes by default, see csrc/common.cuh)  */
#define E2E_PREFIX_POLY_ESTRIN   64 /* with E2E_PREFIX_POLY_MATH: evaluate the polynomial pairwise (shorter
                                       dependent chain, 2 more instructions)                             */

/* flags of e2e_beam_combine_prune */
#define E2E_BEAM_USE_CTC 1
#define E2E_BEAM_USE_LM  2

const char *e2e_last_error(void);
int e2e_abi_version(void);
/* Row pitch (in floats) of the posterior tensor for a vocabulary of V tokens:
 * V rounded up to a multiple of 4 so that every row is a 16-byte aligned bulk
 * copy source. */
int e2e_padded_vocab(int V);

/* (1) CTC posterior.  Replaces F.log_softmax(self.asr.ctc_layer(enc), dim=-1) minus
 * the Linear (src/decode.py:94-95; ctc_layer = Linear + ReLU, src/asr.py:29-32):
 *   x[t][u][v] = log_softmax_v( relu?(logits[u][t][v]) )     t < enc_len[u]
 * Rows t >= enc_len[u] and pad columns v in [V,Vp) are set to E2E_CTC_LOGZERO.
 * logits: [U][Tmax][V] row-major (the Linear's output).  enc_len may be NULL (= Tmax). */
int e2e_ctc_log_softmax(const float *logits, int U, int Tmax, int V, const int *enc_len,
                        int apply_relu, float *x, int Vp, void *stream);

/* State of the empty prefix.  Replaces CTCPrefixScore.init_state (src/ctc.py:19-27):
 *   r0[u][t][0][0] = logzero ; r0[u][t][0][1] = sum_{tau<=t} x[tau][u][blank]  (sequential fp32)
 * r0: [U][Tmax][1][2]. */
int e2e_ctc_init_state(const float *x, int Tmax, int U, int Vp, const int *enc_len,
                       float *r0, void *stream);

/* (2) Prefix scores of every (hypothesis, candidate) extension.  Replaces
 * CTCPrefixScore.cheap_compute (src/ctc.py:68-108) — and .full_compute
 * (src/ctc.py:29-66) with E2E_PREFIX_FULL — for all live hypotheses of all
 * utterances in one launch.
 *   r_prev     [U][Tmax][lanes_prev][2]  states written by the previous step (or r0, lanes_prev=1)
 *   prev_lane  [U*B]  lane of hypothesis n's own state inside r_prev
 *   last_tok   [U*B]  last token of hypothesis n's prefix (ignored when prefix_len[n]==0)
 *   prefix_len [U*B]  len(g) of hypothesis n
 *   n_live     [U]    live slots per utterance (slots 0..n_live-1); NULL = B everywhere
 *   cand       [U*B][C] candidate token ids (ignored with E2E_PREFIX_FULL, where C must equal V)
 *   psi        [U*B][C]            out: prefix log-probabilities
 *   r_out      [U][Tmax][B*C][2]   out: states of the extended prefixes
 *   status     [U]                 in/out: OR-ed E2E_STATUS_* bits (may be NULL)
 *   n_run      only utterances 0..n_run-1 are processed (<= 0: all U).  A batch sorted by
 *              decreasing length keeps its live utterances as a prefix, so finished ones cost nothing;
 *              U stays the stride of x / history.
 */
int e2e_ctc_prefix_score(const float *x, int Tmax, int U, int Vp, int V, const int *enc_len,
                         const float *r_prev, int lanes_prev,
                         const int *prev_lane, const int *last_tok, const int *prefix_len,
                         const int *n_live, const int *cand, int B, int C, int flags,
                         float *psi, float *r_out, int *status, int n_run, void *stream);

/* (2, beam-search form) ONE fused launch per decode step with LAZY state evaluation (SURVEY.md §7.2-5): the prefix
 * state of every live hypothesis is brought up to date (it was left uncomputed when the hypothesis was only a
 * candidate) and all B*C candidate extensions are scored.  Replaces CTCPrefixScore.cheap_compute (src/ctc.py:68-108)
 * as src/decode.py:131 calls it, together with the state hand-over of src/decode.py:250-254: the recurrence
 * (src/ctc.py:97-101) runs for the <= B hypotheses the beam kept instead of for all B*C candidates — same frames,
 * same order, same fp32 operations, hence the same values — and the candidates only run psi (src/ctc.py:103).
 *   r_prev      [U][Tmax][lanes_prev][2]  states of the PARENTS (previous step's r_out; the e2e_ctc_init_state
 *               buffer with lanes_prev = 1 at steps 0 and 1)
 *   parent_slot [U*B]  lane of hypothesis n's parent inside r_prev (e2e_beam_combine_prune's parent_slot; 0 at step 0)
 *   last_tok    [U*B]  last token of hypothesis n (the token that extended the parent)
 *   parent_tok  [U*B]  last token of the parent, -1 if the parent is the empty prefix (may be NULL while every
 *               prefix_len <= 1)
 *   prefix_len  [U*B]  len(g); all live hypotheses of an utterance have the same length (slot 0 is read).
 *               prefix_len == 0: the hypothesis is the empty prefix, its state is r_prev itself, r_out is not written
 *   n_live, cand, psi, status, n_run as e2e_ctc_prefix_score
 *   r_out       [U][Tmax][B][2]  out: states of the live hypotheses, rows t >= max(1, len-1) - 1 (earlier rows are
 *               log-zero by construction, never read back, and not written)
 * flags: 0 or E2E_PREFIX_POLY_MATH (| E2E_PREFIX_POLY_ESTRIN).  Needs ceil(B/8) + ceil(B*C/32) <= 32 warps per
 * utterance (e2e_ctc_prefix_step_supported). */
int e2e_ctc_prefix_step_supported(int Vp, int B, int C);
int e2e_ctc_prefix_step(const float *x, int Tmax, int U, int Vp, int V, const int *enc_len,
                        const float *r_prev, int lanes_prev,
                        const int *parent_slot, const int *last_tok, const int *parent_tok, const int *prefix_len,
                        const int *n_live, const int *cand, int B, int C, int flags,
                        float *psi, float *r_out, int *status, int n_run, void *stream);

/* (3a) Attention log-softmax statistics + CTC candidate pre-pruning.  Replaces
 * F.log_softmax(cur_prob) and cur_prob.topk(ctc_beam_size) (src/decode.py:122,129-130).
 *   att_logits [U*B][ld] decoder outputs (char_trans), row pitch ld >= V
 *   att_stats  [U*B][2]  out: (max_v logits, log sum_v exp(logits-max)) so that
 *                        log_softmax(v) = (logits[v]-max) - lse
 *   cand       [U*B][C]  out: ids of the C largest log-probs, best first (ties: lower id first);
 *                        C may be 0 (no CTC) in which case only the statistics are produced */
int e2e_beam_candidates(const float *att_logits, int ld, int U, int B, int V, int C,
                        const int *n_live, float *att_stats, int *cand, void *stream);

/* (3b) Score combine + <eos> threshold + top-k + length-normalised prune of one decode
 * step for every utterance.  Replaces src/decode.py:134-177 and Hypothesis.addTopk /
 * avgScore (src/decode.py:214-263).
 * Beam state (updated IN PLACE, all [U][B] unless noted):
 *   n_live [U], last_tok, prefix_len, score_sum (sequential fp32 sum of token scores),
 *   ctc_prob (psi of the hypothesis), prev_lane;
 *   n_active [U] (may be NULL) receives n_live for utterances that still have a step to run
 *   and 0 for the others — it is the `n_live` argument of the NEXT step's (2)/(3a) calls
 * Per-step outputs:
 *   parent_slot [U][B]  slot of each new hypothesis' parent (identity for idle utterances) — the
 *                       caller gathers decoder / LM / attention states with it
 *   hist_tok, hist_parent (int32) and hist_score (fp32): row `step` of [Smax][U][B]
 * Closed (<eos>-terminated) hypotheses are kept per utterance, stably sorted by mean score and
 * truncated to the best fin_cap (>= B, so nothing the final selection could return is lost):
 *   fin_count [U]; fin_step, fin_parent (int32), fin_sum, fin_score (fp32): [U][fin_cap]
 * Utterances with step >= max_len[u] are left untouched; only utterances 0..n_run-1 are visited
 * (<= 0: all U).
 *   parent_row, last_tok64 [U][B] int64 (either may be NULL): u*B + parent_slot and last_tok again, in the
 *   index type the caller's state gathers / embedding look-ups take, so that no conversion kernels are needed.
 *   parent_tok [U][B] int32 (may be NULL): the last token of each new hypothesis' PARENT (-1 for the empty prefix) —
 *   what e2e_ctc_prefix_step needs to tell a repeated token (src/ctc.py:89-91) when it builds the survivor's state.
 *   lm_logits may be NULL iff E2E_BEAM_USE_LM is clear; cand/psi iff E2E_BEAM_USE_CTC is clear. */
int e2e_beam_combine_prune(const float *att_logits, int ld_att, const float *att_stats,
                           const float *lm_logits, int ld_lm,
                           const int *cand, const float *psi,
                           int U, int B, int V, int C, int step,
                           const int *min_len, const int *max_len,
                           float ctc_weight, float lm_weight, float eos_threshold, int flags,
                           int *n_live, int *n_active, int *last_tok, int *prefix_len,
                           float *score_sum, float *ctc_prob, int *prev_lane,
                           int *parent_slot,
                           int *hist_tok, int *hist_parent, float *hist_score,
                           int *fin_count, int *fin_step, int *fin_parent, float *fin_sum, float *fin_score,
                           int fin_cap, int *status, int n_run,
                           long long *parent_row, long long *last_tok64, int *parent_tok, void *stream);

/* Final N-best selection + back-tracking.  Replaces src/decode.py:180-183 and
 * Hypothesis.outIndex (src/decode.py:279-281): closed hypotheses followed by the last
 * beam, stable-sorted by mean token score, best B kept.
 *   out_tok, out_score [U][B][out_cap]; out_len, out_avg [U][B]; out_n [U] */
int e2e_beam_finalize(int U, int B, const int *max_len,
                      const int *n_live, const float *score_sum,
                      const int *hist_tok, const int *hist_parent, const float *hist_score,
                      const int *fin_count, const int *fin_step, const int *fin_parent,
                      const float *fin_sum, const float *fin_score, int fin_cap,
                      int *out_tok, float *out_score, int *out_len, float *out_avg, int *out_n,
                      int out_cap, void *stream);

/* (e) Ragged N-best pack for the one all-gather of the utterance-sharded decode (SURVEY §8e; it takes the place of
 * the per-utterance result lists joblib returns to the parent process, bin/test_asr.py:138-139): the N-best of U
 * decoded utterances (e2e_beam_finalize's outputs, row pitch cap_in) go straight into the rank's gather buffer
 *   hdr     [n_shard][1 + 2B]  per layout slot: n, len_0..len_{B-1}, bits(avg_0)..bits(avg_{B-1})
 *   tok_out [sum_u B*cap_u]    per utterance B hypotheses x cap_u tokens (cap_u = ceil(L_u * max_len_ratio) + 1)
 *   sc_out  the same for the per-token score bits
 * slot[u]: layout slot of decoded row u; tok_off[u]: its first element in tok_out / sc_out; cap[u]: its cap_u.
 * Every rank derives the same layout from the length list, so no ids travel (shard.py). */
int e2e_nbest_pack_ragged(int U, int B, int cap_in, const int *tok, const float *score, const int *len,
                          const float *avg, const int *n, const int *slot, const long long *tok_off,
                          const int *cap, int *hdr, int *tok_out, int *sc_out, void *stream);

/* (next, SURVEY §8f row f-1) The WHOLE location-aware attention step in one kernel:
 * LocationAwareAttention.forward (src/module.py:1152-1173) including the location convolution
 * (Conv1d 1->K, W = 2*kernel_size+1 taps, zero padded, no bias; src/module.py:1140,1163) and
 * BaseAttention._attend (src/module.py:1109-1117) including the context product, for the first
 * n_run utterances x B beam slots (hypothesis n = u*B + b):
 *   feat[n][k][t] = sum_j w_conv[k][j] * prev_att[n][t + j - W/2]
 *   attn[n][t]    = softmax_t( (b_e + sum_a w_e[a] * tanh(key[u][t][a] + query[n][a]
 *                            + tanh(sum_k w_proj[a][k] * feat[n][k][t]))) / temperature ),  t < enc_len[u];
 *                   exactly 0 for t >= enc_len[u]   (u = n / B)
 *   ctx[n][e]     = sum_{t < enc_len[u]} attn[n][t] * value[u][t][e]
 *   key_t [U][A][T] (the keys tanh(proj_k(enc)), src/asr.py:343, stored CHANNEL-major), value [U][T][E],
 *   query [n][A], prev_att [n][T] (zero beyond enc_len[u]),
 *   w_conv [K][W], w_proj [A][K], w_energy [A]; attn [n][T], ctx [n][E].
 *   hyps_per_unit: beam slots a warp carries together, 0 (default) or 1, 2, 4 — the result does not depend on it.
 *   Needs K <= 12, A % 4 == 0, W odd, B <= 32; fastest when T % 4 == 0 and E % 4 == 0. */
int e2e_attention_loc_full(const float *key_t, const float *value, const float *query, const float *prev_att,
                           const int *enc_len, const float *w_conv, const float *w_proj, const float *w_energy,
                           float b_energy, float temperature, int n_run, int B, int T, int A, int K, int W, int E,
                           int hyps_per_unit, float *attn, float *ctx, void *stream);

/* (f-1, multi-head) The same step for attention.num_head = H heads (model.py Attention / LocationAwareAttention with
 * num_head > 1, at the batch-1 meaning the per-hypothesis decode gives them), for the first n_run utterances x B beam
 * slots (hypothesis n = u*B + b):
 *   feat[n][k][t]  = sum_h sum_j w_conv[k][h][j] * prev_att[n][h][t + j - W/2]     (Conv1d H->K, zero padded, no bias)
 *   loc[n][t][a]   = tanh(sum_k w_proj[a][k] * feat[n][k][t])                        (shared by all heads)
 *   attn[n][h][t]  = softmax_t( (b_e + sum_a w_e[a] * tanh(key[u][h][t][a] + query[n][h*A + a] + loc[n][t][a]))
 *                               / temperature ),  t < enc_len[u];  exactly 0 for t >= enc_len[u]
 *   ctx[n][h*E+e]  = sum_{t < enc_len[u]} attn[n][h][t] * value_h[u][t][e]
 *   key_t [U][H][A][T] (tanh(proj_k(enc)) head by head, CHANNEL-major), query [n][H*A] (tanh(proj_q(.)) as is),
 *   prev_att [n][H][T] (zero beyond enc_len[u]), w_conv [K][H][W], w_proj [A][K], w_energy [A]; attn [n][H][T],
 *   ctx [n][H*E] (merge_head's input: the caller applies merge_head).
 *   per_head_values = 0: value [U][T][E], shared by every head (no value projection: each head of a hypothesis attends
 *   its own utterance's encoder output); 1: value [U][T][H*E] (tanh(proj_v(enc)) as is), value_h = columns h*E..h*E+E-1.
 *   hyps_per_unit as e2e_attention_loc_full (the result does not depend on it).  H = 1 gives the bits of
 *   e2e_attention_loc_full.
 *   Needs 1 <= H <= 4, K <= 12, A % 4 == 0, W odd, B <= 32 and the filters, per-channel constants, one alignment window
 *   per warp and the queries of at least one group of beam slots within the kernel's shared memory: every such shape is
 *   accepted by e2e_attention_loc_heads_supported (1 / 0), which callers query before choosing this path; any other
 *   returns E2E_ERR_UNSUPPORTED before a launch.  Every beam 1..32 with H <= 4 is supported at A = 300, W = 201, K <= 12. */
int e2e_attention_loc_heads_supported(int B, int H, int A, int K, int W);
int e2e_attention_loc_heads(const float *key_t, const float *value, const float *query, const float *prev_att,
                            const int *enc_len, const float *w_conv, const float *w_proj, const float *w_energy,
                            float b_energy, float temperature, int n_run, int B, int H, int T, int A, int K, int W, int E,
                            int per_head_values, int hyps_per_unit, float *attn, float *ctx, void *stream);

/* (next, SURVEY §8f row f-2) One-token LSTM step of the batched RNNLM (src/lm.py:27-38: nn.LSTM on a
 * [1,1] token) and speller (src/asr.py:259-266).  The recurrent GEMMs stay library calls on an exact 3-piece
 * bf16 split of the fp32 operands; these two entry points are everything around them.
 *
 * e2e_lstm_split_rows: dst[r][p*K + off + c] = piece_p(src[row(r)][c]) for p = 0,1,2 and c < w, where
 *   x = piece_0 + piece_1 + piece_2 exactly (piece_0 = bf16(x), piece_1 = bf16(x - piece_0), ...),
 *   row(r) = row_idx ? row_idx[r] : r   (row_idx: int64, the surviving hypotheses' parent rows —
 *   the state hand-over of src/decode.py:250-257 without copying states).
 *   src fp32 [*][src_pitch]; dst bf16 [n][dst_pitch], dst_pitch >= 3*K: the A operand [a1 | a2 | a3] of the GEMMs. */
int e2e_lstm_split_rows(const float *src, long long src_pitch, const long long *row_idx, int n, int w,
                        void *dst_bf16, long long dst_pitch, int K, int off, void *stream);

/* e2e_lstm_split_rows for up to 8 (source, destination) pairs in ONE launch — the recurrent halves of all layers of an
 * LSTM stack.  The arrays are HOST arrays of n_src entries (device pointers / sizes); every source must be 16-byte
 * vectorisable (width, pitches, K, off multiples of 4). */
int e2e_lstm_split_rows_multi(int n_src, const float *const *srcs_host, const long long *src_pitches_host, const int *widths_host,
                              void *const *dsts_bf16_host, const long long *dst_pitches_host, const int *Ks_host, const int *offs_host,
                              const long long *row_idx, int n, void *stream);

/* e2e_lstm_cell: z = gates[r] + bias (+ table[tok[r]]), gate order i,f,g,o (torch.nn.LSTM);
 *   c'[r] = sigmoid(z_f) * c_prev[row(r)] + sigmoid(z_i) * tanh(z_g);  h'[r] = sigmoid(z_o) * tanh(c'[r])
 *   (fp32, every product and sum rounded separately like the reference's element-wise ops), and, if
 *   a_next_bf16 is given, the 3-piece split of h'[r] into columns [off_next, off_next+D) of the next
 *   layer's A operand (geometry as above).
 *   gates fp32 [n][gates_pitch >= 4D]; bias [4D] (b_ih + b_hh); table [V][4D] + tok int64 [n] (the
 *   layer-0 input projection of the V possible embeddings) or NULL; c_prev [*][D]; c_new, h_new [n][D]. */
int e2e_lstm_cell(const float *gates, long long gates_pitch, const float *bias, const float *table, const long long *tok,
                  const float *c_prev, const long long *row_idx, int n, int D,
                  float *c_new, float *h_new, void *a_next_bf16, long long a_pitch, int K_next, int off_next,
                  void *stream);

/* The same three entry points for the 2-piece fp16 operand format (src/lm.py:27-38 only: every GEMM input of the RNNLM
 * step is an LSTM hidden state, |h| < 1, so a fixed power-of-two scale keeps both pieces in fp16's normal range):
 *   piece_0 = fp16(scale*x), piece_1 = fp16(scale*x - piece_0), scale*x == piece_0 + piece_1 up to 2^-22 |scale*x|;
 *   dst fp16 [n][dst_pitch >= 2*K]: the A operand [a1 | a2].  Against weights split the same way
 *   (scale_w*W == w1 + w2) three partial products a1 w1 + (a1 w2 + a2 w1) replace the six of the bf16 format — half the
 *   tensor-core work — and the GEMM result is (scale*scale_w) * (x W^T):
 * e2e_lstm_cell_f16x2 multiplies the gates by gate_scale = 1/(scale*scale_w) (exact, a power of two) before the bias
 * is added, and writes h' as the 2-piece split of next_scale*h'.  All scales must be powers of two in 2^-60..2^60. */
int e2e_lstm_split_rows_f16x2(const float *src, long long src_pitch, const long long *row_idx, int n, int w,
                              void *dst_f16, long long dst_pitch, int K, int off, float scale, void *stream);
int e2e_lstm_split_rows_multi_f16x2(int n_src, const float *const *srcs_host, const long long *src_pitches_host, const int *widths_host,
                                    void *const *dsts_f16_host, const long long *dst_pitches_host, const int *Ks_host, const int *offs_host,
                                    const long long *row_idx, int n, float scale, void *stream);
int e2e_lstm_cell_f16x2(const float *gates, long long gates_pitch, float gate_scale, const float *bias, const float *table,
                        const long long *tok, const float *c_prev, const long long *row_idx, int n, int D,
                        float *c_new, float *h_new, void *a_next_f16, long long a_pitch, int K_next, int off_next,
                        float next_scale, void *stream);

/* One-token GRU step (nn.GRU; src/lm.py:5-38 and src/asr.py:183-270 with module: GRU), the sibling of e2e_lstm_cell.
 * The caller's GEMM produces four D-wide gate blocks [r | z | n_x | n_h] per row: for a layer with input x the weight is
 * [[W_ir, W_hr], [W_iz, W_hz], [W_in, 0], [0, W_hn]] against A = [x | h] and bias = [b_ir+b_hr | b_iz+b_hz | b_in | b_hn];
 * for a tabled layer 0 the table row is [E W_ir^T + b_ir | E W_iz^T + b_iz | E W_in^T + b_in | 0], the weight
 * [[W_hr], [W_hz], [0], [W_hn]] and bias = [b_hr | b_hz | 0 | b_hn].  With z_q = gates[r][q] + bias_q (+ table[tok[r]][q]):
 *   r = sigmoid(z_r);  u = sigmoid(z_z);  n = tanh(z_nx + r * z_nh);  h'[r] = (h_prev[row(r)] - n) * u + n
 *   (fp32, every product and sum rounded separately, ATen's CPU GRU cell order), and, if a_next is given, the split of
 *   h'[r] into the next layer's A operand exactly as e2e_lstm_cell writes it.  h_prev [*][D]; h_new [n][D] (not h_prev).
 * e2e_gru_cell_f16x2 takes gate_scale / next_scale as e2e_lstm_cell_f16x2 does (|h| < 1 holds for a GRU state too). */
int e2e_gru_cell(const float *gates, long long gates_pitch, const float *bias, const float *table, const long long *tok,
                 const float *h_prev, const long long *row_idx, int n, int D,
                 float *h_new, void *a_next_bf16, long long a_pitch, int K_next, int off_next, void *stream);
int e2e_gru_cell_f16x2(const float *gates, long long gates_pitch, float gate_scale, const float *bias, const float *table,
                       const long long *tok, const float *h_prev, const long long *row_idx, int n, int D,
                       float *h_new, void *a_next_f16, long long a_pitch, int K_next, int off_next, float next_scale, void *stream);

/* (next, SURVEY §8f row f-4) 3x3 "same" convolutions of the VGG front end (src/module.py:672-686) as
 * fp32-accurate tensor-core GEMMs: unfold a block of NHWC pixels into the GEMM's A operand as the exact
 * 3-piece bf16 split [a1 | a2 | a3] of every fp32 value,
 *   out[p - first_pixel][piece*9C + (dy*3+dx)*C + c] = piece(in[n][h+dy-1][w+dx-1][c])   (zero outside the image
 *   and for source rows h+dy-1 >= valid_rows[n]: the masking a padded batch row needs to equal a batch-1 call),
 * p = (n*H + h)*W + w.  The GEMM against weight.permute(2,3,1,0).reshape(9C, Cout) is a library call.
 *   in_nhwc fp32 [N][H][W][C], C % 4 == 0; out bf16 [n_pixels][27*C]. */
int e2e_conv3x3_unfold_split(const float *in_nhwc, const int *valid_rows, int N, int H, int W, int C,
                             long long first_pixel, int n_pixels, void *out_bf16, void *stream);

/* In place on the GEMM result (NHWC): y = relu(y + bias) on rows h < valid_rows[n], 0 elsewhere
 * (Conv2d bias + nn.ReLU of src/module.py:672-686 + the inter-layer masking). */
int e2e_conv_bias_relu_mask(float *y_nhwc, const float *bias, const int *valid_rows, int N, int H, int W, int C,
                            long long first_pixel, long long n_pixels, void *stream);

/* The same convolution as ONE implicit split GEMM on the tcgen05 tensor cores (csrc/conv_igemm.cu, built into
 * libe2e_asr_b200_tc.so, which this library links against and loads from its own directory): the A operand is
 * split from the NHWC input on the way into shared memory (no unfolded operand), the six partial products run into
 * three fp32 accumulators in the K order of the library GEMMs, and the epilogue of the unfold path is fused, so the
 * result equals unfold + mm/addmm/addmm + e2e_conv_bias_relu_mask(_pool) bit for bit.
 *   w_split_bf16 [3][Cout][9C] = the bf16 pieces w1, w2, w3 of Wmat^T (stepper.SplitLinear's split), 16-byte aligned;
 *   epilogue 0: out [N*H*W][Cout] = the raw GEMM result y;  1: out [N][H][W][Cout] = relu(y + bias), 0 on rows
 *   h >= valid_rows[n];  2: out [N][ceil(H/2)][ceil(W/2)][Cout] = the 2x2 ceil-mode max pool of that.
 * Shapes outside e2e_conv3x3_igemm_supported (C and Cout in {128, 256}) return E2E_ERR_UNSUPPORTED before a launch. */
int e2e_conv3x3_igemm_supported(int C, int Cout);
int e2e_conv3x3_igemm(const float *in_nhwc, const int *valid_rows, int N, int H, int W, int C,
                      const void *w_split_bf16, const float *bias, int Cout, int epilogue, float *out, void *stream);

/* (next, SURVEY §8f row f-4) Whole-sequence LSTM recurrence of an encoder layer (RNNLayer, src/module.py:1003-1081:
 * nn.LSTM, optionally bidirectional) over PACKED utterances, one persistent launch per layer:
 *   for every utterance n, direction d and its frames t in walking order (d = 0: 0..len-1, d = 1: len-1..0)
 *     z = gates[frame_off[n] + t][gate_off_d : gate_off_d + 4H] + bias_d + W_hh_d h_prev      (gate order i,f,g,o)
 *     c = sigmoid(z_f) c_prev + sigmoid(z_i) tanh(z_g);  h = sigmoid(z_o) tanh(c);  out[frame_off[n] + t][out_off_d : +H] = h
 *   from zero initial state.  gates = x W_ih^T of all packed frames is the caller's (library) GEMM.
 *   w_t_d [H][H][4] with w_t[k][u][g] = W_hh[g*H + u][k] (16-byte aligned);  bias_d [4H] = b_ih + b_hh (or NULL).
 *   group_first / group_rows [n_groups]: the CTA -> utterance grouping (rows in 1..16; utterances sorted by
 *   decreasing length; give long utterances small groups).  n_dirs 1 or 2.  H <= 384. */
int e2e_lstm_sequence(const float *gates, long long gates_pitch, float *out, long long out_pitch,
                      const int *frame_off, const int *lens, const int *group_first, const int *group_rows,
                      int N, int H, int n_groups, int n_dirs,
                      const float *bias_fw, const float *w_t_fw, int gate_off_fw, int out_off_fw,
                      const float *bias_bw, const float *w_t_bw, int gate_off_bw, int out_off_bw,
                      void *stream);

/* e2e_lstm_sequence for an nn.GRU layer (RNNLayer with module: GRU), same packing, grouping and limits:
 *   z_{r,z,nx} = gates[frame_off[n] + t][gate_off_d : gate_off_d + 3H] + bias_d[0 : 3H]             (gate order r,z,n)
 *   z_nh = bias_d[3H : 4H] + W_hn h_prev;  r = sigmoid(z_r + W_hr h_prev);  u = sigmoid(z_z + W_hz h_prev)
 *   n = tanh(z_nx + r * z_nh);  h = (h_prev - n) * u + n;  out[frame_off[n] + t][out_off_d : +H] = h
 *   bias_d [4H] = [b_ir + b_hr | b_iz + b_hz | b_in | b_hn] (the 3H input-side bias followed by b_hn; or NULL);
 *   w_t_d [H][H][4] with w_t[k][u][g] = W_hh[g*H + u][k] for g < 3 and w_t[k][u][3] = 0;  gates_pitch >= 3H. */
int e2e_gru_sequence(const float *gates, long long gates_pitch, float *out, long long out_pitch,
                     const int *frame_off, const int *lens, const int *group_first, const int *group_rows,
                     int N, int H, int n_groups, int n_dirs,
                     const float *bias_fw, const float *w_t_fw, int gate_off_fw, int out_off_fw,
                     const float *bias_bw, const float *w_t_bw, int gate_off_bw, int out_off_bw,
                     void *stream);

/* First VGG layer (Conv2d Cin->Cout 3x3 "same" + bias + ReLU, src/module.py:672-674) straight from the feature
 * frames: feat [N][L][Cin*F] (a frame is Cin blocks of F bins, src/module.py:688-690; row pitch of an utterance
 * feat_pitch_n floats), weight [Cout][Cin][3][3], out [N][L][F][Cout] NHWC.  Input rows t >= valid_rows[n] read as 0. */
int e2e_conv1_direct(const float *feat, long long feat_pitch_n, const float *weight, const float *bias,
                     const int *valid_rows, int N, int L, int F, int Cin, int Cout, float *out_nhwc, void *stream);

/* e2e_conv_bias_relu_mask fused with the 2x2 stride-2 ceil-mode max pooling that follows the 2nd and 4th
 * convolution (src/module.py:676,683): out [N][ceil(H/2)][ceil(W/2)][C] from the GEMM result y [N][H][W][C]. */
int e2e_conv_bias_relu_mask_pool(const float *y_nhwc, const float *bias, const int *valid_rows, int N, int H, int W, int C,
                                 float *out_nhwc, void *stream);

/* The front end in the 2-piece fp16 operand format (see e2e_lstm_split_rows_f16x2): three partial GEMM products instead
 * of six and a third less unfolded data.  The activations are ReLU outputs of no fixed range, so the scale travels on
 * the device: a word `amax` holds the float bits of max|x| over the rows of a layer's input that the next layer reads
 * (x >= 0; zero it before the producing kernel runs), and
 *   act_scale(amax) = 2^(14 - floor(log2(amax)))  (1 if amax == 0; clamped to 2^-60..2^60)
 * puts that maximum in [2^14, 2^15).
 *   e2e_conv1_direct_amax:              e2e_conv1_direct + max of the outputs on rows t < valid_rows[n] -> atomicMax(amax_out)
 *   e2e_conv3x3_unfold_split_f16x2:     out fp16 [n_pixels][18*C] = [a1 | a2], a1 = fp16(s*x), a2 = fp16(s*x - a1), s = act_scale(*amax_in)
 *   e2e_conv_bias_relu_mask_scaled:     y = relu(y * inv_w_scale / act_scale(*amax_in) + bias) (masked as above); inv_w_scale = 1/scale_w
 *   e2e_conv_bias_relu_mask_pool_scaled of the weights' own split; max of the result -> atomicMax(amax_out) if given. */
int e2e_conv1_direct_amax(const float *feat, long long feat_pitch_n, const float *weight, const float *bias,
                          const int *valid_rows, int N, int L, int F, int Cin, int Cout, float *out_nhwc,
                          unsigned *amax_out, void *stream);
int e2e_conv3x3_unfold_split_f16x2(const float *in_nhwc, const int *valid_rows, int N, int H, int W, int C,
                                   long long first_pixel, int n_pixels, const unsigned *amax_in, void *out_f16, void *stream);
int e2e_conv_bias_relu_mask_scaled(float *y_nhwc, const float *bias, const int *valid_rows, int N, int H, int W, int C,
                                   long long first_pixel, long long n_pixels, const unsigned *amax_in, float inv_w_scale,
                                   unsigned *amax_out, void *stream);
int e2e_conv_bias_relu_mask_pool_scaled(const float *y_nhwc, const float *bias, const int *valid_rows, int N, int H, int W, int C,
                                        float *out_nhwc, const unsigned *amax_in, float inv_w_scale, unsigned *amax_out,
                                        void *stream);

/* Host -> device copy of the VALID frames of n rows of a zero-padded [U][Lmax][D] fp32 feature tensor in pinned host memory
 * (the `.to(device)` of bin/test_asr.py:161-163, without the padding): device row r receives the first lens_host[order_host[r]]
 * frames of host row order_host[r]; one asynchronous copy per row on `stream`; after every `chunk` rows events[r / chunk]
 * (cudaEvent_t, caller-created; may be NULL) is recorded.  row_pitch = Lmax * D floats.  lens_host / order_host / events are
 * HOST arrays. */
int e2e_copy_rows_h2d(const float *host, float *dev, long long row_pitch, int D, const int *lens_host,
                      const long long *order_host, int n, int chunk, void *const *events, void *stream);

/* Number of kernel launches issued through this library by the calling process
 * (for bench.py's gpu_launches claim). */
long long e2e_launch_count(void);
/* Adds n to that count: the library's kernels that ran as nodes of a CUDA graph the caller replayed. */
void e2e_add_launch_count(long long n);

#ifdef __cplusplus
}
#endif
#endif /* E2E_ASR_B200_H */
