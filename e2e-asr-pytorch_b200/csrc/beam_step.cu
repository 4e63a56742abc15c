// Kernels (3a)/(3b) and the final N-best selection of the joint CTC/attention(+LM) beam search.
//   (3a) beam_candidates_kernel : attention log-softmax statistics + top-C candidate ids
//        (src/decode.py:122,129-130)
//   (3b) beam_combine_prune_kernel : score blend, <eos> threshold, top-B per parent, pooled
//        length-normalised prune to B, beam bookkeeping (src/decode.py:134-177,214-263)
//   beam_finalize_kernel : closed + live hypotheses, stable sort by mean score, back-tracking
//        (src/decode.py:180-183,279-281)
// None of this is a dense contraction: one warp per hypothesis row, shuffle reductions, no
// tensor cores.
#include "common.cuh"
#include <limits.h>

namespace e2e {

// log_softmax(v) from the row statistics, in the operation order (x - max) - lse
__device__ __forceinline__ float logp_from(float logit, float mx, float lse)
{
    return __fsub_rn(__fsub_rn(logit, mx), lse);
}

// Row statistics (max, log-sum-exp of the shifted row) computed by one warp.
__device__ __forceinline__ void warp_row_stats(const float *__restrict__ row, int V, int lane, float &mx, float &lse)
{
    float m = -INFINITY;
    for (int v = lane; v < V; v += 32) m = fmaxf(m, __ldg(row + v));
    m = warp_max(m);
    float s = 0.0f;
    for (int v = lane; v < V; v += 32) s += expf(__ldg(row + v) - m);
    s = warp_sum(s);
    mx = m;
    lse = logf(s);
}

// Selects the k best entries of f(v), v in [0,V), best first; ties go to the lower index.
// Works by repeated arg-max over the entries that come strictly after the previous winner in
// (value desc, index asc) order, so no "taken" marks are needed.  emit(rank, value, index) is
// called by every lane with identical arguments; index == -1 when fewer than k entries exist.
template <typename F, typename E>
__device__ __forceinline__ void warp_select_topk(int V, int k, int lane, F f, E emit)
{
    float last_v = INFINITY;
    int last_i = -1;
    for (int r = 0; r < k; ++r) {
        float bv = -INFINITY;
        int bi = INT_MAX;
        for (int v = lane; v < V; v += 32) {
            const float val = f(v);
            const bool eligible = (val < last_v) || (val == last_v && v > last_i);
            if (eligible && (val > bv || (val == bv && v < bi))) { bv = val; bi = v; }
        }
        warp_argmax(bv, bi);
        if (bi == INT_MAX) { emit(r, -INFINITY, -1); continue; }
        emit(r, bv, bi);
        last_v = bv;
        last_i = bi;
    }
}

// The same selection for WIDE rows (the 10k subword vocabulary) in ONE pass over the row: every lane streams its entries
// v = lane, lane + 32, ... through visit(v) -> value and keeps its own k best in a sorted list in shared memory
// (lst_v / lst_i: [k][32], this lane's column; later equal values stay behind earlier ones), then the lists' heads are
// merged by k warp arg-max rounds (ties to the lower index).  Every entry is evaluated once instead of once per round.
template <typename F, typename E>
__device__ __forceinline__ void warp_select_topk_stream(int V, int k, int lane, F visit, E emit, float *lst_v, int *lst_i)
{
    for (int r = 0; r < k; ++r) { lst_v[r * 32 + lane] = -INFINITY; lst_i[r * 32 + lane] = INT_MAX; }
    float worst = -INFINITY;                               // this lane's k-th best so far
    int filled = 0;
    for (int v = lane; v < V; v += 32) {
        const float x = visit(v);
        if (filled < k || x > worst) {
            int pos = filled < k ? filled : k - 1;
            while (pos > 0 && lst_v[(pos - 1) * 32 + lane] < x) {
                lst_v[pos * 32 + lane] = lst_v[(pos - 1) * 32 + lane];
                lst_i[pos * 32 + lane] = lst_i[(pos - 1) * 32 + lane];
                --pos;
            }
            lst_v[pos * 32 + lane] = x;
            lst_i[pos * 32 + lane] = v;
            if (filled < k) ++filled;
            if (filled == k) worst = lst_v[(k - 1) * 32 + lane];
        }
    }
    int head = 0;                                          // next unread entry of this lane's list
    for (int r = 0; r < k; ++r) {
        float bv = head < filled ? lst_v[head * 32 + lane] : -INFINITY;
        int bi = head < filled ? lst_i[head * 32 + lane] : INT_MAX;
        const int mine = bi;
        warp_argmax(bv, bi);
        if (bi == INT_MAX) { emit(r, -INFINITY, -1); continue; }
        emit(r, bv, bi);
        if (mine == bi) ++head;
    }
}

// The same selection over values a lane already holds in registers: lane l owns v = l, l + 32, ... (NV per lane).
template <int NV, typename E>
__device__ __forceinline__ void warp_select_topk_cached(const float (&val)[NV], int V, int k, int lane, E emit)
{
    float last_v = INFINITY;
    int last_i = -1;
    for (int r = 0; r < k; ++r) {
        float bv = -INFINITY;
        int bi = INT_MAX;
#pragma unroll
        for (int q = 0; q < NV; ++q) {
            const int v = lane + 32 * q;
            const float x = val[q];
            const bool eligible = v < V && ((x < last_v) || (x == last_v && v > last_i));
            if (eligible && (x > bv || (x == bv && v < bi))) { bv = x; bi = v; }
        }
        warp_argmax(bv, bi);
        if (bi == INT_MAX) { emit(r, -INFINITY, -1); continue; }
        emit(r, bv, bi);
        last_v = bv;
        last_i = bi;
    }
}

// ---------------------------------------------------------------------------------------------
// (3a) one warp per hypothesis
// ---------------------------------------------------------------------------------------------
constexpr int kCandWarps = 4;

// NV > 0 (V <= 32 * NV): the row's log-probs are evaluated once into registers and the top-C rounds work on those.
template <int NV>
__global__ void __launch_bounds__(kCandWarps * 32)
beam_candidates_kernel(const float *__restrict__ att_logits, int ld, int U, int B, int V, int C,
                       const int *__restrict__ n_live, float2 *__restrict__ att_stats, int *__restrict__ cand)
{
    const int lane = threadIdx.x & 31;
    const int n = blockIdx.x * kCandWarps + (threadIdx.x >> 5);
    if (n >= U * B) return;
    const int u = n / B, b = n - u * B;
    if (n_live && b >= n_live[u]) return;
    const float *row = att_logits + (long long)n * ld;
    float mx, lse;
    warp_row_stats(row, V, lane, mx, lse);
    if (lane == 0) att_stats[n] = make_float2(mx, lse);
    if (C <= 0) return;
    int *out = cand + (long long)n * C;
    if constexpr (NV > 0) {
        float lp[NV];
#pragma unroll
        for (int q = 0; q < NV; ++q) {
            const int v = lane + 32 * q;
            lp[q] = v < V ? logp_from(__ldg(row + v), mx, lse) : -INFINITY;
        }
        warp_select_topk_cached<NV>(lp, V, C, lane, [&](int r, float, int idx) { if (lane == 0) out[r] = idx; });
    } else {
        extern __shared__ __align__(16) unsigned char cand_smem[];          // [warps][C][32] values | [warps][C][32] ids
        float *lv = reinterpret_cast<float *>(cand_smem) + (size_t)(threadIdx.x >> 5) * C * 32;
        int *li = reinterpret_cast<int *>(cand_smem) + (size_t)kCandWarps * C * 32 + (size_t)(threadIdx.x >> 5) * C * 32;
        warp_select_topk_stream(
            V, C, lane, [&](int v) { return logp_from(__ldg(row + v), mx, lse); },
            [&](int r, float, int idx) { if (lane == 0) out[r] = idx; }, lv, li);
    }
}

// ---------------------------------------------------------------------------------------------
// (3a') embedding fusion: (3a) for models decoded with the word-embedding plug-in (src/plugin.py,
//       EmbeddingRegularizer.fuse_prob, called at src/decode.py:~118-122).  One warp per hypothesis.
// ---------------------------------------------------------------------------------------------
struct EmbFuseParams {
    const float *dec; int ld_dec; const float *emb; int ld_emb;
    int U, B, V, C;
    const float *scale; int n_scale;        // relu(temp): 1 or V entries
    const float *lam; int n_lam;            // the mixing weight (after the sigmoid of a learnable one): 1 or V entries
    float eps;
    const int *n_live; float *logp; int ld_out; float2 *att_stats; int *cand;
};

// log((1 - lam) * dec_prob + lam * emb_prob + eps), every operation rounded in plugin.py's order
__device__ __forceinline__ float fused_logp(float pd, float pe, float lam, float eps)
{
    const float mix = __fadd_rn(__fmul_rn(__fsub_rn(1.0f, lam), pd), __fmul_rn(lam, pe));
    return logf(__fadd_rn(mix, eps));
}

// softmax(x)[v] = exp(x[v] - max) * (1 / sum): the reciprocal form of ATen's row softmax
template <int NV>
__global__ void __launch_bounds__(kCandWarps * 32)
emb_fuse_candidates_kernel(const EmbFuseParams p)
{
    const int lane = threadIdx.x & 31;
    const int n = blockIdx.x * kCandWarps + (threadIdx.x >> 5);
    if (n >= p.U * p.B) return;
    const int u = n / p.B, b = n - u * p.B;
    if (p.n_live && b >= p.n_live[u]) return;
    const int V = p.V, C = p.C;
    const float *drow = p.dec + (long long)n * p.ld_dec;
    const float *erow = p.emb + (long long)n * p.ld_emb;
    float *out = p.logp + (long long)n * p.ld_out;
    auto scaled_emb = [&](int v) { return __fmul_rn(__ldg(p.scale + (p.n_scale == 1 ? 0 : v)), __ldg(erow + v)); };
    auto lam_of = [&](int v) { return __ldg(p.lam + (p.n_lam == 1 ? 0 : v)); };
    // (3b) forms its attention log-prob as (x - max) - lse: zero statistics pass the fused row through unchanged
    if (lane == 0) p.att_stats[n] = make_float2(0.0f, 0.0f);
    int *cand = C > 0 ? p.cand + (long long)n * C : nullptr;
    auto emit = [&](int r, float, int idx) { if (lane == 0) cand[r] = idx; };
    if constexpr (NV > 0) {
        // narrow rows: both rows live in registers, one read of each
        float xd[NV], xe[NV];
        float md = -INFINITY, me = -INFINITY;
#pragma unroll
        for (int q = 0; q < NV; ++q) {
            const int v = lane + 32 * q;
            xd[q] = v < V ? __ldg(drow + v) : -INFINITY;
            xe[q] = v < V ? scaled_emb(v) : -INFINITY;
            md = fmaxf(md, xd[q]);
            me = fmaxf(me, xe[q]);
        }
        md = warp_max(md);
        me = warp_max(me);
        float sd = 0.0f, se = 0.0f;
#pragma unroll
        for (int q = 0; q < NV; ++q) {
            if (lane + 32 * q < V) {
                xd[q] = expf(xd[q] - md);
                xe[q] = expf(xe[q] - me);
                sd += xd[q];
                se += xe[q];
            }
        }
        const float rd = __fdiv_rn(1.0f, warp_sum(sd)), re = __fdiv_rn(1.0f, warp_sum(se));
        float lp[NV];
#pragma unroll
        for (int q = 0; q < NV; ++q) {
            const int v = lane + 32 * q;
            lp[q] = -INFINITY;
            if (v < V) {
                lp[q] = fused_logp(__fmul_rn(xd[q], rd), __fmul_rn(xe[q], re), lam_of(v), p.eps);
                out[v] = lp[q];
            }
        }
        if (C > 0) warp_select_topk_cached<NV>(lp, V, C, lane, emit);
    } else {
        // wide rows: maxima, then sums, then one pass that writes the fused row and feeds the streaming top-C lists
        float md = -INFINITY, me = -INFINITY;
        for (int v = lane; v < V; v += 32) {
            md = fmaxf(md, __ldg(drow + v));
            me = fmaxf(me, scaled_emb(v));
        }
        md = warp_max(md);
        me = warp_max(me);
        float sd = 0.0f, se = 0.0f;
        for (int v = lane; v < V; v += 32) {
            sd += expf(__ldg(drow + v) - md);
            se += expf(scaled_emb(v) - me);
        }
        const float rd = __fdiv_rn(1.0f, warp_sum(sd)), re = __fdiv_rn(1.0f, warp_sum(se));
        auto visit = [&](int v) -> float {
            const float pd = __fmul_rn(expf(__ldg(drow + v) - md), rd);
            const float pe = __fmul_rn(expf(scaled_emb(v) - me), re);
            const float lp = fused_logp(pd, pe, lam_of(v), p.eps);
            out[v] = lp;
            return lp;
        };
        if (C > 0) {
            extern __shared__ __align__(16) unsigned char fuse_smem[];           // [warps][C][32] values | [warps][C][32] ids
            float *lv = reinterpret_cast<float *>(fuse_smem) + (size_t)(threadIdx.x >> 5) * C * 32;
            int *li = reinterpret_cast<int *>(fuse_smem) + (size_t)kCandWarps * C * 32 + (size_t)(threadIdx.x >> 5) * C * 32;
            warp_select_topk_stream(V, C, lane, visit, emit, lv, li);
        } else {
            for (int v = lane; v < V; v += 32) visit(v);
        }
    }
}

// ---------------------------------------------------------------------------------------------
// (3b) one CTA per utterance, one warp per parent hypothesis, then a pooled rank sort
// ---------------------------------------------------------------------------------------------
struct CombineParams {
    const float *att_logits; int ld_att; const float2 *att_stats;
    const float *lm_logits; int ld_lm;
    const int *cand; const float *psi;
    int U, B, V, C, step;
    const int *min_len, *max_len;
    float w_ctc, w_att, w_lm, eos_threshold; int flags;
    int *n_live, *n_active, *last_tok, *prefix_len; float *score_sum, *ctc_prob; int *prev_lane;
    int *parent_slot, *hist_tok, *hist_parent; float *hist_score;
    long long *parent_row, *last_tok64;     // optional 64-bit copies for the host's gathers (row = u*B + parent slot)
    int *parent_tok;                        // optional: last token of each survivor's PARENT (-1: the empty prefix)
    int *fin_count, *fin_step, *fin_parent; float *fin_sum, *fin_score; int fin_cap;
    int *status;
};

// NV > 0 (V <= 32 * NV, the character vocabularies): every lane evaluates the attention log-probs and the blended scores of
// its NV vocabulary entries ONCE, into registers, and the top-k rounds and the <eos> scan work on those; NV == 0: any V,
// the scores are re-evaluated per round.  Same operations per score either way, hence the same values.
template <int NV>
__global__ void __launch_bounds__(1024)
beam_combine_prune_kernel(const CombineParams p)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int u = blockIdx.x;
    const int B = p.B, C = p.C, V = p.V;
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;    // warp w handles parent slot w
    int *out_parent = p.parent_slot + (long long)u * B;
    const bool idle = p.step >= p.max_len[u];
    if (idle) {
        for (int i = threadIdx.x; i < B; i += blockDim.x) {
            out_parent[i] = i;
            if (p.parent_row) p.parent_row[(long long)u * B + i] = (long long)u * B + i;
        }
        return;
    }
    const bool use_ctc = (p.flags & E2E_BEAM_USE_CTC) != 0, use_lm = (p.flags & E2E_BEAM_USE_LM) != 0;
    const int live = p.n_live[u];

    // shared: child_tok/child_lane [B*B] int, child_score/child_sum/child_psi/child_key [B*B] float,
    //         cnt[B] int, term_flag[B] int, term_score[B] float, cand ids/deltas per warp [B*C]
    int *c_tok = reinterpret_cast<int *>(smem_raw);
    int *c_lane = c_tok + B * B;
    float *c_score = reinterpret_cast<float *>(c_lane + B * B);
    float *c_sum = c_score + B * B;
    float *c_psi = c_sum + B * B;
    float *c_key = c_psi + B * B;
    int *cnt = reinterpret_cast<int *>(c_key + B * B);
    int *term = cnt + B;
    float *term_sc = reinterpret_cast<float *>(term + B);
    int *w_cand = reinterpret_cast<int *>(term_sc + B);
    float *w_delta = reinterpret_cast<float *>(w_cand + B * (C > 0 ? C : 1));
    float *top_v = w_delta + B * (C > 0 ? C : 1);              // [B][B] winners per parent
    int *top_i = reinterpret_cast<int *>(top_v + B * B);
    int *par_tok = top_i + B * B;                              // [B] the parents' own last tokens
    // wide rows only (NV == 0): per-warp streaming top-B lists [B][B][32] x (value, id) and candidate bitmaps [B][ceil(V/32)]
    float *stream_v = reinterpret_cast<float *>(par_tok + B);
    int *stream_i = reinterpret_cast<int *>(stream_v + (NV == 0 ? (size_t)B * B * 32 : 0));
    const int bit_words = (V + 31) >> 5;
    unsigned *cand_bits = reinterpret_cast<unsigned *>(stream_i + (NV == 0 ? (size_t)B * B * 32 : 0));

    if (threadIdx.x < B) {
        cnt[threadIdx.x] = 0; term[threadIdx.x] = 0;
        par_tok[threadIdx.x] = (p.step > 0 && threadIdx.x < live) ? p.last_tok[u * B + threadIdx.x] : -1;
    }
    __syncthreads();

    if (w < live) {
        const int n = u * B + w;
        const float *att = p.att_logits + (long long)n * p.ld_att;
        const float2 ast = p.att_stats[n];
        const float *lm = use_lm ? p.lm_logits + (long long)n * p.ld_lm : nullptr;
        float lmx = 0.0f, llse = 0.0f;
        if (use_lm) warp_row_stats(lm, V, lane, lmx, llse);
        int *mycand = w_cand + w * (C > 0 ? C : 1);
        float *mydelta = w_delta + w * (C > 0 ? C : 1);
        if (use_ctc) {
            const float parent_psi = p.ctc_prob[n];
            for (int j = lane; j < C; j += 32) {
                mycand[j] = p.cand[(long long)n * C + j];
                mydelta[j] = __fsub_rn(p.psi[(long long)n * C + j], parent_psi);     // decode.py:134
            }
            __syncwarp();
        }
        auto blended = [&](int v) -> float {
            float cur = logp_from(__ldg(att + v), ast.x, ast.y);
            if (use_ctc) {
                float spread = E2E_DEC_LOG_ZERO;                                     // decode.py:137-139
                for (int j = 0; j < C; ++j)
                    if (mycand[j] == v) { spread = mydelta[j]; break; }
                cur = __fadd_rn(__fmul_rn(p.w_att, cur), __fmul_rn(p.w_ctc, spread));  // decode.py:140
                if (v == 0) cur = E2E_DEC_LOG_ZERO;                                  // decode.py:141
            }
            if (use_lm) cur = __fadd_rn(cur, __fmul_rn(p.w_lm, logp_from(__ldg(lm + v), lmx, llse)));   // decode.py:151
            return cur;
        };
        float *tv = top_v + w * B;
        int *ti = top_i + w * B;
        // The eos test looks at the pure attention log-probs when CTC is on; with CTC off the
        // reference's in-place "+=" of the LM term aliases them (SURVEY.md §8a-Q2).
        const bool alias = (!use_ctc) && use_lm;
        float best_other = -INFINITY, eos_lp = -INFINITY;
        if constexpr (NV > 0) {
            float bval[NV];
#pragma unroll
            for (int q = 0; q < NV; ++q) {
                const int v = lane + 32 * q;
                bval[q] = -INFINITY;
                if (v < V) {
                    bval[q] = blended(v);
                    const float plain = alias ? bval[q] : logp_from(__ldg(att + v), ast.x, ast.y);
                    if (v >= 2) best_other = fmaxf(best_other, plain);
                    if (v == E2E_CTC_EOS) eos_lp = plain;
                }
            }
            warp_select_topk_cached<NV>(bval, V, B, lane, [&](int r, float val, int idx) {
                if (lane == 0) { tv[r] = val; ti[r] = idx; }
            });
            best_other = warp_max(best_other);
            eos_lp = __shfl_sync(E2E_FULL_MASK, eos_lp, E2E_CTC_EOS & 31);
        } else if constexpr (NV < 0) {
            // any width, no extra shared memory: the scores are re-evaluated in every top-k round (beam sizes whose streaming lists
            // would not fit)
            warp_select_topk(V, B, lane, blended, [&](int r, float val, int idx) {
                if (lane == 0) { tv[r] = val; ti[r] = idx; }
            });
            for (int v = 2 + lane; v < V; v += 32)
                best_other = fmaxf(best_other, alias ? blended(v) : logp_from(__ldg(att + v), ast.x, ast.y));
            best_other = warp_max(best_other);
            if (V > 1) eos_lp = alias ? blended(E2E_CTC_EOS) : logp_from(__ldg(att + E2E_CTC_EOS), ast.x, ast.y);
        } else {
            // wide rows: ONE pass — every entry is blended once, feeds this lane's top-B list and the <eos> scan; a bitmap of the
            // candidate ids replaces the C compares per entry
            float *lv = stream_v + (size_t)w * B * 32;
            int *li = stream_i + (size_t)w * B * 32;
            unsigned *bits = cand_bits + (size_t)w * bit_words;
            for (int i = lane; i < bit_words; i += 32) bits[i] = 0u;
            __syncwarp();
            if (use_ctc)
                for (int j = lane; j < C; j += 32) atomicOr(bits + (mycand[j] >> 5), 1u << (mycand[j] & 31));
            __syncwarp();
            auto visit = [&](int v) -> float {
                const float plain_att = logp_from(__ldg(att + v), ast.x, ast.y);
                float cur = plain_att;
                if (use_ctc) {
                    float spread = E2E_DEC_LOG_ZERO;
                    if ((bits[v >> 5] >> (v & 31)) & 1u)
                        for (int j = 0; j < C; ++j)
                            if (mycand[j] == v) { spread = mydelta[j]; break; }
                    cur = __fadd_rn(__fmul_rn(p.w_att, cur), __fmul_rn(p.w_ctc, spread));
                    if (v == 0) cur = E2E_DEC_LOG_ZERO;
                }
                if (use_lm) cur = __fadd_rn(cur, __fmul_rn(p.w_lm, logp_from(__ldg(lm + v), lmx, llse)));
                const float plain = alias ? cur : plain_att;
                if (v >= 2) best_other = fmaxf(best_other, plain);
                if (v == E2E_CTC_EOS) eos_lp = plain;
                return cur;
            };
            warp_select_topk_stream(V, B, lane, visit, [&](int r, float val, int idx) {
                if (lane == 0) { tv[r] = val; ti[r] = idx; }
            }, lv, li);
            best_other = warp_max(best_other);
            eos_lp = __shfl_sync(E2E_FULL_MASK, eos_lp, E2E_CTC_EOS & 31);
        }
        __syncwarp();
        // ---- <eos> threshold + child creation (Hypothesis.addTopk, decode.py:219-263) ----------
        if (lane == 0) {
            const float parent_sum = p.score_sum[n];
            int made = 0;
            for (int r = 0; r < B; ++r) {
                const int tok = ti[r];
                if (tok < 0) break;                         // fewer than B vocabulary entries
                const float sc = tv[r];
                if (tok == E2E_CTC_EOS && (double)eos_lp > (double)p.eos_threshold * (double)best_other) {
                    term[w] = 1;
                    term_sc[w] = sc;
                    continue;
                }
                int jsel = 0;
                float child_psi = 0.0f;
                if (use_ctc) {
                    jsel = -1;
                    for (int j = 0; j < C; ++j)
                        if (mycand[j] == tok) { jsel = j; break; }
                    if (jsel < 0) {                         // reference: ValueError at decode.py:252
                        if (p.status) atomicOr(p.status + u, E2E_STATUS_TOKEN_NOT_CAND);
                        jsel = 0;
                    }
                    child_psi = p.psi[(long long)n * C + jsel];
                }
                const int slot = w * B + made;
                c_tok[slot] = tok;
                c_lane[slot] = w * (C > 0 ? C : 1) + jsel;
                c_score[slot] = sc;
                c_sum[slot] = (p.step == 0) ? sc : __fadd_rn(parent_sum, sc);      // python sum(): 0 + s0 + s1 ...
                c_psi[slot] = child_psi;
                c_key[slot] = __fdiv_rn(c_sum[slot], (float)(p.step + 1));          // avgScore, decode.py:214-217
                ++made;
            }
            cnt[w] = made;
        }
    }
    __syncthreads();

    // ---- closed hypotheses (decode.py:167-170): parent order, only once step >= min_len ---------
    // The list is kept stably sorted by mean score and truncated to fin_cap entries: the final
    // selection (decode.py:180-183) is a stable sort of closed ++ live hypotheses cut to B, so with
    // fin_cap >= B nothing that could be returned is ever dropped.
    if (threadIdx.x == 0 && p.step >= p.min_len[u]) {
        int fc = p.fin_count[u];
        const long long base = (long long)u * p.fin_cap;
        for (int b = 0; b < live; ++b) {
            if (!term[b]) continue;
            const float ps = p.score_sum[u * B + b];
            const float fsum = (p.step == 0) ? term_sc[b] : __fadd_rn(ps, term_sc[b]);
            const float key = __fdiv_rn(fsum, (float)(p.step + 1));
            int pos = fc;                                   // stable: after every entry with key >= ours
            while (pos > 0 && !(__fdiv_rn(p.fin_sum[base + pos - 1], (float)(p.fin_step[base + pos - 1] + 1)) >= key)) --pos;
            if (pos >= p.fin_cap) continue;
            const int last = fc < p.fin_cap ? fc : p.fin_cap - 1;
            for (int i = last; i > pos; --i) {
                p.fin_step[base + i] = p.fin_step[base + i - 1];
                p.fin_parent[base + i] = p.fin_parent[base + i - 1];
                p.fin_score[base + i] = p.fin_score[base + i - 1];
                p.fin_sum[base + i] = p.fin_sum[base + i - 1];
            }
            p.fin_step[base + pos] = p.step;
            p.fin_parent[base + pos] = b;
            p.fin_score[base + pos] = term_sc[b];
            p.fin_sum[base + pos] = fsum;
            if (fc < p.fin_cap) ++fc;
        }
        p.fin_count[u] = fc;
    }
    __syncthreads();     // all reads of the old beam state are done; it may be overwritten now

    // ---- pooled prune: stable sort by mean score, keep B (decode.py:175-176) --------------------
    // compact position of child (parent b, k-th child) = sum_{b'<b} cnt[b'] + k  == list order
    int total = 0;
    for (int b = 0; b < live; ++b) total += cnt[b];
    const int keep = total < B ? total : B;
    const long long hrow = ((long long)p.step * p.U + u) * B;
    for (int i = threadIdx.x; i < B * B; i += blockDim.x) {
        const int b = i / B, k = i - b * B;
        if (b >= live || k >= cnt[b]) continue;
        // list position = (parent, k-th child) order; a child of an earlier parent, or an earlier child of the same parent,
        // comes first among equal keys
        const float key = c_key[i];
        int rank = 0;
        for (int b2 = 0; b2 < live; ++b2) {
            const int n2 = cnt[b2];
            for (int k2 = 0; k2 < n2; ++k2) {
                const float key2 = c_key[b2 * B + k2];
                if (key2 > key || (key2 == key && (b2 < b || (b2 == b && k2 < k)))) ++rank;
            }
        }
        if (rank < B) {
            const int o = u * B + rank;
            p.last_tok[o] = c_tok[i];
            if (p.last_tok64) p.last_tok64[o] = c_tok[i];
            if (p.parent_row) p.parent_row[o] = (long long)u * B + b;
            if (p.parent_tok) p.parent_tok[o] = par_tok[b];
            p.prefix_len[o] = p.step + 1;
            p.score_sum[o] = c_sum[i];
            p.ctc_prob[o] = c_psi[i];
            p.prev_lane[o] = c_lane[i];
            out_parent[rank] = b;
            p.hist_tok[hrow + rank] = c_tok[i];
            p.hist_parent[hrow + rank] = b;
            p.hist_score[hrow + rank] = c_score[i];
        }
    }
    for (int i = keep + threadIdx.x; i < B; i += blockDim.x) {      // unused slots: keep gathers in range
        out_parent[i] = 0;
        if (p.parent_row) p.parent_row[(long long)u * B + i] = (long long)u * B;
        p.hist_tok[hrow + i] = 0;
        p.hist_parent[hrow + i] = 0;
        p.hist_score[hrow + i] = 0.0f;
    }
    if (threadIdx.x == 0) {
        p.n_live[u] = keep;
        if (p.n_active) p.n_active[u] = (p.step + 1 < p.max_len[u]) ? keep : 0;   // rows the next step's kernels touch
    }
}

static size_t combine_smem_bytes(int B, int C, int V, bool stream)
{
    const int Cc = C > 0 ? C : 1;
    size_t words = (size_t)(6 * B * B + 4 * B + 2 * B * Cc + 2 * B * B);
    if (stream) words += (size_t)2 * B * B * 32 + (size_t)B * ((V + 31) / 32);        // streaming lists + candidate bitmaps
    return words * 4 + 16;
}

// ---------------------------------------------------------------------------------------------
// final selection: one CTA per utterance
// ---------------------------------------------------------------------------------------------
struct FinalParams {
    int U, B; const int *max_len, *n_live; const float *score_sum;
    const int *hist_tok, *hist_parent; const float *hist_score;
    const int *fin_count, *fin_step, *fin_parent; const float *fin_sum, *fin_score; int fin_cap;
    int *out_tok; float *out_score; int *out_len; float *out_avg; int *out_n; int out_cap;
};

__global__ void __launch_bounds__(128)
beam_finalize_kernel(const FinalParams p)
{
    const int u = blockIdx.x, B = p.B;
    const int S = p.max_len[u];                     // every live hypothesis has exactly S tokens
    const int fc = p.fin_count[u];
    const int live = (S > 0) ? p.n_live[u] : 0;
    const int total = fc + live;
    auto key_of = [&](int e) -> float {             // list order: closed first, then the last beam
        if (e < fc) {
            const long long o = (long long)u * p.fin_cap + e;
            return __fdiv_rn(p.fin_sum[o], (float)(p.fin_step[o] + 1));
        }
        return __fdiv_rn(p.score_sum[u * B + (e - fc)], (float)S);
    };
    for (int e = threadIdx.x; e < total; e += blockDim.x) {
        const float key = key_of(e);
        int rank = 0;
        for (int e2 = 0; e2 < total; ++e2) {
            const float k2 = key_of(e2);
            if (k2 > key || (k2 == key && e2 < e)) ++rank;
        }
        if (rank >= B) continue;
        const long long ob = (long long)u * B + rank;
        int *tok = p.out_tok + ob * p.out_cap;
        float *sc = p.out_score + ob * p.out_cap;
        int len, slot, s;
        if (e < fc) {
            const long long o = (long long)u * p.fin_cap + e;
            len = p.fin_step[o] + 1;
            if (len <= p.out_cap) { tok[len - 1] = E2E_CTC_EOS; sc[len - 1] = p.fin_score[o]; }
            slot = p.fin_parent[o];
            s = len - 2;
        } else {
            len = S;
            slot = e - fc;
            s = len - 1;
        }
        for (; s >= 0; --s) {
            const long long hidx = ((long long)s * p.U + u) * B + slot;
            if (s < p.out_cap) { tok[s] = p.hist_tok[hidx]; sc[s] = p.hist_score[hidx]; }
            slot = p.hist_parent[hidx];
        }
        p.out_len[ob] = len;
        p.out_avg[ob] = key;
    }
    if (threadIdx.x == 0) p.out_n[u] = total < B ? total : B;
}

// ---------------------------------------------------------------------------------------------
// ragged N-best pack: one CTA per decoded utterance, straight from beam_finalize's outputs into the
// rank's gather buffer (shard.py: headers | tokens | score bits)
// ---------------------------------------------------------------------------------------------
struct PackParams {
    int U, B, cap_in;
    const int *tok; const float *score; const int *len; const float *avg; const int *n;
    const int *slot; const long long *tok_off; const int *cap;
    int *hdr, *tok_out, *sc_out;
};

__global__ void __launch_bounds__(256)
nbest_pack_kernel(const PackParams p)
{
    const int u = blockIdx.x, B = p.B;
    const int cap = p.cap[u];
    int *hdr = p.hdr + (long long)p.slot[u] * (1 + 2 * B);
    if (threadIdx.x == 0) hdr[0] = p.n[u];
    for (int b = threadIdx.x; b < B; b += blockDim.x) {
        hdr[1 + b] = p.len[u * B + b];
        hdr[1 + B + b] = __float_as_int(p.avg[u * B + b]);
    }
    const long long base = p.tok_off[u];
    for (int i = threadIdx.x; i < B * cap; i += blockDim.x) {
        const int b = i / cap, k = i - b * cap;
        const long long src = ((long long)u * B + b) * p.cap_in + k;
        const bool have = k < p.cap_in;
        p.tok_out[base + i] = have ? p.tok[src] : 0;
        p.sc_out[base + i] = have ? __float_as_int(p.score[src]) : 0;
    }
}

}  // namespace e2e

extern "C" int e2e_nbest_pack_ragged(int U, int B, int cap_in, const int *tok, const float *score, const int *len,
                                     const float *avg, const int *n, const int *slot, const long long *tok_off,
                                     const int *cap, int *hdr, int *tok_out, int *sc_out, void *stream)
{
    using namespace e2e;
    if (!tok || !score || !len || !avg || !n || !slot || !tok_off || !cap || !hdr || !tok_out || !sc_out)
        return set_error(E2E_ERR_ARG, "e2e_nbest_pack_ragged: null pointer");
    if (U <= 0 || B <= 0 || cap_in <= 0) return set_error(E2E_ERR_ARG, "e2e_nbest_pack_ragged: bad size");
    PackParams p;
    p.U = U; p.B = B; p.cap_in = cap_in; p.tok = tok; p.score = score; p.len = len; p.avg = avg; p.n = n;
    p.slot = slot; p.tok_off = tok_off; p.cap = cap; p.hdr = hdr; p.tok_out = tok_out; p.sc_out = sc_out;
    nbest_pack_kernel<<<U, 256, 0, static_cast<cudaStream_t>(stream)>>>(p);
    count_launch();
    return check_launch("e2e_nbest_pack_ragged");
}

extern "C" int e2e_beam_candidates(const float *att_logits, int ld, int U, int B, int V, int C,
                                   const int *n_live, float *att_stats, int *cand, void *stream)
{
    using namespace e2e;
    if (!att_logits || !att_stats || (C > 0 && !cand)) return set_error(E2E_ERR_ARG, "e2e_beam_candidates: null pointer");
    if (U <= 0 || B <= 0 || V <= 0 || C < 0 || ld < V || C > V) return set_error(E2E_ERR_ARG, "e2e_beam_candidates: bad size");
    const int N = U * B;
    void (*kern)(const float *, int, int, int, int, int, const int *, float2 *, int *) =
        V <= 32 ? beam_candidates_kernel<1> : V <= 64 ? beam_candidates_kernel<2> : V <= 128 ? beam_candidates_kernel<4> : beam_candidates_kernel<0>;
    const size_t smem = V > 128 ? (size_t)kCandWarps * C * 32 * 8 : 0;      // per-lane top-C lists of the streaming selection
    if (smem > 48 * 1024) {
        if (smem > 200 * 1024) return set_error(E2E_ERR_UNSUPPORTED, "e2e_beam_candidates: C too large");
        cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return set_error(E2E_ERR_LAUNCH, "cudaFuncSetAttribute: %s", cudaGetErrorString(e));
    }
    kern<<<(N + kCandWarps - 1) / kCandWarps, kCandWarps * 32, smem, static_cast<cudaStream_t>(stream)>>>(
        att_logits, ld, U, B, V, C, n_live, reinterpret_cast<float2 *>(att_stats), cand);
    count_launch();
    return check_launch("e2e_beam_candidates");
}

extern "C" int e2e_emb_fuse_candidates(const float *dec_logits, int ld_dec, const float *emb_logits, int ld_emb,
                                       int U, int B, int V, int C, const float *scale, int n_scale,
                                       const float *lam, int n_lam, float eps, const int *n_live,
                                       float *logp, int ld_out, float *att_stats, int *cand, void *stream)
{
    using namespace e2e;
    if (!dec_logits || !emb_logits || !scale || !lam || !logp || !att_stats || (C > 0 && !cand))
        return set_error(E2E_ERR_ARG, "e2e_emb_fuse_candidates: null pointer");
    if (U <= 0 || B <= 0 || V <= 0 || C < 0 || C > V || ld_dec < V || ld_emb < V || ld_out < V)
        return set_error(E2E_ERR_ARG, "e2e_emb_fuse_candidates: bad size");
    if ((n_scale != 1 && n_scale != V) || (n_lam != 1 && n_lam != V))
        return set_error(E2E_ERR_ARG, "e2e_emb_fuse_candidates: scale / lam must have 1 or V entries");
    if (!(eps > 0.0f) || !isfinite(eps)) return set_error(E2E_ERR_ARG, "e2e_emb_fuse_candidates: eps must be positive and finite");
    EmbFuseParams p;
    p.dec = dec_logits; p.ld_dec = ld_dec; p.emb = emb_logits; p.ld_emb = ld_emb;
    p.U = U; p.B = B; p.V = V; p.C = C;
    p.scale = scale; p.n_scale = n_scale; p.lam = lam; p.n_lam = n_lam; p.eps = eps;
    p.n_live = n_live; p.logp = logp; p.ld_out = ld_out; p.att_stats = reinterpret_cast<float2 *>(att_stats); p.cand = cand;
    const int N = U * B;
    void (*kern)(EmbFuseParams) = V <= 32 ? emb_fuse_candidates_kernel<1> : V <= 64 ? emb_fuse_candidates_kernel<2>
                                : V <= 128 ? emb_fuse_candidates_kernel<4> : emb_fuse_candidates_kernel<0>;
    const size_t smem = V > 128 ? (size_t)kCandWarps * C * 32 * 8 : 0;      // per-lane top-C lists of the streaming selection
    if (smem > 48 * 1024) {
        if (smem > 200 * 1024) return set_error(E2E_ERR_UNSUPPORTED, "e2e_emb_fuse_candidates: C too large");
        cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return set_error(E2E_ERR_LAUNCH, "cudaFuncSetAttribute: %s", cudaGetErrorString(e));
    }
    kern<<<(N + kCandWarps - 1) / kCandWarps, kCandWarps * 32, smem, static_cast<cudaStream_t>(stream)>>>(p);
    count_launch();
    return check_launch("e2e_emb_fuse_candidates");
}

extern "C" int e2e_beam_combine_prune(const float *att_logits, int ld_att, const float *att_stats,
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
                                      long long *parent_row, long long *last_tok64, int *parent_tok, void *stream)
{
    using namespace e2e;
    const bool use_ctc = (flags & E2E_BEAM_USE_CTC) != 0, use_lm = (flags & E2E_BEAM_USE_LM) != 0;
    if (!att_logits || !att_stats || !min_len || !max_len || !n_live || !last_tok || !prefix_len || !score_sum || !ctc_prob || !prev_lane ||
        !parent_slot || !hist_tok || !hist_parent || !hist_score || !fin_count || !fin_step || !fin_parent || !fin_sum || !fin_score)
        return set_error(E2E_ERR_ARG, "e2e_beam_combine_prune: null pointer");
    if ((use_lm && !lm_logits) || (use_ctc && (!cand || !psi || C <= 0)))
        return set_error(E2E_ERR_ARG, "e2e_beam_combine_prune: flags need lm_logits / cand+psi");
    if (U <= 0 || B <= 0 || B > 32 || V <= 0 || step < 0 || fin_cap <= 0 || ld_att < V || (use_lm && ld_lm < V))
        return set_error(E2E_ERR_ARG, "e2e_beam_combine_prune: bad size (beam size must be 1..32)");
    if (fin_cap < B) return set_error(E2E_ERR_ARG, "e2e_beam_combine_prune: fin_cap must be >= B");
    CombineParams p;
    p.att_logits = att_logits; p.ld_att = ld_att; p.att_stats = reinterpret_cast<const float2 *>(att_stats);
    p.lm_logits = lm_logits; p.ld_lm = ld_lm; p.cand = cand; p.psi = psi;
    p.U = U; p.B = B; p.V = V; p.C = use_ctc ? C : 0; p.step = step; p.min_len = min_len; p.max_len = max_len;
    // (1 - w) is formed in double like the reference's python float, then rounded once to fp32
    p.w_ctc = ctc_weight; p.w_att = (float)(1.0 - (double)ctc_weight); p.w_lm = lm_weight; p.eos_threshold = eos_threshold;
    p.flags = flags;
    p.n_live = n_live; p.n_active = n_active; p.last_tok = last_tok; p.prefix_len = prefix_len; p.score_sum = score_sum; p.ctc_prob = ctc_prob; p.prev_lane = prev_lane;
    p.parent_slot = parent_slot; p.hist_tok = hist_tok; p.hist_parent = hist_parent; p.hist_score = hist_score;
    p.parent_row = parent_row; p.last_tok64 = last_tok64; p.parent_tok = parent_tok;
    p.fin_count = fin_count; p.fin_step = fin_step; p.fin_parent = fin_parent; p.fin_sum = fin_sum; p.fin_score = fin_score;
    p.fin_cap = fin_cap; p.status = status;
    bool stream_sel = V > 128;
    if (stream_sel && combine_smem_bytes(B, p.C, V, true) > 160 * 1024) stream_sel = false;      // multi-pass selection instead
    const size_t smem = combine_smem_bytes(B, p.C, V, stream_sel);
    if (n_run <= 0 || n_run > U) n_run = U;
    void (*kern)(CombineParams) = V <= 32 ? beam_combine_prune_kernel<1> : V <= 64 ? beam_combine_prune_kernel<2>
                                : V <= 128 ? beam_combine_prune_kernel<4> : stream_sel ? beam_combine_prune_kernel<0> : beam_combine_prune_kernel<-1>;
    if (smem > 48 * 1024) {
        cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return set_error(E2E_ERR_LAUNCH, "cudaFuncSetAttribute: %s", cudaGetErrorString(e));
    }
    kern<<<n_run, B * 32, smem, static_cast<cudaStream_t>(stream)>>>(p);
    count_launch();
    return check_launch("e2e_beam_combine_prune");
}

extern "C" int e2e_beam_finalize(int U, int B, const int *max_len,
                                 const int *n_live, const float *score_sum,
                                 const int *hist_tok, const int *hist_parent, const float *hist_score,
                                 const int *fin_count, const int *fin_step, const int *fin_parent,
                                 const float *fin_sum, const float *fin_score, int fin_cap,
                                 int *out_tok, float *out_score, int *out_len, float *out_avg, int *out_n,
                                 int out_cap, void *stream)
{
    using namespace e2e;
    if (!max_len || !n_live || !score_sum || !hist_tok || !hist_parent || !hist_score || !fin_count || !fin_step ||
        !fin_parent || !fin_sum || !fin_score || !out_tok || !out_score || !out_len || !out_avg || !out_n)
        return set_error(E2E_ERR_ARG, "e2e_beam_finalize: null pointer");
    if (U <= 0 || B <= 0 || fin_cap <= 0 || out_cap <= 0) return set_error(E2E_ERR_ARG, "e2e_beam_finalize: bad size");
    FinalParams p;
    p.U = U; p.B = B; p.max_len = max_len; p.n_live = n_live; p.score_sum = score_sum;
    p.hist_tok = hist_tok; p.hist_parent = hist_parent; p.hist_score = hist_score;
    p.fin_count = fin_count; p.fin_step = fin_step; p.fin_parent = fin_parent; p.fin_sum = fin_sum; p.fin_score = fin_score;
    p.fin_cap = fin_cap;
    p.out_tok = out_tok; p.out_score = out_score; p.out_len = out_len; p.out_avg = out_avg; p.out_n = out_n; p.out_cap = out_cap;
    beam_finalize_kernel<<<U, 128, 0, static_cast<cudaStream_t>(stream)>>>(p);
    count_launch();
    return check_launch("e2e_beam_finalize");
}
