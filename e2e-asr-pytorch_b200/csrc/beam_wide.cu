// (3b) for beams up to 64: score blend, <eos> threshold, top-B per parent, pooled length-normalised prune to B, beam
// bookkeeping (src/decode.py:134-177,214-263) — what beam_combine_prune_kernel (beam_step.cu) does for beams up to 32, with
// the same fp32 operations per score in the same order, so at B <= 32 both give the same bits.
//
// The narrow kernel gives every parent its own warp (B*32 threads) and ranks every child against every other child
// ((B^2)^2 compares).  Here one CTA per utterance still does the whole step, but
//   * a CTA of nw <= 32 warps loops over the parents (warp w takes w, w + nw, ...), so the per-warp shared memory (the
//     candidate ids, the top-B list and, for wide rows, the streaming lists) is paid nw times, not B times;
//   * a child's rank in the pooled stable sort is its index k in its own parent's list plus, for every other parent, a
//     binary search in that parent's list.  A parent's children come out of the top-B selection in descending score, and
//     their keys (sum + s) / (step + 1) are monotone in s in fp32 (both roundings are monotone), so every list is
//     already sorted by (key desc, k asc).  B^2 * B * log2(B) compares instead of B^4.
#include "beam_select.cuh"

namespace e2e {

constexpr int kWideMaxB = 64;
constexpr size_t kWideSmemCap = 200 * 1024;

// shared words: children [5][B*B] (tok, lane, score, sum, key) + cnt, term, term_sc, par_tok [B] ...
__host__ __device__ inline size_t wide_fixed_words(int B) { return (size_t)5 * B * B + 4 * B; }
// ... + per warp: candidate ids and deltas [C], the parent's top-B (value, id), and for the one-pass selection of wide rows
// the per-lane top-B lists [B][32] x (value, id) and the candidate bitmap [ceil(V/32)]
__host__ __device__ inline size_t wide_warp_words(int B, int C, int V, bool stream)
{
    const int Cc = C > 0 ? C : 1;
    return (size_t)2 * Cc + 2 * B + (stream ? (size_t)2 * B * 32 + (size_t)((V + 31) / 32) : 0);
}

// NV > 0 (V <= 32 * NV): every lane holds its NV blended scores in registers; NV == 0: one streaming pass per parent;
// NV < 0: any width without per-lane lists, the scores are re-evaluated in every top-k round.
template <int NV>
__global__ void __launch_bounds__(1024)
beam_combine_prune_wide_kernel(const CombineParams p)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int u = blockIdx.x;
    const int B = p.B, C = p.C, V = p.V;
    const int Cc = C > 0 ? C : 1;
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5, nw = blockDim.x >> 5;
    int *out_parent = p.parent_slot + (long long)u * B;
    if (p.step >= p.max_len[u]) {
        for (int i = threadIdx.x; i < B; i += blockDim.x) {
            out_parent[i] = i;
            if (p.parent_row) p.parent_row[(long long)u * B + i] = (long long)u * B + i;
        }
        return;
    }
    const bool use_ctc = (p.flags & E2E_BEAM_USE_CTC) != 0, use_lm = (p.flags & E2E_BEAM_USE_LM) != 0;
    const int live = p.n_live[u];

    int *c_tok = reinterpret_cast<int *>(smem_raw);
    int *c_lane = c_tok + B * B;
    float *c_score = reinterpret_cast<float *>(c_lane + B * B);
    float *c_sum = c_score + B * B;
    float *c_key = c_sum + B * B;
    int *cnt = reinterpret_cast<int *>(c_key + B * B);
    int *term = cnt + B;
    float *term_sc = reinterpret_cast<float *>(term + B);
    int *par_tok = reinterpret_cast<int *>(term_sc + B);
    int *wbase = par_tok + B + w * (int)wide_warp_words(B, C, V, NV == 0);
    int *mycand = wbase;
    float *mydelta = reinterpret_cast<float *>(mycand + Cc);
    float *tv = mydelta + Cc;
    int *ti = reinterpret_cast<int *>(tv + B);
    float *lv = reinterpret_cast<float *>(ti + B);             // NV == 0 only
    int *li = reinterpret_cast<int *>(lv + B * 32);
    const int bit_words = (V + 31) >> 5;
    unsigned *bits = reinterpret_cast<unsigned *>(li + B * 32);

    for (int i = threadIdx.x; i < B; i += blockDim.x) {
        cnt[i] = 0; term[i] = 0;
        par_tok[i] = (p.step > 0 && i < live) ? p.last_tok[u * B + i] : -1;
    }
    __syncthreads();

    // The eos test looks at the pure attention log-probs when CTC is on; with CTC off the reference's in-place "+=" of the
    // LM term aliases them (SURVEY.md §8a-Q2).
    const bool alias = (!use_ctc) && use_lm;
    const float denom = (float)(p.step + 1);
    for (int b = w; b < live; b += nw) {                       // warp-uniform
        const int n = u * B + b;
        const float *att = p.att_logits + (long long)n * p.ld_att;
        const float2 ast = p.att_stats[n];
        const float *lm = use_lm ? p.lm_logits + (long long)n * p.ld_lm : nullptr;
        float lmx = 0.0f, llse = 0.0f;
        if (use_lm) warp_row_stats(lm, V, lane, lmx, llse);
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
        auto keep_top = [&](int r, float val, int idx) { if (lane == 0) { tv[r] = val; ti[r] = idx; } };
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
            warp_select_topk_cached<NV>(bval, V, B, lane, keep_top);
            best_other = warp_max(best_other);
            eos_lp = __shfl_sync(E2E_FULL_MASK, eos_lp, E2E_CTC_EOS & 31);
        } else if constexpr (NV < 0) {
            warp_select_topk(V, B, lane, blended, keep_top);
            for (int v = 2 + lane; v < V; v += 32)
                best_other = fmaxf(best_other, alias ? blended(v) : logp_from(__ldg(att + v), ast.x, ast.y));
            best_other = warp_max(best_other);
            if (V > 1) eos_lp = alias ? blended(E2E_CTC_EOS) : logp_from(__ldg(att + E2E_CTC_EOS), ast.x, ast.y);
        } else {
            // one pass: every entry is blended once, feeds this lane's top-B list and the <eos> scan; a bitmap of the
            // candidate ids replaces the C compares per entry
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
            warp_select_topk_stream(V, B, lane, visit, keep_top, lv, li);
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
                    term[b] = 1;
                    term_sc[b] = sc;
                    continue;
                }
                int jsel = 0;
                if (use_ctc) {
                    jsel = -1;
                    for (int j = 0; j < C; ++j)
                        if (mycand[j] == tok) { jsel = j; break; }
                    if (jsel < 0) {                         // reference: ValueError at decode.py:252
                        if (p.status) atomicOr(p.status + u, E2E_STATUS_TOKEN_NOT_CAND);
                        jsel = 0;
                    }
                }
                const int slot = b * B + made;
                c_tok[slot] = tok;
                c_lane[slot] = b * Cc + jsel;
                c_score[slot] = sc;
                c_sum[slot] = (p.step == 0) ? sc : __fadd_rn(parent_sum, sc);      // python sum(): 0 + s0 + s1 ...
                c_key[slot] = __fdiv_rn(c_sum[slot], denom);                       // avgScore, decode.py:214-217
                ++made;
            }
            cnt[b] = made;
        }
        __syncwarp();                                       // the next parent overwrites this warp's lists
    }
    __syncthreads();

    // ---- closed hypotheses (decode.py:167-170): parent order, only once step >= min_len ---------
    // Kept stably sorted by mean score and truncated to fin_cap >= B entries, as in beam_combine_prune_kernel.
    if (threadIdx.x == 0 && p.step >= p.min_len[u]) {
        int fc = p.fin_count[u];
        const long long base = (long long)u * p.fin_cap;
        for (int b = 0; b < live; ++b) {
            if (!term[b]) continue;
            const float ps = p.score_sum[u * B + b];
            const float fsum = (p.step == 0) ? term_sc[b] : __fadd_rn(ps, term_sc[b]);
            const float key = __fdiv_rn(fsum, denom);
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

    // ---- pooled prune: stable sort by mean score in (parent, k-th child) list order, keep B (decode.py:175-176) ------
    int total = 0;
    for (int b = 0; b < live; ++b) total += cnt[b];
    const int keep = total < B ? total : B;
    const long long hrow = ((long long)p.step * p.U + u) * B;
    for (int i = threadIdx.x; i < B * B; i += blockDim.x) {
        const int b = i / B, k = i - b * B;
        if (b >= live || k >= cnt[b]) continue;
        const float key = c_key[i];
        // before (b, k): the k earlier children of its own parent, and from parent b2 every child with a larger key, or an
        // equal one when b2 < b — a prefix of b2's list, found by binary search
        int rank = k;
        for (int b2 = 0; b2 < live; ++b2) {
            if (b2 == b) continue;
            const float *kl = c_key + b2 * B;
            int lo = 0, hi = cnt[b2];
            if (b2 < b) {
                while (lo < hi) { const int mid = (lo + hi) >> 1; if (kl[mid] >= key) lo = mid + 1; else hi = mid; }
            } else {
                while (lo < hi) { const int mid = (lo + hi) >> 1; if (kl[mid] > key) lo = mid + 1; else hi = mid; }
            }
            rank += lo;
            if (rank >= B) break;
        }
        if (rank < B) {
            const int o = u * B + rank;
            const int jsel = c_lane[i] - b * Cc;
            p.last_tok[o] = c_tok[i];
            if (p.last_tok64) p.last_tok64[o] = c_tok[i];
            if (p.parent_row) p.parent_row[o] = (long long)u * B + b;
            if (p.parent_tok) p.parent_tok[o] = par_tok[b];
            p.prefix_len[o] = p.step + 1;
            p.score_sum[o] = c_sum[i];
            p.ctc_prob[o] = use_ctc ? p.psi[(long long)(u * B + b) * C + jsel] : 0.0f;
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

}  // namespace e2e

extern "C" int e2e_beam_combine_prune_wide(const float *att_logits, int ld_att, const float *att_stats,
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
        return set_error(E2E_ERR_ARG, "e2e_beam_combine_prune_wide: null pointer");
    if ((use_lm && !lm_logits) || (use_ctc && (!cand || !psi || C <= 0)))
        return set_error(E2E_ERR_ARG, "e2e_beam_combine_prune_wide: flags need lm_logits / cand+psi");
    if (U <= 0 || B <= 0 || B > kWideMaxB || V <= 0 || step < 0 || fin_cap <= 0 || ld_att < V || (use_lm && ld_lm < V))
        return set_error(E2E_ERR_ARG, "e2e_beam_combine_prune_wide: bad size (beam size must be 1..%d)", kWideMaxB);
    if (fin_cap < B) return set_error(E2E_ERR_ARG, "e2e_beam_combine_prune_wide: fin_cap must be >= B");
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

    // as many warps as parents (at most 32) or as fit next to the children's arrays
    const size_t fixed = wide_fixed_words(B) * 4 + 16;
    auto warps_fitting = [&](bool stream) -> int {
        const size_t per = wide_warp_words(B, p.C, V, stream) * 4;
        if (fixed + per > kWideSmemCap) return 0;
        const size_t fit = (kWideSmemCap - fixed) / per;
        const int want = B < 32 ? B : 32;
        return fit < (size_t)want ? (int)fit : want;
    };
    const bool stream_sel = V > 128 && warps_fitting(true) > 0;
    const int warps = warps_fitting(stream_sel);
    if (warps == 0)
        return set_error(E2E_ERR_UNSUPPORTED, "e2e_beam_combine_prune_wide: B=%d, C=%d, V=%d needs more than %zu bytes of shared memory",
                         B, p.C, V, kWideSmemCap);
    const size_t smem = fixed + (size_t)warps * wide_warp_words(B, p.C, V, stream_sel) * 4;
    if (n_run <= 0 || n_run > U) n_run = U;
    void (*kern)(CombineParams) = V <= 32 ? beam_combine_prune_wide_kernel<1> : V <= 64 ? beam_combine_prune_wide_kernel<2>
                                : V <= 128 ? beam_combine_prune_wide_kernel<4> : stream_sel ? beam_combine_prune_wide_kernel<0>
                                : beam_combine_prune_wide_kernel<-1>;
    if (smem > 48 * 1024) {
        cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return set_error(E2E_ERR_LAUNCH, "cudaFuncSetAttribute: %s", cudaGetErrorString(e));
    }
    kern<<<n_run, warps * 32, smem, static_cast<cudaStream_t>(stream)>>>(p);
    count_launch();
    return check_launch("e2e_beam_combine_prune_wide");
}
