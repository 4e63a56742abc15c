// Device helpers shared by the (3b) combine/prune kernels of beam_step.cu (beams up to 32) and beam_wide.cu (up to 64):
// row statistics, the three top-k selections (ties to the lower index) and the kernels' parameter block.
#pragma once
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

}  // namespace e2e
