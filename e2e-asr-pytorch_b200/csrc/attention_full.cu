// Whole location-aware attention step in one kernel (SURVEY.md §8f row f-1):
//     feat   = loc_conv(prev_att)                                 src/module.py:1163 (Conv1d 1->K, 2P+1 taps, zero padded)
//     loc    = tanh(loc_proj(feat^T))                             src/module.py:1163
//     energy = gen_energy(tanh(key + query + loc))                src/module.py:1168
//     attn   = softmax(mask(energy / temperature))                src/module.py:1109-1113
//     ctx    = attn x value                                       src/module.py:1114
// for every hypothesis n = u*B + b of the first n_run utterances.  Nothing of shape
// [U*B, T, *] is ever materialised: per step the kernel reads key/value of each utterance,
// the previous alignments and the queries, and writes the new alignments and contexts.
//
// Two launches, both sized by the work and not by the batch: few long utterances (the tail of a
// decode) are spread over many CTAs, many utterances get one CTA each.
//   kernel A (energies): CTA <-> (utterance, share of its units); the work is cut into warp-sized units (32 consecutive frames) x (NB beam
//     slots) that the warps take round robin, so a 113-frame and an 825-frame utterance keep their
//     lanes equally busy; lane <-> frame.  A unit stages the +-P frame window of its NB previous
//     alignments in warp-private shared memory, runs the K-filter convolution into registers and
//     then walks the A channels: the key arrives channel-major (key_t[u][a][t]: one coalesced
//     128-byte load per channel per warp), the per-channel constants (loc_proj row, gen_energy
//     weight, the B queries) are shared-memory broadcasts.  tanh(x) = 1 - 2/(1 + exp(2x)) through
//     MUFU.EX2 + MUFU.RCP (absolute error ~2e-7); 4 MUFU per (hypothesis, frame, channel) make
//     this phase MUFU/issue bound by construction.  Frames t >= enc_len[u] are never touched.
//     Energies are parked in the output alignment rows (global, L2 resident).
//   kernel B, CTA <-> (utterance, group of beam slots):
//     masked softmax, one warp per beam slot, in place on the alignment rows; then the context:
//     thread <-> 4 output columns, the group's alignments against one pass over the utterance's
//     value rows (16-byte coalesced loads, 4 frames in flight).
// Results do not depend on NB (every hypothesis sees the same operations in the same order).
//
// Multi-head form (H = attention.num_head heads, e2e_attention_loc_heads): the location convolution reads all H
// previous alignments of a hypothesis (Conv1d H->K) into ONE set of K features, which every head shares.  So kernel A
// convolves the H channels into the same f[NB][KP] registers (one head's window staged at a time), and in the channel
// loop computes tanh(loc) once per (hypothesis, frame, channel) and uses it for the H energies: 2 + 2H MUFU per
// (hypothesis, frame, channel) instead of 4H for independent heads.  Kernel B runs one softmax warp per (slot, head)
// row, then the context product, whose (slot, head) rows are taken 8 at a time (8 accumulators per column): with values
// shared by the heads every chunk of 8 rows, of any heads, reads the same value rows, so a CTA's b slots take
// ceil(H*b/8) passes over its utterance's value rows (the single-head kernel: ceil(b/8)); with per-head values (v_proj)
// the rows of one head go together over that head's columns, ceil(b/8) passes per head.  H = 1 is the same template, instantiated as
// the single-head kernel has always been (3 CTAs per SM, every slot of an utterance in one CTA).
#include "common.cuh"
#include <stdlib.h>

namespace e2e {

constexpr int kAfThreads = 256;
constexpr int kAfWarps = kAfThreads / 32;
constexpr int kAfMaxK = 12;
constexpr int kAfMaxB = 32;
constexpr int kAfMaxH = 4;
// Multi-head instances run 2 CTAs per SM (<= 128 registers a thread for f[NB][KP], NB*H accumulators and 4*H keys in
// flight), so a CTA may take a little under half of an SM's 228 KB of shared memory.
constexpr int kAfHeadsMinBlocks = 2;
constexpr size_t kAfHeadsSmemBudget = 112 * 1024;

__device__ __forceinline__ float af_tanh(float x)
{
    const float t = ex2_approx(x * 2.8853900817779268f);      // exp(2x)
    float r;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(1.0f + t));
    return fmaf(-2.0f, r, 1.0f);
}

struct AttFullParams {
    const float *key_t, *value, *query, *prev_att; const int *enc_len;
    const float *w_conv, *w_proj, *w_energy; float b_energy, temperature;
    int B, T, A, K, W, E;
    int H;              // heads: rows [H][T] of a hypothesis in prev_att / attn, blocks of A in query, of [A][T] in key_t
    int v_pitch;        // row pitch of value: E (one value set shared by the heads) or H*E (head h's columns at h*E)
    int v_heads;        // 1: per-head values
    int slot_cta;       // kernel A: beam slots whose queries a CTA stages (B, unless shared memory forces smaller groups)
    int slot_groups;    // kernel A: ceil(B / slot_cta) CTA groups per utterance
    int unit_ctas;      // kernel A: CTAs per (utterance, slot group) (they share its units round robin)
    int slot_ctas;      // kernel B: CTAs per utterance; each takes ceil(B / slot_ctas) beam slots
    float *attn, *ctx;
};

// shared memory (floats): wc [H][W][KP] | cst [A][16] (loc_proj row 0..11, gen_energy weight at 12) |
//                         q [A][H][Bq] | pa [warps][NB][32 + W - 1]
#ifndef E2E_AF_MINBLOCKS
#define E2E_AF_MINBLOCKS 3
#endif
// Value rows in flight per thread in the context product of kernel B (one 16-byte load each).  The product walks an
// utterance's value rows once, sequentially per output column, so it lives on memory-level parallelism: round 1
// measured it at ~4x its HBM floor with 4.  Tuning knob for tools/sweep_prefix_variants.py (the accumulation order,
// hence the result, does not depend on it).
#ifndef E2E_AF_CTX_FRAMES
#define E2E_AF_CTX_FRAMES 8          // measured (profiles/r02_f_attention_ctx_variants.jsonl): 8 rows in flight 267 vs 362 us on 600 x 824 frames, equal on 2620 x 180; 16: slower
#endif
template <int NB, int KP, int H>
__global__ void __launch_bounds__(kAfThreads, H == 1 ? E2E_AF_MINBLOCKS : kAfHeadsMinBlocks)
attention_energy_kernel(const AttFullParams p)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int ug = blockIdx.x / p.unit_ctas, part = blockIdx.x - ug * p.unit_ctas;
    const int u = ug / p.slot_groups, s_lo = (ug - u * p.slot_groups) * p.slot_cta;
    const int T = p.T, A = p.A, K = p.K, W = p.W, P = W / 2, B = p.B;
    const int Bs = min(p.slot_cta, B - s_lo);                 // this CTA's beam slots: s_lo .. s_lo + Bs - 1
    const int Tu = min(p.enc_len[u], T);
    const int Bq = (p.slot_cta + 3) & ~3;                      // query row pitch
    const int win = 32 + W - 1;                                // frames a unit's convolution reads per hypothesis
    float *wc = reinterpret_cast<float *>(smem_raw);
    float4 *cst = reinterpret_cast<float4 *>(wc + ((H * W * KP + 3) & ~3));
    float *qs = reinterpret_cast<float *>(cst + (size_t)A * 4);
    float *pa = qs + (size_t)A * H * Bq + (size_t)warp * NB * win;
    const size_t n0 = (size_t)u * B + s_lo;                    // this CTA's first hypothesis
    float *arow = p.attn + n0 * H * T;                         // its alignment rows [Bs][H][T]

    // ---- stage: filters, per-channel constants, queries ----------------------------------------------
    for (int i = tid; i < H * W * KP; i += kAfThreads) {
        const int h = i / (W * KP), r = i - h * (W * KP);
        const int j = r / KP, k = r - j * KP;
        wc[i] = (k < K) ? __ldg(p.w_conv + ((size_t)k * H + h) * W + j) : 0.0f;      // w_conv [K][H][W]
    }
    for (int a = tid; a < A; a += kAfThreads) {
        float w[16];
#pragma unroll
        for (int k = 0; k < 16; ++k) w[k] = 0.0f;
#pragma unroll
        for (int k = 0; k < kAfMaxK; ++k)
            if (k < K) w[k] = __ldg(p.w_proj + (size_t)a * K + k);
        w[12] = __ldg(p.w_energy + a);
#pragma unroll
        for (int q = 0; q < 4; ++q) cst[a * 4 + q] = make_float4(w[4 * q], w[4 * q + 1], w[4 * q + 2], w[4 * q + 3]);
    }
    for (int i = tid; i < A * H * Bq; i += kAfThreads) {
        const int a = i / (H * Bq), r = i - a * (H * Bq);
        const int h = r / Bq, b = r - h * Bq;
        qs[i] = (b < Bs) ? __ldg(p.query + ((n0 + b) * H + h) * A + a) : 0.0f;        // query [n][H*A]
    }
    __syncthreads();

    // ---- energies, warp-sized units (frame tile, NB beam slots) ---------------------------------------
    const int n_tiles = (Tu + 31) / 32, n_groups = (Bs + NB - 1) / NB;
    for (int unit = part + warp * p.unit_ctas; unit < n_tiles * n_groups; unit += kAfWarps * p.unit_ctas) {
        const int tile = unit / n_groups, g = unit - tile * n_groups;
        const int t0 = tile * 32, b0 = g * NB;                 // b0: first slot of the unit, relative to s_lo
        const int t = t0 + lane;
        // location features: f[b][k] = sum_h sum_j w_conv[k][h][j] * prev_att[b][h][t + j - P], one head's window at a time
        float f[NB][KP];                                       // read only by lanes with t < Tu
        for (int h = 0; h < H; ++h) {
            __syncwarp();                                      // the previous window is no longer read
            for (int i = lane; i < NB * win; i += 32) {
                const int b = i / win, tt = t0 - P + (i - b * win);
                pa[i] = (b0 + b < Bs && tt >= 0 && tt < Tu) ? __ldg(p.prev_att + ((n0 + b0 + b) * H + h) * T + tt) : 0.0f;
            }
            __syncwarp();
            if (t < Tu) {
                if (h == 0) {
#pragma unroll
                    for (int b = 0; b < NB; ++b)
#pragma unroll
                        for (int k = 0; k < KP; ++k) f[b][k] = 0.0f;
                }
                const float *pat = pa + lane;
                const float *wch = wc + h * W * KP;
#pragma unroll 2
                for (int j = 0; j < W; ++j) {
                    float wj[KP];
#pragma unroll
                    for (int k2 = 0; k2 < KP / 2; ++k2) {
                        const float2 w2 = *reinterpret_cast<const float2 *>(wch + j * KP + 2 * k2);
                        wj[2 * k2] = w2.x; wj[2 * k2 + 1] = w2.y;
                    }
#pragma unroll
                    for (int b = 0; b < NB; ++b) {
                        const float a = pat[b * win + j];
#pragma unroll
                        for (int k = 0; k < KP; ++k) f[b][k] = fmaf(wj[k], a, f[b][k]);
                    }
                }
            }
        }
        if (t < Tu) {
            const float *kcol = p.key_t + (size_t)u * H * A * T + t;    // key_t[u][h][a][t]: coalesced across the warp's frames
            float acc[NB][H];
#pragma unroll
            for (int b = 0; b < NB; ++b)
#pragma unroll
                for (int h = 0; h < H; ++h) acc[b][h] = p.b_energy;
            for (int a4 = 0; a4 < A / 4; ++a4) {
                float kk[4][H];
#pragma unroll
                for (int i = 0; i < 4; ++i)
#pragma unroll
                    for (int h = 0; h < H; ++h) kk[i][h] = __ldg(kcol + ((size_t)h * A + a4 * 4 + i) * T);
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    const int a = a4 * 4 + i;
                    const float4 c0 = cst[a * 4], c1 = cst[a * 4 + 1], c2 = cst[a * 4 + 2], c3 = cst[a * 4 + 3];
                    const float wp[kAfMaxK] = {c0.x, c0.y, c0.z, c0.w, c1.x, c1.y, c1.z, c1.w, c2.x, c2.y, c2.z, c2.w};
                    const float we = c3.x;
                    float qq[H][NB];
#pragma unroll
                    for (int h = 0; h < H; ++h) {
                        const float *qa = qs + ((size_t)a * H + h) * Bq + b0;
                        if (NB == 4) {
                            const float4 q4 = *reinterpret_cast<const float4 *>(qa);
                            qq[h][0] = q4.x; qq[h][1 % NB] = q4.y; qq[h][2 % NB] = q4.z; qq[h][3 % NB] = q4.w;
                        } else if (NB == 2) {
                            const float2 q2 = *reinterpret_cast<const float2 *>(qa);
                            qq[h][0] = q2.x; qq[h][1 % NB] = q2.y;
                        } else {
                            qq[h][0] = qa[0];
                        }
                    }
#pragma unroll
                    for (int b = 0; b < NB; ++b) {
                        float loc = wp[0] * f[b][0];
#pragma unroll
                        for (int k = 1; k < KP; ++k) loc = fmaf(wp[k], f[b][k], loc);
                        const float tl = af_tanh(loc);                  // shared by the H heads
#pragma unroll
                        for (int h = 0; h < H; ++h) {
                            const float x = (kk[i][h] + qq[h][b]) + tl;
                            acc[b][h] = fmaf(we, af_tanh(x), acc[b][h]);
                        }
                    }
                }
            }
#pragma unroll
            for (int b = 0; b < NB; ++b)
                if (b0 + b < Bs)
#pragma unroll
                    for (int h = 0; h < H; ++h) arow[((size_t)(b0 + b) * H + h) * T + t] = __fdiv_rn(acc[b][h], p.temperature);
        }
    }
}

// kernel B: masked softmax + context for beam slots [b_lo, b_hi) of one utterance
__global__ void __launch_bounds__(kAfThreads)
attention_softmax_context_kernel(const AttFullParams p)
{
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int u = blockIdx.x / p.slot_ctas, part = blockIdx.x - u * p.slot_ctas;
    const int T = p.T, B = p.B, H = p.H, E = p.E;
    const int Tu = min(p.enc_len[u], T);
    const int per = (B + p.slot_ctas - 1) / p.slot_ctas;
    const int b_lo = part * per, b_hi = min(B, b_lo + per);
    float *arow = p.attn + (size_t)u * B * H * T;              // this utterance's alignment rows [B][H][T]

    // ---- masked softmax over t, one warp per (beam slot, head) row (module.py:1109-1113) ----------------
    for (int r = b_lo * H + warp; r < b_hi * H; r += kAfWarps) {
        float *row = arow + (size_t)r * T;
        float m = -INFINITY;
        for (int t = lane; t < Tu; t += 32) m = fmaxf(m, row[t]);
        m = warp_max(m);
        float sum = 0.0f;
        for (int t = lane; t < Tu; t += 32) {
            const float e = expf(row[t] - m);
            row[t] = e;
            sum += e;
        }
        sum = warp_sum(sum);
        for (int t = lane; t < T; t += 32) row[t] = (t < Tu) ? __fdiv_rn(row[t], sum) : 0.0f;
    }
    __syncthreads();

    // ---- ctx[b][h*E + e] = sum_t attn[b][h][t] * value_h[u][t][e]  (module.py:1114) ---------------------
    // Row r = b*H + h of the alignments is row r of ctx viewed as [B*H][E].  Rows that read the same value columns are
    // chunked together, 8 rows per pass over the value rows: all (slot, head) rows when the heads share the values
    // (ceil(H*b/8) passes), the slots of one head (row step H, that head's columns) with per-head values.
    // thread <-> 4 consecutive columns (one 16-byte load per frame, whole row coalesced), 4 frames in flight;
    // rows in chunks of 8 accumulators per column
    const int n_sets = p.v_heads ? H : 1, rs = p.v_heads ? H : 1;
    const int rows = p.v_heads ? b_hi - b_lo : (b_hi - b_lo) * H;
    const int vp_ = p.v_pitch;
    constexpr int kBC = 8;
    const bool t_vec = (T & 3) == 0;
    for (int hs = 0; hs < n_sets; ++hs) {
        const float *vbase = p.value + (size_t)u * T * vp_ + (size_t)hs * E;
        const int r0 = b_lo * H + hs;
        for (int bc = 0; bc < rows; bc += kBC) {
            const int nb = min(kBC, rows - bc);
            const float *ar = arow + (size_t)(r0 + bc * rs) * T;
            float *co = p.ctx + ((size_t)u * B * H + r0 + bc * rs) * E;
            if ((E & 3) == 0) {
                for (int e = tid * 4; e < E; e += kAfThreads * 4) {
                    float acc[kBC][4];
    #pragma unroll
                    for (int b = 0; b < kBC; ++b)
    #pragma unroll
                        for (int i = 0; i < 4; ++i) acc[b][i] = 0.0f;
                    const float *vp = vbase + e;
                    int t = 0;
                    constexpr int kF = E2E_AF_CTX_FRAMES;                        // multiple of 4
                    for (; t + kF <= Tu; t += kF) {
                        float4 v[kF];
    #pragma unroll
                        for (int q = 0; q < kF; ++q) v[q] = __ldg(reinterpret_cast<const float4 *>(vp + (size_t)(t + q) * vp_));
    #pragma unroll
                        for (int b = 0; b < kBC; ++b) {
                            if (b < nb) {
    #pragma unroll
                                for (int q0 = 0; q0 < kF; q0 += 4) {
                                    float a[4];
                                    if (t_vec) {                                 // broadcast load (L1), 16 bytes when rows are aligned
                                        const float4 a4 = *reinterpret_cast<const float4 *>(ar + (size_t)b * rs * T + t + q0);
                                        a[0] = a4.x; a[1] = a4.y; a[2] = a4.z; a[3] = a4.w;
                                    } else {
    #pragma unroll
                                        for (int q = 0; q < 4; ++q) a[q] = ar[(size_t)b * rs * T + t + q0 + q];
                                    }
    #pragma unroll
                                    for (int q = 0; q < 4; ++q) {
                                        acc[b][0] = fmaf(a[q], v[q0 + q].x, acc[b][0]); acc[b][1] = fmaf(a[q], v[q0 + q].y, acc[b][1]);
                                        acc[b][2] = fmaf(a[q], v[q0 + q].z, acc[b][2]); acc[b][3] = fmaf(a[q], v[q0 + q].w, acc[b][3]);
                                    }
                                }
                            }
                        }
                    }
                    for (; t < Tu; ++t) {
                        const float4 v = __ldg(reinterpret_cast<const float4 *>(vp + (size_t)t * vp_));
    #pragma unroll
                        for (int b = 0; b < kBC; ++b) {
                            if (b < nb) {
                                const float a = ar[(size_t)b * rs * T + t];
                                acc[b][0] = fmaf(a, v.x, acc[b][0]); acc[b][1] = fmaf(a, v.y, acc[b][1]);
                                acc[b][2] = fmaf(a, v.z, acc[b][2]); acc[b][3] = fmaf(a, v.w, acc[b][3]);
                            }
                        }
                    }
    #pragma unroll
                    for (int b = 0; b < kBC; ++b)
                        if (b < nb)
                            *reinterpret_cast<float4 *>(co + (size_t)b * rs * E + e) = make_float4(acc[b][0], acc[b][1], acc[b][2], acc[b][3]);
                }
            } else {
                for (int e = tid; e < E; e += kAfThreads) {
                    float acc[kBC];
    #pragma unroll
                    for (int b = 0; b < kBC; ++b) acc[b] = 0.0f;
                    const float *vp = vbase + e;
                    for (int t = 0; t < Tu; ++t) {
                        const float v = __ldg(vp + (size_t)t * vp_);
    #pragma unroll
                        for (int b = 0; b < kBC; ++b)
                            if (b < nb) acc[b] = fmaf(ar[(size_t)b * rs * T + t], v, acc[b]);
                    }
    #pragma unroll
                    for (int b = 0; b < kBC; ++b)
                        if (b < nb) co[(size_t)b * rs * E + e] = acc[b];
                }
            }
        }
    }
}

// Shared memory of kernel A (bytes): NB slots a warp carries, KP filter registers, H heads, Bs slots a CTA stages.
static size_t att_full_smem(int NB, int KP, int H, int A, int W, int Bs)
{
    const size_t Bq = (size_t)((Bs + 3) & ~3);
    return ((size_t)((H * W * KP + 3) & ~3) + (size_t)A * 16 + (size_t)A * H * Bq + (size_t)kAfWarps * NB * (32 + W - 1) + 8) * 4;
}

static int att_full_kp(int K) { return K <= 4 ? 4 : (K <= 8 ? 8 : (K <= 10 ? 10 : 12)); }
static int att_full_max_nb(int H) { return H <= 2 ? 4 : 2; }      // registers: NB*KP features + NB*H accumulators

// The ONE place that decides whether and how a shape launches (the launcher and e2e_attention_loc_heads_supported
// both call it).  H = 1: every slot of an utterance in one CTA, up to 200 KB.  H > 1: kAfHeadsSmemBudget; when the
// queries of all B slots do not fit, the slots are cut into CTA groups of slot_cta (a multiple of NB).  Returns
// false when not even one group of NB slots fits.
static bool att_full_plan(int NB, int KP, int H, int A, int W, int B, int *slot_cta, size_t *smem)
{
    if (H == 1) {
        *slot_cta = B;
        *smem = att_full_smem(NB, KP, 1, A, W, B);
        return *smem <= 200 * 1024;
    }
    int bs = B;
    while (bs > 0 && att_full_smem(NB, KP, H, A, W, bs) > kAfHeadsSmemBudget) bs = (bs == B ? (B - 1) / NB * NB : bs - NB);
    *slot_cta = bs;
    *smem = att_full_smem(NB, KP, H, A, W, bs > 0 ? bs : 1);
    return bs > 0;
}

template <int NB, int H>
static int att_full_launch(AttFullParams &p, int KP, int n_run, cudaStream_t st, const char *what)
{
    void (*kern)(AttFullParams) = nullptr;
    switch (KP) {
        case 4: kern = attention_energy_kernel<NB, 4, H>; break;
        case 8: kern = attention_energy_kernel<NB, 8, H>; break;
        case 10: kern = attention_energy_kernel<NB, 10, H>; break;
        default: kern = attention_energy_kernel<NB, 12, H>; break;
    }
    int bs;
    size_t smem;
    if (!att_full_plan(NB, KP, H, p.A, p.W, p.B, &bs, &smem))
        return set_error(E2E_ERR_UNSUPPORTED, "%s: %zu bytes of shared memory needed", what, smem);
    if (smem > 48 * 1024) {
        cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return set_error(E2E_ERR_LAUNCH, "cudaFuncSetAttribute: %s", cudaGetErrorString(e));
    }
    p.slot_cta = bs;
    p.slot_groups = (p.B + bs - 1) / bs;
    // Enough CTAs to cover the machine a few times over whatever the number of utterances: an utterance's
    // units (kernel A) and beam slots (kernel B) are shared out over more CTAs when few utterances are live.
    const int want = 3 * 148;
    const int groups = n_run * p.slot_groups;
    const int max_units = ((p.T + 31) / 32) * ((bs + NB - 1) / NB);
    int ua = (want + groups - 1) / groups;
    ua = ua < 1 ? 1 : (ua > (max_units + kAfWarps - 1) / kAfWarps ? (max_units + kAfWarps - 1) / kAfWarps : ua);
    int ub = (want + n_run - 1) / n_run;
    ub = ub < 1 ? 1 : (ub > p.B ? p.B : ub);
    p.unit_ctas = ua;
    p.slot_ctas = ub;
    kern<<<(unsigned)(groups * ua), kAfThreads, smem, st>>>(p);
    attention_softmax_context_kernel<<<(unsigned)(n_run * ub), kAfThreads, 0, st>>>(p);
    count_launch(2);
    return check_launch(what);
}

template <int H>
static int att_full_launch_nb(AttFullParams &p, int NB, int KP, int n_run, cudaStream_t st, const char *what)
{
    if (NB == 4 && att_full_max_nb(H) >= 4) return att_full_launch<(H <= 2 ? 4 : 2), H>(p, KP, n_run, st, what);
    if (NB >= 2) return att_full_launch<2, H>(p, KP, n_run, st, what);
    return att_full_launch<1, H>(p, KP, n_run, st, what);
}

static void att_full_params(AttFullParams &p, const float *key_t, const float *value, const float *query, const float *prev_att,
                            const int *enc_len, const float *w_conv, const float *w_proj, const float *w_energy, float b_energy,
                            float temperature, int B, int H, int T, int A, int K, int W, int E, int v_heads, float *attn, float *ctx)
{
    p.key_t = key_t; p.value = value; p.query = query; p.prev_att = prev_att; p.enc_len = enc_len;
    p.w_conv = w_conv; p.w_proj = w_proj; p.w_energy = w_energy; p.b_energy = b_energy; p.temperature = temperature;
    p.B = B; p.T = T; p.A = A; p.K = K; p.W = W; p.E = E;
    p.H = H; p.v_heads = v_heads; p.v_pitch = v_heads ? H * E : E;
    p.attn = attn; p.ctx = ctx;
}

}  // namespace e2e

extern "C" int e2e_attention_loc_full(const float *key_t, const float *value, const float *query, const float *prev_att,
                                      const int *enc_len, const float *w_conv, const float *w_proj, const float *w_energy,
                                      float b_energy, float temperature, int n_run, int B, int T, int A, int K, int W, int E,
                                      int hyps_per_unit, float *attn, float *ctx, void *stream)
{
    using namespace e2e;
    if (!key_t || !value || !query || !prev_att || !enc_len || !w_conv || !w_proj || !w_energy || !attn || !ctx)
        return set_error(E2E_ERR_ARG, "e2e_attention_loc_full: null pointer");
    if (n_run <= 0 || B <= 0 || T <= 0 || A <= 0 || K <= 0 || W <= 0 || E <= 0) return set_error(E2E_ERR_ARG, "e2e_attention_loc_full: bad size");
    if (K > kAfMaxK || (A & 3) != 0 || (W & 1) == 0 || B > kAfMaxB)
        return set_error(E2E_ERR_UNSUPPORTED, "e2e_attention_loc_full: needs loc_kernel_num <= 12, dim %% 4 == 0, an odd filter length and beam <= 32");
    if ((reinterpret_cast<uintptr_t>(value) & 15) || (reinterpret_cast<uintptr_t>(ctx) & 15) || (reinterpret_cast<uintptr_t>(attn) & 15))
        return set_error(E2E_ERR_ARG, "e2e_attention_loc_full: value, attn and ctx must be 16-byte aligned");
    int NB = hyps_per_unit;
    if (NB <= 0) NB = n_run >= 2 * 148 ? 4 : 2;       // big launches: more reuse per constant load; small ones: more units
    if (NB != 1 && NB != 2 && NB != 4) return set_error(E2E_ERR_ARG, "e2e_attention_loc_full: hyps_per_unit must be 0, 1, 2 or 4");
    while (NB > 1 && NB / 2 >= B) NB /= 2;
    AttFullParams p;
    att_full_params(p, key_t, value, query, prev_att, enc_len, w_conv, w_proj, w_energy, b_energy, temperature, B, 1, T, A, K, W, E, 0,
                    attn, ctx);
    return att_full_launch_nb<1>(p, NB, att_full_kp(K), n_run, static_cast<cudaStream_t>(stream), "e2e_attention_loc_full");
}

extern "C" int e2e_attention_loc_heads_supported(int B, int H, int A, int K, int W)
{
    using namespace e2e;
    if (B <= 0 || H <= 0 || A <= 0 || K <= 0 || W <= 0) return 0;
    if (H > kAfMaxH || K > kAfMaxK || (A & 3) != 0 || (W & 1) == 0 || B > kAfMaxB) return 0;
    int bs;
    size_t smem;
    return att_full_plan(1, att_full_kp(K), H, A, W, B, &bs, &smem) ? 1 : 0;     // the launcher narrows NB down to 1 if it must
}

extern "C" int e2e_attention_loc_heads(const float *key_t, const float *value, const float *query, const float *prev_att,
                                       const int *enc_len, const float *w_conv, const float *w_proj, const float *w_energy,
                                       float b_energy, float temperature, int n_run, int B, int H, int T, int A, int K, int W, int E,
                                       int per_head_values, int hyps_per_unit, float *attn, float *ctx, void *stream)
{
    using namespace e2e;
    if (!key_t || !value || !query || !prev_att || !enc_len || !w_conv || !w_proj || !w_energy || !attn || !ctx)
        return set_error(E2E_ERR_ARG, "e2e_attention_loc_heads: null pointer");
    if (n_run <= 0 || B <= 0 || H <= 0 || T <= 0 || A <= 0 || K <= 0 || W <= 0 || E <= 0)
        return set_error(E2E_ERR_ARG, "e2e_attention_loc_heads: bad size");
    if (per_head_values != 0 && per_head_values != 1) return set_error(E2E_ERR_ARG, "e2e_attention_loc_heads: per_head_values must be 0 or 1");
    if (hyps_per_unit != 0 && hyps_per_unit != 1 && hyps_per_unit != 2 && hyps_per_unit != 4)
        return set_error(E2E_ERR_ARG, "e2e_attention_loc_heads: hyps_per_unit must be 0, 1, 2 or 4");
    if (!e2e_attention_loc_heads_supported(B, H, A, K, W))
        return set_error(E2E_ERR_UNSUPPORTED, "e2e_attention_loc_heads: unsupported shape (B=%d H=%d A=%d K=%d W=%d): needs heads <= %d, "
                         "loc_kernel_num <= 12, dim %% 4 == 0, an odd filter length, beam <= 32 and the staging within shared memory",
                         B, H, A, K, W, kAfMaxH);
    if ((reinterpret_cast<uintptr_t>(value) & 15) || (reinterpret_cast<uintptr_t>(ctx) & 15) || (reinterpret_cast<uintptr_t>(attn) & 15))
        return set_error(E2E_ERR_ARG, "e2e_attention_loc_heads: value, attn and ctx must be 16-byte aligned");
    int NB = hyps_per_unit > 0 ? hyps_per_unit : (n_run >= 2 * 148 ? 4 : 2);
    if (NB > att_full_max_nb(H)) NB = att_full_max_nb(H);
    while (NB > 1 && NB / 2 >= B) NB /= 2;
    const int KP = att_full_kp(K);
    int bs;
    size_t smem;
    while (NB > 1 && !att_full_plan(NB, KP, H, A, W, B, &bs, &smem)) NB /= 2;
    AttFullParams p;
    att_full_params(p, key_t, value, query, prev_att, enc_len, w_conv, w_proj, w_energy, b_energy, temperature, B, H, T, A, K, W, E,
                    H > 1 ? per_head_values : 0, attn, ctx);
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const char *what = "e2e_attention_loc_heads";
    switch (H) {
        case 1: return att_full_launch_nb<1>(p, NB, KP, n_run, st, what);
        case 2: return att_full_launch_nb<2>(p, NB, KP, n_run, st, what);
        case 3: return att_full_launch_nb<3>(p, NB, KP, n_run, st, what);
        default: return att_full_launch_nb<4>(p, NB, KP, n_run, st, what);
    }
}
