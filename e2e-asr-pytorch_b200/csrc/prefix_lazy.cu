// Kernel (2), batched beam-search form: ONE fused launch per decode step that
//   (a) brings the prefix state r of every LIVE hypothesis up to date (B chains per utterance), and
//   (b) scores all B*C candidate extensions (psi only).
// Replaces CTCPrefixScore.cheap_compute (src/ctc.py:68-108) as src/decode.py:131 calls it, with LAZY state
// evaluation (SURVEY.md §7.2-5): psi of an extension only needs the state of its PARENT (src/ctc.py:103), and of the
// B*C states cheap_compute builds only the <= B the beam keeps are ever read again (src/decode.py:250-254).  So the
// state of a hypothesis is computed once, one step later, when it has survived the prune — by the same sequential
// fp32 recurrence over the same frames, hence the same bits — and the B*C candidate lanes run the psi reduction alone:
//     state lanes (B per utterance)  r0' = logaddexp(r0, phi_parent) + x[t][tok]    r1' = logaddexp(r1, r0) + x[t][blank]
//     psi lanes (B*C per utterance)  psi = logaddexp(psi, phi_hyp[t-1] + x[t][cand])
// Per utterance-frame that is 2B + B*C log-add-exp chain steps (+ 2B for the phi values) instead of 3*B*C, and 8B bytes
// of state written instead of 8*B*C (12x less at C = 12).  The byte figure of SURVEY.md §8d (12 + 12/C per
// candidate-frame) stays the unit the roofline is reported in; the DRAM traffic actually moved is measured beside it.
//
// The recursion is sequential in t, so a launch is bound either by instruction issue (machine-filling launches) or by
// the latency of ONE dependent log-add-exp per frame (the tail of a decode: few long utterances).  Both ask for the
// same thing: chain warps whose instruction stream is the chain and nothing else.  One CTA per utterance, three kinds
// of warps, all meeting at one __syncthreads per tile of kT frames:
//   * STATE warps (8 hypotheses each, 4 lanes per hypothesis): lane role 0 carries the r0 chain, role 1 the r1 chain
//     one frame behind it — r1[t] needs r0[t-1], which travels by a shuffle issued a whole iteration before it is
//     consumed, so no shuffle latency sits on the chain.  Operands (phi of the parent, x) are loaded four frames ahead;
//     results go to a shared-memory tile only.
//   * HELPER warps (one per state warp) do everything else, one tile ahead / behind: the TMA box copies of the
//     posterior rows (ring of 4, mbarrier completion), cp.async (LDGSTS) staging of the parents' states and their
//     conversion to phi_parent = logaddexp(r0, r1) (r1 alone for a repeated token), the conversion of the finished
//     state tile into (sum, blank) pairs for the psi lanes, and its coalesced write-out to the step's state buffer.
//   * PSI warps (one lane per (hypothesis, candidate)) run two tiles behind the state warps.
// Large vocabularies (Vp > 256): every chain lane fetches its own column of x with 4-byte cp.async, double buffered.
// All live hypotheses of an utterance have the same length s (the decode step), so the first frame is uniform per CTA.
// Step 0 (s == 0): the hypothesis is the empty prefix, whose state is the init buffer itself (passed as r_prev).
#include "common.cuh"
#include <string.h>
#include <cuda.h>

namespace e2e {

struct LazyParams {
    const float *x; int Tmax, U, Vp, V;
    const int *enc_len;
    const float2 *r_prev; int lanes_prev;
    const int *parent_slot, *last_tok, *parent_tok, *prefix_len, *n_live, *cand;
    int B, C, flags;
    float *psi; float2 *r_out; int *status;
    int state_warps, psi_warps;
};

constexpr int kLazyMaxRowFloats = 256;

__host__ __device__ constexpr int lazy_pair_pitch(int tile) { return 2 * tile + 2; }

struct LazySmem {
    size_t xs, cur, pairs, pphi, stage, misc, bars, total;
};
__host__ __device__ inline LazySmem lazy_smem_layout(bool gather, int math, int threads, int Vp, int B, int tile)
{
    LazySmem s;
    size_t off = (math == kMathLut) ? (size_t)kLutNodes * kLutCopies * 16 : 0;
    off = (off + 127) & ~(size_t)127;
    s.xs = off;
    off += gather ? (size_t)2 * tile * threads * 4 : (size_t)4 * tile * Vp * 4;
    off = (off + 127) & ~(size_t)127;
    s.cur = off;      off += (size_t)2 * (tile + 1) * B * 8;
    s.pairs = off;    off += (size_t)2 * B * lazy_pair_pitch(tile) * 4;
    s.stage = off;    off += (size_t)2 * B * tile * 8;
    s.pphi = off;     off += (size_t)2 * B * (tile + 1) * 4;
    s.misc = off;     off += (size_t)(2 * B) * 4;
    off = (off + 7) & ~(size_t)7;
    s.bars = off;     off += 4 * 8;
    s.total = (off + 15) & ~(size_t)15;
    return s;
}

__device__ __forceinline__ void lazy_tma_load_tile(void *dst_smem, const CUtensorMap *map, int u, int t0, uint64_t *bar)
{
    asm volatile("cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];"
                 ::"r"(smem_u32(dst_smem)), "l"(reinterpret_cast<uint64_t>(map)), "r"(0), "r"(u), "r"(t0), "r"(smem_u32(bar))
                 : "memory");
}
__device__ __forceinline__ void lazy_cp_async_8(void *dst_smem, const void *src)
{
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(smem_u32(dst_smem)), "l"(src) : "memory");
}
__device__ __forceinline__ void lazy_cp_async_4(void *dst_smem, const void *src)
{
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(smem_u32(dst_smem)), "l"(src) : "memory");
}
__device__ __forceinline__ void lazy_cp_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void lazy_cp_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

#ifndef E2E_LAZY_MINBLOCKS
#define E2E_LAZY_MINBLOCKS 6
#endif

// kGather: column-gather staging of x (large vocabularies).  kFixed: the shape the beam search runs all day
// (Vp = 32, B = 8, C = 12: one state, one helper and three psi warps) with every stride an immediate.
// kT: frames per tile.  kBig: CTAs of more than 160 threads (beam sizes whose lanes need more than 5 warps).
template <bool kGather, int kMath, bool kFixed, int kT, bool kBig>
__global__ void __launch_bounds__(kBig ? 1024 : 160, kBig ? 1 : E2E_LAZY_MINBLOCKS)
prefix_lazy_kernel(const LazyParams p, const __grid_constant__ CUtensorMap tmap)
{
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const int tid = threadIdx.x, nt = blockDim.x, lane = tid & 31, wid = tid >> 5;
    const int u = blockIdx.x;
    const int T = p.enc_len ? p.enc_len[u] : p.Tmax;
    const int live = p.n_live ? p.n_live[u] : p.B;
    const int B = kFixed ? 8 : p.B, C = kFixed ? 12 : p.C, Vp = kFixed ? 32 : p.Vp;
    const int SW = kFixed ? 1 : p.state_warps;
    if (T <= 0 || live <= 0) return;                    // idle utterance (uniform exit)
    const int s = p.prefix_len[u * B];                  // length of every live hypothesis of this utterance
    const int start_h = s > 1 ? s : 1;                  // first frame of the psi reduction    (src/ctc.py:78)
    const int start_p = s > 2 ? s - 1 : 1;              // first frame of the state recurrence (the parents' start)
    const bool passthrough = s == 0;                    // the hypothesis IS the empty prefix: its state is r_prev
    constexpr int kPairP = lazy_pair_pitch(kT);
    const int sB2 = 2 * B;                              // floats per row of a state tile

    const LazySmem L = lazy_smem_layout(kGather, kMath, nt, Vp, B, kT);
    float4 *lut_base = reinterpret_cast<float4 *>(smem_raw);
    float *xs = reinterpret_cast<float *>(smem_raw + L.xs);
    float2 *cur = reinterpret_cast<float2 *>(smem_raw + L.cur);
    float *pairs = reinterpret_cast<float *>(smem_raw + L.pairs);
    float2 *stage = reinterpret_cast<float2 *>(smem_raw + L.stage);
    float *pphi = reinterpret_cast<float *>(smem_raw + L.pphi);
    int *s_pslot = reinterpret_cast<int *>(smem_raw + L.misc);
    int *s_spec = s_pslot + B;
    uint64_t *bars = reinterpret_cast<uint64_t *>(smem_raw + L.bars);
    const uint32_t lut = softplus_lut_adj(lut_base + (tid & (kLutCopies - 1)));
    const float2 dead = make_float2(E2E_CTC_LOGZERO, E2E_CTC_LOGZERO);

    const bool is_state = wid < SW;
    const bool is_helper = !is_state && wid < 2 * SW;
    const bool is_psi = wid >= 2 * SW;
    // ---- too long: the reference raises IndexError at psi = r[start-1, 0, :] (src/ctc.py:85) ----------------------
    if (start_h - 1 >= T) {
        if (tid == 0 && p.status) atomicOr(p.status + u, E2E_STATUS_PREFIX_TOO_LONG);
        if (is_psi) {
            const int pl = (wid - 2 * SW) * 32 + lane;
            if (pl < live * C) p.psi[(long long)u * B * C + pl] = E2E_CTC_LOGZERO;
        }
        return;
    }

    // ---- per-lane setup ---------------------------------------------------------------------------------------------
    // state lanes: 4 lanes per hypothesis
    const int hh = lane >> 2, role = lane & 3;
    const int hs = wid * 8 + hh;                                  // hypothesis (beam slot) of a state lane
    const int hs_c = hs < B ? hs : B - 1;                         // clamped: keeps idle lanes' addresses inside the tiles
    const bool s_act = is_state && hs < live && role < 2;
    int s_tok = 0;
    // helper lanes
    const int hw = wid - SW;                                      // serves hypotheses hw*8 .. hw*8+7
    // psi lanes
    const int pw = wid - 2 * SW;
    const int pl = pw * 32 + lane;                                // lane within the utterance: h*C + j
    const bool p_act = is_psi && pl < live * C;
    const int ph = p_act ? pl / C : 0;
    const int pj = p_act ? pl - ph * C : 0;
    int c_tok = 0;
    bool p_spec = false;
    if (is_state) {
        if (hs < live) {
            const int n = u * B + hs;
            s_tok = p.last_tok[n];
            if (role == 0) {
                s_pslot[hs] = p.parent_slot[n];
                s_spec[hs] = (s >= 2 && p.parent_tok && s_tok == p.parent_tok[n]) ? 1 : 0;    // repeated token (src/ctc.py:89-91)
            }
        } else if (hs < B && role == 0) {
            s_pslot[hs] = 0;
            s_spec[hs] = 0;
        }
    } else if (p_act) {
        const int n = u * B + ph;
        c_tok = p.cand[(long long)n * C + pj];
        p_spec = s > 0 && c_tok == p.last_tok[n];
    }
    if (kMath == kMathLut) softplus_lut_to_smem(lut_base, tid, nt);
    if (!kGather && tid == 0) {
        mbar_init(&bars[0], 1);
        mbar_init(&bars[1], 1);
        mbar_init(&bars[2], 1);
        mbar_init(&bars[3], 1);
        mbar_fence_init();
    }
    __syncthreads();

    const long long xrow0 = (long long)u * Vp;
    const long long xstride = (long long)p.U * Vp;
    const int jl = (T - 1) / kT;                                  // last tile
    const int j0s = start_p / kT;                                 // first tile of the state warps
    const int j0p = start_h / kT;                                 // first tile of the psi warps (j0s or j0s + 1)
    const int first_row = start_p - 1;                            // first state row that exists (the row before the first computed frame)
    const float2 *__restrict__ rprev_u = p.r_prev + ((long long)u * p.Tmax) * p.lanes_prev;
    float2 *__restrict__ rout_u = p.r_out + ((long long)u * p.Tmax) * B;
    const bool x_issuer = !kGather && tid == SW * 32;             // lane 0 of helper warp 0

    // posterior tile j -> ring stage j & 3 (rows variant)
    auto issue_x = [&](int j) {
        uint64_t *bar = &bars[j & 3];
        mbar_arrive_expect_tx(bar, (uint32_t)kT * Vp * 4u);
        lazy_tma_load_tile(xs + (size_t)(j & 3) * kT * Vp, &tmap, u, j * kT, bar);
    };
    auto wait_x = [&](int j) { mbar_wait(&bars[j & 3], (uint32_t)(((j - j0s) >> 2) & 1)); };
    // gather variant: this chain lane's column of tile j -> its own slots of stage j & 1
    const int my_col = is_state ? (role == 0 ? s_tok : E2E_CTC_BLANK) : c_tok;
    auto fetch_col = [&](int j) {
        const int t0 = j * kT, rows = min(kT, T - t0);
        float *dst = xs + (size_t)(j & 1) * kT * nt + tid;
        const float *src = p.x + (long long)t0 * xstride + xrow0 + my_col;
        for (int tt = 0; tt < rows; ++tt) lazy_cp_async_4(dst + tt * nt, src + (long long)tt * xstride);
    };
    // helper: raw parent states of tile j (entry (eh, tt) <-> frame j*kT + tt - 1) -> staging slot j & 1
    auto fetch_parents = [&](int j) {
        float2 *dst = stage + ((size_t)(j & 1) * B + hw * 8) * kT;
#pragma unroll
        for (int e = lane; e < 8 * kT; e += 32) {
            const int eh = e / kT, tt = e - eh * kT;
            const int hyp = hw * 8 + eh, ts = j * kT + tt - 1;
            if (hyp < live && ts >= 0 && ts < T) lazy_cp_async_8(dst + e, rprev_u + (long long)ts * p.lanes_prev + s_pslot[hyp]);
            else if (hyp < B) dst[e] = dead;
        }
    };
    // helper: phi of the parents for tile j: logaddexp(r0, r1), or r1 alone for a repeated token
    auto convert_parents = [&](int j) {
        const float2 *src = stage + ((size_t)(j & 1) * B + hw * 8) * kT;
        float *dst = pphi + ((size_t)(j & 1) * B + hw * 8) * (kT + 1);
#pragma unroll
        for (int e = lane; e < 8 * kT; e += 32) {
            const int eh = e / kT, tt = e - eh * kT;
            const int hyp = hw * 8 + eh;
            if (hyp < B) {
                const float2 a = src[e];
                const float sum = logaddexp<kMath>(a.x, a.y, lut);
                dst[eh * (kT + 1) + tt] = s_spec[hyp] ? a.y : sum;
            }
        }
    };
    // helper: finished state tile j -> (sum, blank) pairs for the psi lanes + the step's state buffer (coalesced)
    auto publish_tile = [&](int j) {
        const int t0 = j * kT;
        const float2 *cb = cur + (size_t)(j & 1) * (kT + 1) * B;
        float *pb = pairs + (size_t)(j & 1) * B * kPairP;
#pragma unroll
        for (int e = lane; e < 8 * kT; e += 32) {
            const int tt = e >> 3, eh = e & 7;
            const int hyp = hw * 8 + eh, ts = t0 + tt - 1;          // entry tt <-> state row t0 + tt - 1
            if (hyp < B) {
                float2 a;
                if (passthrough) a = (hyp < live && ts >= 0 && ts < T) ? __ldg(rprev_u + (long long)ts * p.lanes_prev + s_pslot[hyp]) : dead;
                else a = cb[tt * B + hyp];
                *reinterpret_cast<float2 *>(pb + hyp * kPairP + 2 * tt) = make_float2(logaddexp<kMath>(a.x, a.y, lut), a.y);
                if (!passthrough && hyp < live && ts >= first_row && ts < T) rout_u[(long long)ts * B + hyp] = a;
            }
        }
        if (!passthrough && j == jl && lane < 8) {                  // the last row (its r1 came from the drain step)
            const int hyp = hw * 8 + lane;
            if (hyp < live) rout_u[(long long)(T - 1) * B + hyp] = cb[(T - t0) * B + hyp];
        }
    };

    // ---- prologue ---------------------------------------------------------------------------------------------------
    if (x_issuer) issue_x(j0s);
    if (is_helper && !passthrough) {
        fetch_parents(j0s);
        lazy_cp_commit();
        lazy_cp_wait<0>();
        __syncwarp();
        convert_parents(j0s);
        if (j0s + 1 <= jl) fetch_parents(j0s + 1);
        lazy_cp_commit();
    }
    if (kGather) {
        if (is_state && !passthrough) { fetch_col(j0s); lazy_cp_commit(); }
        if (is_psi && j0p <= jl) { fetch_col(j0p); lazy_cp_commit(); }
    }
    // chain registers.  state lanes: v = r0 (role 0) / r1 (role 1, one frame behind); s0_prev = r0 two frames back (what
    // role 1 needs); xl_prev = x[t-1][blank] for role 1.  The initial values make role 1's first (warm-up) step log-zero.
    float v = E2E_CTC_LOGZERO, s0_prev = E2E_CTC_LOGZERO, xl_prev = 0.0f;
    if (is_state && !passthrough && role == 0 && s == 1 && hs < live)
        v = __ldg(p.x + xrow0 + s_tok);                            // r[0,0] = x[0,c] for an extension of the empty prefix (src/ctc.py:82-83)
    float psi = E2E_CTC_LOGZERO;
    if (p_act && s == 0) psi = __ldg(p.x + xrow0 + c_tok);        // psi = r[start-1,0,:] (src/ctc.py:85)
    __syncthreads();

    // iteration k: state warps chain tile k+1, helpers prepare tile k+2's parents and publish tile k, psi warps chain tile k-1
    for (int k = j0s - 1; k <= jl + 1; ++k) {
        if (is_state) {
            const int j = k + 1;
            if (j <= jl && !passthrough) {
                const int t0 = j * kT, rows = min(kT, T - t0);
                float2 *cb = cur + (size_t)(j & 1) * (kT + 1) * B;
                int tt = 0;
                if (j == j0s) {
                    tt = start_p - t0;
                    if (role == 0 && s_act) cb[tt * B + hs].x = v;    // the row before the first computed frame: (x[0,c] | log-zero, .)
                } else if (role == 0 && s_act) {
                    cb[hs].x = v;                                   // r0 of the last frame of the previous tile
                }
                const float *xp;
                int xstep;
                if (kGather) {
                    if (j + 1 <= jl) fetch_col(j + 1);
                    lazy_cp_commit();
                    lazy_cp_wait<1>();
                    xp = xs + (size_t)(j & 1) * kT * nt + tid; xstep = nt;
                } else {
                    wait_x(j);
                    xp = xs + (size_t)(j & 3) * kT * Vp + (role == 0 ? s_tok : E2E_CTC_BLANK); xstep = Vp;
                }
                const float *php = pphi + ((size_t)(j & 1) * B + hs_c) * (kT + 1) + tt;
                float *sp_ptr = reinterpret_cast<float *>(cb + hs_c) + (role == 0 ? sB2 : 1) + tt * sB2;   // role 0: row tt+1 .x; role 1: row tt .y
                xp += tt * xstep;
                const int src0 = lane & ~3;
                auto frame = [&](float phv, float xl, int q) {
                    const float s0n = __shfl_sync(E2E_FULL_MASK, v, src0);
                    const float b = role == 0 ? phv : s0_prev;
                    const float add = role == 0 ? xl : xl_prev;
                    v = __fadd_rn(logaddexp<kMath>(v, b, lut), add);
                    if (s_act) sp_ptr[q * sB2] = v;
                    s0_prev = s0n;
                    xl_prev = xl;
                };
                if (tt + 4 <= rows) {
                    // groups of four frames, software pipelined: the operands of the NEXT group are loaded before the current
                    // group's chain is issued, so no shared-memory latency is exposed between groups
                    float ph4[4], x4[4];
#pragma unroll
                    for (int q = 0; q < 4; ++q) { ph4[q] = php[q]; x4[q] = xp[q * xstep]; }
                    for (; tt + 8 <= rows; tt += 4) {
                        float pn[4], xn[4];
#pragma unroll
                        for (int q = 0; q < 4; ++q) { pn[q] = php[4 + q]; xn[q] = xp[(4 + q) * xstep]; }
#pragma unroll
                        for (int q = 0; q < 4; ++q) frame(ph4[q], x4[q], q);
#pragma unroll
                        for (int q = 0; q < 4; ++q) { ph4[q] = pn[q]; x4[q] = xn[q]; }
                        php += 4; xp += 4 * xstep; sp_ptr += 4 * sB2;
                    }
#pragma unroll
                    for (int q = 0; q < 4; ++q) frame(ph4[q], x4[q], q);
                    php += 4; xp += 4 * xstep; sp_ptr += 4 * sB2;
                    tt += 4;
                }
                for (; tt < rows; ++tt) {
                    frame(php[0], xp[0], 0);
                    php += 1; xp += xstep; sp_ptr += sB2;
                }
                if (j == jl) {
                    // drain: r1 of the last frame (role 0 has nothing left to do)
                    const float r1_last = __fadd_rn(logaddexp<kMath>(v, s0_prev, lut), xl_prev);
                    if (role == 1 && s_act) sp_ptr[0] = r1_last;
                }
            }
        } else if (is_helper) {
            if (x_issuer && k + 2 >= j0s + 1 && k + 2 <= jl) issue_x(k + 2);    // reuses the stage of tile k-2
            if (!passthrough) {
                lazy_cp_wait<0>();
                __syncwarp();
                if (k + 2 <= jl && k + 2 > j0s) convert_parents(k + 2);
                if (k + 3 <= jl) fetch_parents(k + 3);
                lazy_cp_commit();
            }
            if (k >= j0s && k <= jl) publish_tile(k);
        } else {
            const int j = k - 1;
            if (j >= j0p && j >= j0s && j <= jl) {
                const int t0 = j * kT, rows = min(kT, T - t0);
                const float *xp;
                int xstep;
                if (kGather) {
                    if (j + 1 <= jl) fetch_col(j + 1);
                    lazy_cp_commit();
                    lazy_cp_wait<1>();
                    xp = xs + (size_t)(j & 1) * kT * nt + tid; xstep = nt;
                } else {
                    wait_x(j);
                    xp = xs + (size_t)(j & 3) * kT * Vp + c_tok; xstep = Vp;
                }
                if (p_act) {
                    int tt = (j == j0p) ? start_h - t0 : 0;
                    const float *php = pairs + ((size_t)(j & 1) * B + ph) * kPairP + (p_spec ? 1 : 0) + 2 * tt;
                    xp += tt * xstep;
                    if (tt + 4 <= rows) {
                        float a4[4];                                   // software pipelined like the state loop
#pragma unroll
                        for (int q = 0; q < 4; ++q) a4[q] = __fadd_rn(php[2 * q], xp[q * xstep]);
                        for (; tt + 8 <= rows; tt += 4) {
                            float an[4];
#pragma unroll
                            for (int q = 0; q < 4; ++q) an[q] = __fadd_rn(php[8 + 2 * q], xp[(4 + q) * xstep]);
#pragma unroll
                            for (int q = 0; q < 4; ++q) psi = logaddexp<kMath>(psi, a4[q], lut);
#pragma unroll
                            for (int q = 0; q < 4; ++q) a4[q] = an[q];
                            php += 8; xp += 4 * xstep;
                        }
#pragma unroll
                        for (int q = 0; q < 4; ++q) psi = logaddexp<kMath>(psi, a4[q], lut);
                        php += 8; xp += 4 * xstep;
                        tt += 4;
                    }
                    for (; tt < rows; ++tt) {
                        psi = logaddexp<kMath>(psi, __fadd_rn(php[0], xp[0]), lut);
                        php += 2; xp += xstep;
                    }
                }
            }
        }
        __syncthreads();
    }

    if (p_act) {
        if (c_tok == E2E_CTC_EOS) {                                   // P(<eos> | g) = P(g)   (src/ctc.py:106-107)
            float2 a;
            if (passthrough) a = __ldg(rprev_u + (long long)(T - 1) * p.lanes_prev + s_pslot[ph]);
            else a = cur[(size_t)(jl & 1) * (kT + 1) * B + (T - jl * kT) * B + ph];
            psi = logaddexp<kMath>(a.x, a.y, lut);
        }
        p.psi[(long long)(u * B + ph) * C + pj] = psi;
    }
}

typedef void (*LazyKernel)(LazyParams, CUtensorMap);

int make_posterior_map_lazy(CUtensorMap *map, const float *x, int Tmax, int U, int Vp, int tile);   // prefix_score.cu

template <bool kGather, bool kFixed, int kT, bool kBig>
static LazyKernel pick_math(int math)
{
    if (math == kMathPoly) return prefix_lazy_kernel<kGather, kMathPoly, kFixed, kT, kBig>;
    if (math == kMathPolyEstrin) return prefix_lazy_kernel<kGather, kMathPolyEstrin, kFixed, kT, kBig>;
    return prefix_lazy_kernel<kGather, kMathLut, kFixed, kT, kBig>;
}

constexpr size_t kLazySmemCap = 200 * 1024;

// The frame tile of a launch: 16-frame tiles for machine-filling launches (more CTAs per SM), 32-frame tiles for the tail
// (fewer barriers per chain) unless their shared memory exceeds the cap (the column-gather form at beams 18-23 and wider
// rows of candidates); 0 when not even the 16-frame tile fits.
static int lazy_tile(bool gather, int math, int threads, int Vp, int B, bool machine_filling)
{
    if (!machine_filling && lazy_smem_layout(gather, math, threads, Vp, B, 32).total <= kLazySmemCap) return 32;
    return lazy_smem_layout(gather, math, threads, Vp, B, 16).total <= kLazySmemCap ? 16 : 0;
}
}  // namespace e2e

extern "C" int e2e_ctc_prefix_step_supported(int Vp, int B, int C)
{
    using namespace e2e;
    if (B <= 0 || C <= 0 || Vp <= 0) return 0;
    const int SW = (B + 7) / 8, PW = (B * C + 31) / 32;
    if (2 * SW + PW > 32) return 0;
    // the table form of the log-add-exp needs the most shared memory: what fits with it fits with every math
    return lazy_tile(Vp > kLazyMaxRowFloats, kMathLut, (2 * SW + PW) * 32, Vp, B, true) > 0 ? 1 : 0;
}

extern "C" int e2e_ctc_prefix_step(const float *x, int Tmax, int U, int Vp, int V, const int *enc_len,
                                   const float *r_prev, int lanes_prev,
                                   const int *parent_slot, const int *last_tok, const int *parent_tok, const int *prefix_len,
                                   const int *n_live, const int *cand, int B, int C, int flags,
                                   float *psi, float *r_out, int *status, int n_run, void *stream)
{
    using namespace e2e;
    if (!x || !r_prev || !parent_slot || !last_tok || !prefix_len || !cand || !psi || !r_out)
        return set_error(E2E_ERR_ARG, "e2e_ctc_prefix_step: null pointer");
    if (Tmax <= 0 || U <= 0 || V <= 0 || B <= 0 || C <= 0 || lanes_prev <= 0)
        return set_error(E2E_ERR_ARG, "e2e_ctc_prefix_step: non-positive size");
    if (Vp != e2e_padded_vocab(V)) return set_error(E2E_ERR_ARG, "e2e_ctc_prefix_step: Vp=%d, expected %d", Vp, e2e_padded_vocab(V));
    if ((reinterpret_cast<uintptr_t>(x) & 15) || (reinterpret_cast<uintptr_t>(r_out) & 7) || (reinterpret_cast<uintptr_t>(r_prev) & 7))
        return set_error(E2E_ERR_ARG, "e2e_ctc_prefix_step: misaligned buffer");
    if (!e2e_ctc_prefix_step_supported(Vp, B, C))
        return set_error(E2E_ERR_UNSUPPORTED, "e2e_ctc_prefix_step: B=%d, C=%d needs more than 32 warps per utterance (use e2e_ctc_prefix_score)", B, C);
    if (flags & (E2E_PREFIX_FAST_MATH | E2E_PREFIX_LIBM_MATH | E2E_PREFIX_FULL))
        return set_error(E2E_ERR_UNSUPPORTED, "e2e_ctc_prefix_step: only the table and polynomial log-add-exp are built for the fused step");
    if (n_run <= 0 || n_run > U) n_run = U;

    LazyParams p;
    p.x = x; p.Tmax = Tmax; p.U = U; p.Vp = Vp; p.V = V; p.enc_len = enc_len;
    p.r_prev = reinterpret_cast<const float2 *>(r_prev); p.lanes_prev = lanes_prev;
    p.parent_slot = parent_slot; p.last_tok = last_tok; p.parent_tok = parent_tok; p.prefix_len = prefix_len;
    p.n_live = n_live; p.cand = cand; p.B = B; p.C = C; p.flags = flags;
    p.psi = psi; p.r_out = reinterpret_cast<float2 *>(r_out); p.status = status;
    p.state_warps = (B + 7) / 8;
    p.psi_warps = (B * C + 31) / 32;
    const int threads = (2 * p.state_warps + p.psi_warps) * 32;
    const bool big = threads > 160;
    const bool gather = Vp > kLazyMaxRowFloats;
    const bool fixed = !gather && Vp == 32 && B == 8 && C == 12;     // char vocabulary, beam 8 (BASELINE cfg2)
    // Polynomial log-add-exp: Horner (14 instructions, 10 dependent after the MUFU) for machine-filling launches, which are
    // bound by instruction issue; the pairwise (Estrin) evaluation (17 instructions, 6 dependent) for launches that cannot
    // fill the machine and last as long as the longest utterance's dependent chain.  E2E_PREFIX_POLY_ESTRIN forces the latter.
    static const int estrin_below = []() {
        const char *e = getenv("E2E_LAZY_ESTRIN_BELOW");             // tuning knob: utterances below which Estrin is used
        return e ? atoi(e) : 200;        // measured (profiles/r02_i_prefix_micro_estrin.jsonl): -10 % at 64 utterances, +6 % at 600
    }();
    const int math = (flags & E2E_PREFIX_POLY_MATH) ? (((flags & E2E_PREFIX_POLY_ESTRIN) || n_run < estrin_below) ? kMathPolyEstrin : kMathPoly) : kMathLut;
    static const int small_from = []() {
        const char *e = getenv("E2E_LAZY_SMALL_TILE_FROM");          // tuning knob: utterances from which the 16-frame tile is used
        return e ? atoi(e) : 1500;       // measured: 16-frame tiles win from ~1500 utterances up, 32-frame tiles below (profiles/r02_e_prefix_micro_tiles.jsonl)
    }();
    // (64-frame tiles were measured for the deep tail — profiles/r02_o_prefix_micro_tiles64.jsonl: 1-4 % slower than 32; not built)
    const int tile = lazy_tile(gather, math, threads, Vp, B, n_run >= small_from);
    if (tile == 0) return set_error(E2E_ERR_UNSUPPORTED, "e2e_ctc_prefix_step: B=%d, Vp=%d needs more shared memory than a CTA has", B, Vp);
    LazyKernel kern;
    if (fixed) kern = tile == 16 ? pick_math<false, true, 16, false>(math) : pick_math<false, true, 32, false>(math);
    else if (gather) kern = tile == 16 ? (big ? pick_math<true, false, 16, true>(math) : pick_math<true, false, 16, false>(math))
                                       : (big ? pick_math<true, false, 32, true>(math) : pick_math<true, false, 32, false>(math));
    else kern = tile == 16 ? (big ? pick_math<false, false, 16, true>(math) : pick_math<false, false, 16, false>(math))
                           : (big ? pick_math<false, false, 32, true>(math) : pick_math<false, false, 32, false>(math));
    const LazySmem L = lazy_smem_layout(gather, math, threads, Vp, B, tile);
    CUtensorMap map;
    memset(&map, 0, sizeof(map));
    if (!gather) {
        const int rc = make_posterior_map_lazy(&map, x, Tmax, U, Vp, tile);
        if (rc != E2E_OK) return rc;
    }
    if (L.total > 48 * 1024) {
        cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)L.total);
        if (e != cudaSuccess) return set_error(E2E_ERR_LAUNCH, "cudaFuncSetAttribute: %s", cudaGetErrorString(e));
    }
    kern<<<(unsigned)n_run, threads, L.total, static_cast<cudaStream_t>(stream)>>>(p, map);
    count_launch();
    return check_launch("e2e_ctc_prefix_step");
}
