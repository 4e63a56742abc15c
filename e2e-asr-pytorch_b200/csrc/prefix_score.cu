// Kernel (2): batched CTC prefix-score recursion.
// Replaces CTCPrefixScore.cheap_compute / full_compute (src/ctc.py:29-108) for every live
// (utterance, beam slot, candidate) in one launch.
//
// Mapping.  A prefix-state "lane" l = slot*C + j of one utterance walks the encoder frames
// t = start..T-1 sequentially in fp32 (the reference's order).  Per frame it needs
//     r0' = logaddexp(r0, phi) + x_c      r1' = logaddexp(r1, r0) + x_blank       (the recurrence)
//     psi = logaddexp(psi, phi + x_c)                                              (a running reduction)
// i.e. three log-add-exp that only meet through r0.  The kernel is bound by instruction issue,
// not by HBM (SURVEY.md §7.2-5; DESIGN.md §6), so the layout minimises instructions per
// candidate-frame: ONE thread per lane carries all three chains (the three log-add-exp are
// independent inside a frame, so the thread itself has the instruction-level parallelism that
// hides their latency; the phi and x_c loads are shared by two of them), every per-frame address
// is a constant offset from a pointer that is bumped once per 4 frames, and the state leaves as
// one coalesced float2 per lane per frame.
// A CTA covers up to 128 consecutive lanes of ONE utterance, so its threads share the
// utterance's posterior rows x[t][u][:] and the few parent states.  Frames are processed in
// tiles of kTile:
//   * "rows" variant (Vp <= kMaxRowFloats): the tile's posterior rows are brought into shared
//     memory by the TMA engine, double buffered, completion on an mbarrier, so the gather
//     x[t][cand] becomes a conflict-free LDS.  The tile is a [kTile frames] x [1 utterance] x [Vp]
//     box of the frame-major [T][U][Vp] tensor: ONE cp.async.bulk.tensor (UTMALDG) through a
//     tensor map built by the host wrapper; E2E_PREFIX_ROW_COPIES selects the older form, one
//     cp.async.bulk (UBLKCP) per 16B-aligned row, which costs the issuing warp a 32-trip loop;
//   * "gather" variant (large vocabularies): each thread fetches its own column
//     x[t][u][cand] for the whole tile with independent loads and parks it in shared memory.
//   The parents' states are turned into phi tiles in shared memory once per hypothesis
//     phi[h][t] = ( logaddexp(r_prev[t][0], r_prev[t][1]),  r_prev[t][1] )
//   and are software pipelined without holding registers: the raw states of tile k+1 are
//   copied into a staging buffer with cp.async (LDGSTS) before tile k is computed and turned into
//   phi afterwards, so one __syncthreads per tile is all the synchronisation there is.
#include "common.cuh"
#include <stdlib.h>
#include <string.h>
#include <cuda.h>      // CUtensorMap (types only; the encoder is fetched from the driver at run time)

namespace e2e {

#ifndef E2E_PS_MINBLOCKS
#define E2E_PS_MINBLOCKS 6           // register cap 85: measured 19 % faster than a cap of 64 (tools/sweep_prefix_variants.py)
#endif
#ifndef E2E_PS_UNROLL
#define E2E_PS_UNROLL 4
#endif
// Frames per shared-memory tile (template parameter kT of the kernel): 16 for machine-filling launches (smaller
// tiles -> less shared memory -> more resident CTAs: 0.149 vs 0.162 ms on the 2620-utterance launch), 32 for
// small ones, whose duration is one utterance's chain and which pay per tile (0.083 vs 0.095 ms on 64 x 825 frames).
constexpr int kTileBig = 16, kTileSmall = 32;
__host__ __device__ constexpr int phi_pitch(int tile) { return 2 * tile + 2; }   // floats per phi row: tile x (sum, blank) + pad
constexpr int kMaxRowFloats = 256;   // rows variant up to 1 KB per posterior row
constexpr int kMaxLanes = 128;       // lanes (= threads) per CTA
constexpr int kLutBytes = kLutNodes * kLutCopies * 16;
// the polynomial log-add-exp needs no table: its kernels start their shared-memory layout at offset 0
__host__ __device__ constexpr int lut_bytes(int math) { return (math == kMathPoly || math == kMathPolyEstrin) ? 0 : kLutBytes; }

struct PrefixParams {
    const float *x; int Tmax, U, Vp, V;
    const int *enc_len;
    const float2 *r_prev; int lanes_prev;
    const int *prev_lane, *last_tok, *prefix_len, *n_live, *cand;
    int B, C, flags;
    float *psi; float2 *r_out; int *status;
    int chunks_per_utt;   // CTAs per utterance
    int lanes_per_cta;    // multiple of 32 = blockDim.x
    int hyps_per_cta;     // rows of the phi tile
};

__host__ __device__ inline size_t prefix_xs_bytes(bool gather, int lanes, int Vp, int tile)
{
    // rows: two tiles of posterior rows.  gather: two tiles of per-lane columns + the blank column.
    size_t f = gather ? (size_t)2 * (tile * lanes + tile) : (size_t)2 * tile * Vp;
    return ((f + 31) & ~(size_t)31) * 4;          // 128-byte multiples: TMA destinations stay aligned
}
__host__ __device__ inline size_t prefix_phis_bytes(int H, int tile) { return (size_t)2 * H * phi_pitch(tile) * 4; }
__host__ __device__ inline size_t prefix_stage_bytes(int H, int tile) { return (size_t)H * tile * 8; }   // raw parent states of one tile

// kVp / kLU: compile-time copies of Vp and B*C for the shapes the beam search runs all day
// (0 = take them from the parameters): per-frame offsets then become instruction immediates.
// 3-D tiled TMA load: box (Vp, 1, kTile) at coordinates (0, u, t0) of the [Tmax][U][Vp] posterior tensor.
__device__ __forceinline__ void tma_load_tile(void *dst_smem, const CUtensorMap *map, int u, int t0, uint64_t *bar)
{
    asm volatile("cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];"
                 ::"r"(smem_u32(dst_smem)), "l"(reinterpret_cast<uint64_t>(map)), "r"(0), "r"(u), "r"(t0), "r"(smem_u32(bar))
                 : "memory");
}
__device__ __forceinline__ void cp_async_8(void *dst_smem, const void *src)
{
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(smem_u32(dst_smem)), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_wait_all()
{
    asm volatile("cp.async.wait_all;" ::: "memory");
}

template <bool kGather, int kMath, int kVp, int kLU, bool kTmap, int kT>
__global__ void __launch_bounds__(kMaxLanes, E2E_PS_MINBLOCKS)
prefix_score_kernel(const PrefixParams p, const __grid_constant__ CUtensorMap tmap)
{
    extern __shared__ __align__(128) unsigned char smem_raw[];
    constexpr int kPhiP = phi_pitch(kT);
    const int tid = threadIdx.x, nt = blockDim.x;
    const int nl = nt;
    const int lt = tid;                           // lane index within the CTA
    const int u = blockIdx.x / p.chunks_per_utt;
    const int chunk = blockIdx.x % p.chunks_per_utt;
    const int T = p.enc_len ? p.enc_len[u] : p.Tmax;
    const int live = p.n_live ? p.n_live[u] : p.B;
    const int C = p.C;
    const int LU = kLU ? kLU : p.B * p.C;
    const int Vp = kVp ? kVp : p.Vp;
    const int lane0 = chunk * nl;                 // first lane (within the utterance) of this CTA
    if (T <= 0 || lane0 >= live * C) return;      // nothing to do for this CTA (uniform exit)
    const bool full = (p.flags & E2E_PREFIX_FULL) != 0;
    const bool fill_dead = (p.flags & E2E_PREFIX_SKIP_DEAD_ROWS) == 0;

    // ---- shared memory: LUT replicas | x tiles | phi tiles (x2) | raw parent states | s_plane[H] | s_red[2] | mbarriers[2]
    const int H = p.hyps_per_cta;
    const size_t xs_off = lut_bytes(kMath);
    const size_t phis_off = xs_off + prefix_xs_bytes(kGather, nl, Vp, kT);
    const size_t stage_off = phis_off + prefix_phis_bytes(H, kT);
    const size_t misc_off = stage_off + prefix_stage_bytes(H, kT);
    const size_t bars_off = (misc_off + (size_t)(H + 2) * 4 + 7) & ~(size_t)7;
    float4 *lut_base = reinterpret_cast<float4 *>(smem_raw);
    float *xs = reinterpret_cast<float *>(smem_raw + xs_off);
    float *phis = reinterpret_cast<float *>(smem_raw + phis_off);
    float2 *stage_buf = reinterpret_cast<float2 *>(smem_raw + stage_off);
    int *s_plane = reinterpret_cast<int *>(smem_raw + misc_off);
    int *s_red = s_plane + H;
    uint64_t *bars = reinterpret_cast<uint64_t *>(smem_raw + bars_off);
    const uint32_t lut = softplus_lut_adj(lut_base + (tid & (kLutCopies - 1)));   // this thread's replica
    const int g_tile = kT * nl + kT;                        // gather variant: floats per x tile

    // ---- per-lane setup -----------------------------------------------------------------------
    const int lane_u = lane0 + lt;                // lane within the utterance
    const bool active = lane_u < live * C;
    const int h = active ? lane_u / C : 0;        // beam slot
    const int j = active ? lane_u - h * C : 0;    // candidate index
    const int h_lo = lane0 / C;
    const int n = u * p.B + h;                    // hypothesis index
    int tok = 0, plen = 0, ltok = 0;
    if (active) {
        tok = full ? j : p.cand[(long long)n * C + j];
        plen = p.prefix_len[n];
        ltok = p.last_tok[n];
    }
    const int start = plen > 1 ? plen : 1;
    const bool too_long = active && (start - 1 >= T);
    if (too_long && p.status) atomicOr(p.status + u, E2E_STATUS_PREFIX_TOO_LONG);
    const bool run = active && !too_long;
    const bool special = full ? (tok == (plen > 0 ? ltok : 0)) : (plen > 0 && tok == ltok);

    if (tid == 0) s_red[0] = 0x7fffffff;
    if (kMath == kMathLut) softplus_lut_to_smem(lut_base, tid, nt);
    for (int i = tid; i < H; i += nt) {
        const int hh = h_lo + i;
        s_plane[i] = (hh < live) ? p.prev_lane[u * p.B + hh] : -1;
    }
    if (!kGather && tid == 0) {
        mbar_init(&bars[0], 1);
        mbar_init(&bars[1], 1);
        mbar_fence_init();
    }
    __syncthreads();
    if (run) atomicMin(&s_red[0], start);
    __syncthreads();
    const int cta_start = s_red[0];               // 0x7fffffff if no lane runs
    const long long xrow0 = (long long)u * Vp;    // x[t][u][:] = x + t*U*Vp + xrow0
    const long long xstride = (long long)p.U * Vp;
    float2 *__restrict__ rout = p.r_out + ((long long)u * p.Tmax) * LU + lane_u;
    const float2 *__restrict__ rprev_u = p.r_prev + ((long long)u * p.Tmax) * p.lanes_prev;
    const float2 dead = make_float2(E2E_CTC_LOGZERO, E2E_CTC_LOGZERO);

    float nb = E2E_CTC_LOGZERO, bl = E2E_CTC_LOGZERO;
    if (run && plen == 0) nb = __ldg(p.x + xrow0 + tok);     // r[0,0,:] = x[0, c]  (src/ctc.py:82-83)
    float psi = nb;                                            // psi = r[start-1, 0, :] (src/ctc.py:85)

    if (cta_start != 0x7fffffff) {
        const int first_tile = cta_start / kT;
        const int n_tiles = (T + kT - 1) / kT;
        // rows below the first computed tile are log-zero by construction
        if (run && fill_dead)
            for (int t = 0; t < first_tile * kT && t < T; ++t) rout[(long long)t * LU] = dead;

        auto issue_rows = [&](int k) {   // warp 0 brings posterior tile k into its ring stage
            const int t0 = k * kT;
            uint64_t *bar = &bars[k & 1];
            float *dst = xs + (size_t)(k & 1) * kT * Vp;
            if (kTmap) {
                // one box copy; frames beyond Tmax are zero filled by the TMA unit and still count as bytes
                if (tid == 0) {
                    mbar_arrive_expect_tx(bar, (uint32_t)kT * Vp * 4u);
                    tma_load_tile(dst, &tmap, u, t0, bar);
                }
            } else {
                const int rows = min(kT, T - t0);
                if (tid == 0) mbar_arrive_expect_tx(bar, (uint32_t)rows * Vp * 4u);
                __syncwarp();
                if (tid < rows)
                    bulk_g2s(dst + (size_t)tid * Vp, p.x + (long long)(t0 + tid) * xstride + xrow0, (uint32_t)Vp * 4u, bar);
            }
        };
        // phi tile k, entry (hl, tt) describes r_prev at frame k*kT + tt - 1.  Entry i of a tile is
        // fetched (phi_fetch) and converted (phi_convert) by the same thread, so cp.async.wait_all is
        // all the ordering the staging buffer needs.
        const int n_phi = H * kT;
        auto phi_fetch = [&](int k) {
            for (int i = tid; i < n_phi; i += nt) {
                const int hl = i / kT, tt = i - hl * kT;
                const int ts = k * kT + tt - 1;
                const int pl = s_plane[hl];
                if (pl >= 0 && ts >= 0 && ts < T) cp_async_8(stage_buf + i, rprev_u + (long long)ts * p.lanes_prev + pl);
                else stage_buf[i] = dead;
            }
        };
        auto phi_convert = [&](int k) {
            cp_async_wait_all();
            for (int i = tid; i < n_phi; i += nt) {
                const int hl = i / kT, tt = i - hl * kT;
                const float2 a = stage_buf[i];
                float2 ph;
                ph.x = logaddexp<kMath>(a.x, a.y, lut);
                ph.y = full ? logaddexp<kMath>(E2E_CTC_LOGZERO, a.y, lut) : a.y;
                *reinterpret_cast<float2 *>(phis + (size_t)(k & 1) * H * kPhiP + hl * kPhiP + 2 * tt) = ph;
            }
        };

        if (first_tile < n_tiles) {
            if (!kGather && tid < 32) {
                issue_rows(first_tile);
                if (first_tile + 1 < n_tiles) issue_rows(first_tile + 1);
            }
            phi_fetch(first_tile);
            phi_convert(first_tile);
        }

        // this thread's column inside a phi row (sum or blank-only variant)
        const int phi_col = (h - h_lo) * kPhiP + (special ? 1 : 0);
        uint32_t parity = 0u;                                  // bit s = phase of mbarrier s
        for (int k = first_tile; k < n_tiles; ++k) {
            const int t0 = k * kT;
            const int rows = min(kT, T - t0);
            if (k + 1 < n_tiles) phi_fetch(k + 1);             // in flight while tile k is computed
            const float *xcp, *xbp;   // this thread's candidate column / the blank column of tile row 0
            if (kGather) {
                float *xg = xs + (size_t)(k & 1) * g_tile;     // double buffered: no barrier before the fill
                if (active) {
#pragma unroll 8
                    for (int tt = 0; tt < rows; ++tt)
                        xg[tt * nl + lt] = __ldg(p.x + (long long)(t0 + tt) * xstride + xrow0 + tok);
                }
                if (tid < rows) xg[kT * nl + tid] = __ldg(p.x + (long long)(t0 + tid) * xstride + xrow0 + E2E_CTC_BLANK);
                xcp = xg + lt; xbp = xg + kT * nl;
            } else {
                mbar_wait(&bars[k & 1], (parity >> (k & 1)) & 1u);
                parity ^= 1u << (k & 1);
                const float *xt = xs + (size_t)(k & 1) * kT * Vp;
                xcp = xt + tok; xbp = xt + E2E_CTC_BLANK;
            }
            const int xc_step = kGather ? nl : Vp, xb_step = kGather ? 1 : Vp;
            __syncthreads();    // phi tile k and x tile k visible; all threads have left tile k-1
            if (!kGather && tid < 32 && k > first_tile && k + 1 < n_tiles) issue_rows(k + 1);   // reuses tile k-1's buffer
            if (run) {
                int tt = 0;
                const int tt_first = start - t0;              // first frame of this tile that is computed
                if (tt_first > 0) {
                    const int stop = min(tt_first, rows);
                    // Row 0 of an empty-prefix extension, (x[0,c], logzero), is read back by the child's
                    // first frame (its start is also 1), so it is written even when dead rows are skipped.
                    if (t0 == 0 && plen == 0) rout[0] = make_float2(nb, E2E_CTC_LOGZERO);
                    if (fill_dead)
                        for (; tt < stop; ++tt)
                            if (!(t0 + tt == 0 && plen == 0)) rout[(long long)(t0 + tt) * LU] = dead;
                    tt = stop;
                }
                const float *php = phis + (size_t)(k & 1) * H * kPhiP + phi_col + 2 * tt;
                xcp += tt * xc_step; xbp += tt * xb_step;
                float2 *outp = rout + (long long)(t0 + tt) * LU;
                // 3 LDS, 3 log-add-exp, 1 STG.64 per frame
                auto frame = [&](int q) {
                    const float ph = php[2 * q];
                    const float xc = xcp[q * xc_step];
                    const float xb = xbp[q * xb_step];
                    const float nnb = __fadd_rn(logaddexp<kMath>(nb, ph, lut), xc);
                    const float nbl = __fadd_rn(logaddexp<kMath>(bl, nb, lut), xb);
                    psi = logaddexp<kMath>(psi, __fadd_rn(ph, xc), lut);
                    nb = nnb; bl = nbl;
                    outp[(long long)q * LU] = make_float2(nnb, nbl);
                };
                for (; tt + E2E_PS_UNROLL <= rows; tt += E2E_PS_UNROLL) {
#pragma unroll
                    for (int q = 0; q < E2E_PS_UNROLL; ++q) frame(q);
                    php += 2 * E2E_PS_UNROLL; xcp += E2E_PS_UNROLL * xc_step; xbp += E2E_PS_UNROLL * xb_step;
                    outp += (long long)E2E_PS_UNROLL * LU;
                }
                for (; tt < rows; ++tt) {
                    frame(0);
                    php += 2; xcp += xc_step; xbp += xb_step; outp += LU;
                }
            }
            if (k + 1 < n_tiles) phi_convert(k + 1);           // other phi buffer: nobody reads it before the next barrier
        }
    }

    if (run) {
        const bool eos_lane = !full && tok == E2E_CTC_EOS;       // P(<eos> | g) = P(g)   (src/ctc.py:106-107)
        if (eos_lane) {
            const float2 a = __ldg(rprev_u + (long long)(T - 1) * p.lanes_prev + s_plane[h - h_lo]);
            psi = logaddexp<kMath>(a.x, a.y, lut);
            // psi aliases r[start-1,0,:] in the reference when the time loop never runs (src/ctc.py:85)
            if (start >= T && fill_dead) rout[(long long)(start - 1) * LU] = make_float2(psi, E2E_CTC_LOGZERO);
        }
        p.psi[(long long)n * C + j] = psi;
    } else if (active) {
        p.psi[(long long)n * C + j] = E2E_CTC_LOGZERO;
    }
}

static size_t prefix_smem_bytes(bool gather, int lanes, int Vp, int H, int tile, int math)
{
    size_t b = lut_bytes(math) + prefix_xs_bytes(gather, lanes, Vp, tile) + prefix_phis_bytes(H, tile) + prefix_stage_bytes(H, tile);
    b = ((b + (size_t)(H + 2) * 4 + 7) & ~(size_t)7) + 16;
    return (b + 15) & ~(size_t)15;
}

typedef void (*PrefixKernel)(PrefixParams, CUtensorMap);

// cuTensorMapEncodeTiled, fetched from the driver the process already has loaded (no link-time libcuda).
typedef CUresult (*EncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *, const cuuint64_t *,
                                  const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
EncodeTiledFn tensor_map_encoder()   // also used by conv_igemm.cu
{
    static EncodeTiledFn fn = nullptr;
    static bool tried = false;
    if (!tried) {
        tried = true;
        void *ptr = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<EncodeTiledFn>(ptr);
        else
            cudaGetLastError();
    }
    return fn;
}

// Tensor map of the posterior tensor x [Tmax][U][Vp] (fp32) with a (Vp, 1, tile) box.
static int make_posterior_map(CUtensorMap *map, const float *x, int Tmax, int U, int Vp, int tile)
{
    EncodeTiledFn enc = tensor_map_encoder();
    if (!enc) return set_error(E2E_ERR_LAUNCH, "e2e_ctc_prefix_score: cuTensorMapEncodeTiled is not available from this driver");
    const cuuint64_t dims[3] = {(cuuint64_t)Vp, (cuuint64_t)U, (cuuint64_t)Tmax};
    const cuuint64_t strides[2] = {(cuuint64_t)Vp * 4, (cuuint64_t)U * Vp * 4};
    const cuuint32_t box[3] = {(cuuint32_t)Vp, 1u, (cuuint32_t)tile};
    const cuuint32_t estr[3] = {1u, 1u, 1u};
    const CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, const_cast<float *>(x), dims, strides, box, estr,
                           CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                           CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return set_error(E2E_ERR_LAUNCH, "e2e_ctc_prefix_score: cuTensorMapEncodeTiled failed (CUresult %d)", (int)r);
    return E2E_OK;
}

// the same tensor map for the fused per-step kernel (prefix_lazy.cu)
int make_posterior_map_lazy(CUtensorMap *map, const float *x, int Tmax, int U, int Vp, int tile)
{
    return make_posterior_map(map, x, Tmax, U, Vp, tile);
}

}  // namespace e2e

extern "C" int e2e_ctc_prefix_score(const float *x, int Tmax, int U, int Vp, int V, const int *enc_len,
                                    const float *r_prev, int lanes_prev,
                                    const int *prev_lane, const int *last_tok, const int *prefix_len,
                                    const int *n_live, const int *cand, int B, int C, int flags,
                                    float *psi, float *r_out, int *status, int n_run, void *stream)
{
    using namespace e2e;
    const bool full = (flags & E2E_PREFIX_FULL) != 0;
    if (!x || !r_prev || !prev_lane || !last_tok || !prefix_len || !psi || !r_out || (!full && !cand))
        return set_error(E2E_ERR_ARG, "e2e_ctc_prefix_score: null pointer");
    if (Tmax <= 0 || U <= 0 || V <= 0 || B <= 0 || C <= 0 || lanes_prev <= 0)
        return set_error(E2E_ERR_ARG, "e2e_ctc_prefix_score: non-positive size");
    if (Vp != e2e_padded_vocab(V)) return set_error(E2E_ERR_ARG, "e2e_ctc_prefix_score: Vp=%d, expected %d", Vp, e2e_padded_vocab(V));
    if (full && C != V) return set_error(E2E_ERR_ARG, "e2e_ctc_prefix_score: E2E_PREFIX_FULL needs C == V");
    if ((reinterpret_cast<uintptr_t>(x) & 15) || (reinterpret_cast<uintptr_t>(r_out) & 7) || (reinterpret_cast<uintptr_t>(r_prev) & 7))
        return set_error(E2E_ERR_ARG, "e2e_ctc_prefix_score: misaligned buffer");

    const long long LU = (long long)B * C;
    if (n_run <= 0 || n_run > U) n_run = U;      // only the first n_run utterances are processed
    int nl = (int)((LU + 31) / 32 * 32);
    if (nl > kMaxLanes) {
        // split the utterance's lanes over several CTAs of equal, warp-multiple size
        const int chunks = (int)((LU + kMaxLanes - 1) / kMaxLanes);
        nl = (int)(((LU + chunks - 1) / chunks + 31) / 32 * 32);
    }
    // A small launch cannot fill the machine and its duration is the longest utterance's chain:
    // spread every utterance over one-warp CTAs so that each warp has a scheduler to itself.
    // (Every lane computes the same values whatever the split.)
    static const long long split_below = []() {
        const char *e = getenv("E2E_PREFIX_SPLIT_BELOW");        // tuning knob: CTAs (at full width) below which to split
        return e ? atoll(e) : 2LL * 148;
    }();
    if (nl > 32 && (long long)n_run * ((LU + nl - 1) / nl) < split_below) nl = 32;
    PrefixParams p;
    p.x = x; p.Tmax = Tmax; p.U = U; p.Vp = Vp; p.V = V; p.enc_len = enc_len;
    p.r_prev = reinterpret_cast<const float2 *>(r_prev); p.lanes_prev = lanes_prev;
    p.prev_lane = prev_lane; p.last_tok = last_tok; p.prefix_len = prefix_len; p.n_live = n_live; p.cand = cand;
    p.B = B; p.C = C; p.flags = flags;
    p.psi = psi; p.r_out = reinterpret_cast<float2 *>(r_out); p.status = status;
    p.lanes_per_cta = nl;
    p.chunks_per_utt = (int)((LU + nl - 1) / nl);
    p.hyps_per_cta = (nl + C - 1) / C + 1;
    if (p.hyps_per_cta > B) p.hyps_per_cta = B;
    const long long grid = (long long)n_run * p.chunks_per_utt;
    if (grid > 0x7fffffffLL) return set_error(E2E_ERR_UNSUPPORTED, "e2e_ctc_prefix_score: grid too large");

    const bool gather = Vp > kMaxRowFloats;
    const int math = (flags & E2E_PREFIX_FAST_MATH) ? kMathMufu
                   : (flags & E2E_PREFIX_LIBM_MATH) ? kMathLibm
                   : (flags & E2E_PREFIX_POLY_MATH) ? ((flags & E2E_PREFIX_POLY_ESTRIN) ? kMathPolyEstrin : kMathPoly) : kMathLut;
    const bool fixed = !gather && Vp == 32 && LU == 96;      // char vocabulary, beam 8 (BASELINE cfg2)
    const bool use_map = !gather && !(flags & E2E_PREFIX_ROW_COPIES);
    // Tile size by launch size (only the default-math tensor-map kernels are built with the small tile)
    static const long long small_tile_from = []() {
        const char *e = getenv("E2E_PREFIX_SMALL_TILE_FROM");    // tuning knob: CTAs from which the 16-frame tile is used
        return e ? atoll(e) : 1000LL;
    }();
    const bool tiled_math = math == kMathLut || math == kMathPoly || math == kMathPolyEstrin;      // built with both tile sizes
    const bool big_launch = use_map && tiled_math && grid >= small_tile_from;
    const int tile = big_launch ? kTileBig : kTileSmall;
    const size_t smem = prefix_smem_bytes(gather, nl, Vp, p.hyps_per_cta, tile, math);
    CUtensorMap map;
    memset(&map, 0, sizeof(map));
    if (use_map) {
        const int rc = make_posterior_map(&map, x, Tmax, U, Vp, tile);
        if (rc != E2E_OK) return rc;
    }
    constexpr int TS = kTileSmall, TB = kTileBig;
    PrefixKernel kern;
    if (gather)
        kern = math == kMathLut ? prefix_score_kernel<true, kMathLut, 0, 0, false, TS>
             : math == kMathMufu ? prefix_score_kernel<true, kMathMufu, 0, 0, false, TS>
             : math == kMathLibm ? prefix_score_kernel<true, kMathLibm, 0, 0, false, TS>
             : math == kMathPoly ? prefix_score_kernel<true, kMathPoly, 0, 0, false, TS> : prefix_score_kernel<true, kMathPolyEstrin, 0, 0, false, TS>;
    else if (!use_map)
        kern = math == kMathLut ? prefix_score_kernel<false, kMathLut, 0, 0, false, TS>
             : math == kMathMufu ? prefix_score_kernel<false, kMathMufu, 0, 0, false, TS>
             : math == kMathLibm ? prefix_score_kernel<false, kMathLibm, 0, 0, false, TS>
             : math == kMathPoly ? prefix_score_kernel<false, kMathPoly, 0, 0, false, TS> : prefix_score_kernel<false, kMathPolyEstrin, 0, 0, false, TS>;
    else if (math == kMathLut) {
        if (fixed) kern = big_launch ? prefix_score_kernel<false, kMathLut, 32, 96, true, TB> : prefix_score_kernel<false, kMathLut, 32, 96, true, TS>;
        else kern = big_launch ? prefix_score_kernel<false, kMathLut, 0, 0, true, TB> : prefix_score_kernel<false, kMathLut, 0, 0, true, TS>;
    } else if (math == kMathPoly) {
        if (fixed) kern = big_launch ? prefix_score_kernel<false, kMathPoly, 32, 96, true, TB> : prefix_score_kernel<false, kMathPoly, 32, 96, true, TS>;
        else kern = big_launch ? prefix_score_kernel<false, kMathPoly, 0, 0, true, TB> : prefix_score_kernel<false, kMathPoly, 0, 0, true, TS>;
    } else if (math == kMathPolyEstrin) {
        if (fixed) kern = big_launch ? prefix_score_kernel<false, kMathPolyEstrin, 32, 96, true, TB> : prefix_score_kernel<false, kMathPolyEstrin, 32, 96, true, TS>;
        else kern = big_launch ? prefix_score_kernel<false, kMathPolyEstrin, 0, 0, true, TB> : prefix_score_kernel<false, kMathPolyEstrin, 0, 0, true, TS>;
    } else
        kern = math == kMathMufu ? prefix_score_kernel<false, kMathMufu, 0, 0, true, TS> : prefix_score_kernel<false, kMathLibm, 0, 0, true, TS>;
    if (smem > 48 * 1024) {
        if (smem > 200 * 1024) return set_error(E2E_ERR_UNSUPPORTED, "e2e_ctc_prefix_score: %zu bytes of shared memory needed", smem);
        cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return set_error(E2E_ERR_LAUNCH, "cudaFuncSetAttribute: %s", cudaGetErrorString(e));
    }
    kern<<<(unsigned)grid, nl, smem, static_cast<cudaStream_t>(stream)>>>(p, map);
    count_launch();
    return check_launch("e2e_ctc_prefix_score");
}
