// One-token LSTM step helpers for the batched RNNLM / speller step (SURVEY.md §8f row f-2).
// The recurrent GEMMs stay library calls (bf16 tensor-core GEMMs on a 3-way split of the fp32
// operands, see stepper.py); these two kernels replace the ~25 element-wise launches per layer
// that used to surround them and remove the per-step state permutation:
//   lstm_split_rows_kernel : gathers fp32 rows through the parents' row index and writes their
//                            exact 3-piece bf16 split straight into the GEMM's A operand
//   lstm_cell_kernel       : gates (+ bias, + layer-0 input table) -> (c', h') in fp32 with the
//                            reference's operation order (nn.LSTM cell: src/lm.py:31, src/asr.py:262),
//                            reading c through the parents' row index, and writing the bf16 split
//                            of h' into the NEXT layer's A operand
//   gru_cell_kernel        : the same for an nn.GRU layer (no c state): gates in four blocks [r | z | n_x | n_h]
//                            (+ bias, + table) -> h' in ATen's GRU cell order, h read through the parents' row index
// All are pure HBM streams: one pass over their inputs and outputs, 16-byte accesses.
//
// Two operand formats (template parameter kPieces):
//   3 : x == a1 + a2 + a3, bf16 pieces (24 mantissa bits, any magnitude) — six partial GEMM products
//   2 : s*x ~= a1 + a2, fp16 pieces of the value scaled by a power of two s (22 mantissa bits; for
//       operands of known range such as LSTM hidden states, |h| < 1) — three partial products, half
//       the tensor-core work; the GEMM result carries the factor s_a*s_w, which the cell kernel
//       removes (exactly: a power of two) before the bias is added
#include "common.cuh"
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cmath>

namespace e2e {

// x == a1 + a2 + a3 exactly (barring underflow): a1 = bf16(x), a2 = bf16(x - a1), a3 = bf16(x - a1 - a2)
__device__ __forceinline__ void split3(float x, __nv_bfloat16 &a1, __nv_bfloat16 &a2, __nv_bfloat16 &a3)
{
    a1 = __float2bfloat16_rn(x);
    const float r1 = __fsub_rn(x, __bfloat162float(a1));
    a2 = __float2bfloat16_rn(r1);
    a3 = __float2bfloat16_rn(__fsub_rn(r1, __bfloat162float(a2)));
}

struct alignas(8) Bf16x4 { __nv_bfloat16 v[4]; };

// s*x == a1 + a2 up to 2^-22 |s*x|: a1 = fp16(s*x), a2 = fp16(s*x - a1); s a power of two keeps s*x exact
__device__ __forceinline__ void split2(float x, float s, __half &a1, __half &a2)
{
    const float xs = __fmul_rn(x, s);
    a1 = __float2half_rn(xs);
    a2 = __float2half_rn(__fsub_rn(xs, __half2float(a1)));
}

struct alignas(8) F16x4 { __half v[4]; };

// the kPieces pieces of four consecutive values -> d[c], d[K + c], (d[2K + c]); d counts 16-bit elements
template <int kPieces>
__device__ __forceinline__ void store_pieces4(const float (&x)[4], float scale, unsigned short *d, int K)
{
    if (kPieces == 3) {
        Bf16x4 p0, p1, p2;
#pragma unroll
        for (int i = 0; i < 4; ++i) split3(x[i], p0.v[i], p1.v[i], p2.v[i]);
        *reinterpret_cast<Bf16x4 *>(d) = p0;
        *reinterpret_cast<Bf16x4 *>(d + K) = p1;
        *reinterpret_cast<Bf16x4 *>(d + 2 * K) = p2;
    } else {
        F16x4 p0, p1;
#pragma unroll
        for (int i = 0; i < 4; ++i) split2(x[i], scale, p0.v[i], p1.v[i]);
        *reinterpret_cast<F16x4 *>(d) = p0;
        *reinterpret_cast<F16x4 *>(d + K) = p1;
    }
}

template <int kPieces>
__device__ __forceinline__ void store_pieces1(float x, float scale, unsigned short *d, int K)
{
    if (kPieces == 3) {
        __nv_bfloat16 a1, a2, a3;
        split3(x, a1, a2, a3);
        d[0] = __bfloat16_as_ushort(a1); d[K] = __bfloat16_as_ushort(a2); d[2 * K] = __bfloat16_as_ushort(a3);
    } else {
        __half a1, a2;
        split2(x, scale, a1, a2);
        d[0] = __half_as_ushort(a1); d[K] = __half_as_ushort(a2);
    }
}

// dst[r][p*K + off + c] = piece_p(src[row(r)][c]),  p < kPieces,  c < w;  row(r) = idx ? idx[r] : r
template <bool kVec, int kPieces>
__global__ void __launch_bounds__(256)
lstm_split_rows_kernel(const float *__restrict__ src, long long src_pitch, const long long *__restrict__ idx, int n, int w,
                       unsigned short *__restrict__ dst, long long dst_pitch, int K, int off, float scale)
{
    const int r = blockIdx.y;
    const long long row = idx ? idx[r] : r;
    const float *s = src + row * src_pitch;
    unsigned short *d = dst + (long long)r * dst_pitch + off;
    if (kVec) {
        for (int c = (blockIdx.x * blockDim.x + threadIdx.x) * 4; c < w; c += gridDim.x * blockDim.x * 4) {
            const float4 v = __ldg(reinterpret_cast<const float4 *>(s + c));
            const float x[4] = {v.x, v.y, v.z, v.w};
            store_pieces4<kPieces>(x, scale, d + c, K);
        }
    } else {
        for (int c = blockIdx.x * blockDim.x + threadIdx.x; c < w; c += gridDim.x * blockDim.x)
            store_pieces1<kPieces>(__ldg(s + c), scale, d + c, K);
    }
}

// the same for up to kMaxSplitSrc sources in one launch (blockIdx.z = source): all layers of an LSTM stack at once
constexpr int kMaxSplitSrc = 8;
struct SplitMulti {
    const float *src[kMaxSplitSrc]; long long src_pitch[kMaxSplitSrc]; int w[kMaxSplitSrc];
    unsigned short *dst[kMaxSplitSrc]; long long dst_pitch[kMaxSplitSrc]; int K[kMaxSplitSrc], off[kMaxSplitSrc];
    const long long *idx; int n; float scale;
};

template <int kPieces>
__global__ void __launch_bounds__(256)
lstm_split_rows_multi_kernel(const SplitMulti p)
{
    const int z = blockIdx.z, r = blockIdx.y;
    const long long row = p.idx ? p.idx[r] : r;
    const float *s = p.src[z] + row * p.src_pitch[z];
    unsigned short *d = p.dst[z] + (long long)r * p.dst_pitch[z] + p.off[z];
    const int w = p.w[z], K = p.K[z];
    for (int c = (blockIdx.x * blockDim.x + threadIdx.x) * 4; c < w; c += gridDim.x * blockDim.x * 4) {
        const float4 v = __ldg(reinterpret_cast<const float4 *>(s + c));
        const float x[4] = {v.x, v.y, v.z, v.w};
        store_pieces4<kPieces>(x, p.scale, d + c, K);
    }
}

__device__ __forceinline__ float sigmoid_f32(float x) { return __fdiv_rn(1.0f, __fadd_rn(1.0f, expf(-x))); }

struct CellParams {
    const float *gates; long long gates_pitch; const float *bias; const float *table; const long long *tok;
    const float *c_prev; const long long *idx; int n, D;
    float *c_new, *h_new; unsigned short *a_next; long long a_pitch; int K_next, off_next;
    float gate_scale, next_scale;        // kPieces == 2: gates *= gate_scale (undoes s_a*s_w); h' is split as next_scale*h'
};

__device__ __forceinline__ void lstm_unit(const float (&g)[4], const float (&b)[4], const float *tb, float c, float &c2, float &h2)
{
    float z[4];
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        z[q] = __fadd_rn(g[q], b[q]);                       // y + (b_ih + b_hh)
        if (tb) z[q] = __fadd_rn(tb[q], z[q]);              // + layer-0 input projection
    }
    c2 = __fadd_rn(__fmul_rn(sigmoid_f32(z[1]), c), __fmul_rn(sigmoid_f32(z[0]), tanhf(z[2])));
    h2 = __fmul_rn(sigmoid_f32(z[3]), tanhf(c2));
}

// one thread per (row, kW consecutive hidden units); gate order i, f, g, o (torch.nn.LSTM)
template <int kW, int kPieces>
__global__ void __launch_bounds__(256)
lstm_cell_kernel(const CellParams p)
{
    const int r = blockIdx.y;
    const float *g = p.gates + (long long)r * p.gates_pitch;
    const float *tb = p.table ? p.table + p.tok[r] * (long long)(4 * p.D) : nullptr;
    const long long prow = p.idx ? p.idx[r] : r;
    const float *cp = p.c_prev + prow * p.D;
    for (int d = (blockIdx.x * blockDim.x + threadIdx.x) * kW; d < p.D; d += gridDim.x * blockDim.x * kW) {
        float gv[4][kW], bv[4][kW], tv[4][kW], cv[kW];
        if (kW == 4) {
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const float4 a = __ldg(reinterpret_cast<const float4 *>(g + q * p.D + d));
                const float4 b = __ldg(reinterpret_cast<const float4 *>(p.bias + q * p.D + d));
                gv[q][0] = a.x; gv[q][1] = a.y; gv[q][2] = a.z; gv[q][3] = a.w;
                bv[q][0] = b.x; bv[q][1] = b.y; bv[q][2] = b.z; bv[q][3] = b.w;
                if (tb) {
                    const float4 t = __ldg(reinterpret_cast<const float4 *>(tb + q * p.D + d));
                    tv[q][0] = t.x; tv[q][1] = t.y; tv[q][2] = t.z; tv[q][3] = t.w;
                }
            }
            const float4 c = __ldg(reinterpret_cast<const float4 *>(cp + d));
            cv[0] = c.x; cv[1] = c.y; cv[2] = c.z; cv[3] = c.w;
        } else {
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                gv[q][0] = __ldg(g + q * p.D + d);
                bv[q][0] = __ldg(p.bias + q * p.D + d);
                if (tb) tv[q][0] = __ldg(tb + q * p.D + d);
            }
            cv[0] = __ldg(cp + d);
        }
        float c2[kW], h2[kW];
#pragma unroll
        for (int i = 0; i < kW; ++i) {
            if (kPieces == 2) {
#pragma unroll
                for (int q = 0; q < 4; ++q) gv[q][i] = __fmul_rn(gv[q][i], p.gate_scale);
            }
            const float gi[4] = {gv[0][i], gv[1][i], gv[2][i], gv[3][i]};
            const float bi[4] = {bv[0][i], bv[1][i], bv[2][i], bv[3][i]};
            const float ti[4] = {tb ? tv[0][i] : 0.0f, tb ? tv[1][i] : 0.0f, tb ? tv[2][i] : 0.0f, tb ? tv[3][i] : 0.0f};
            lstm_unit(gi, bi, tb ? ti : nullptr, cv[i], c2[i], h2[i]);
        }
        float *co = p.c_new + (long long)r * p.D + d, *ho = p.h_new + (long long)r * p.D + d;
        if (kW == 4) {
            *reinterpret_cast<float4 *>(co) = make_float4(c2[0], c2[1], c2[2], c2[3]);
            *reinterpret_cast<float4 *>(ho) = make_float4(h2[0], h2[1], h2[2], h2[3]);
        } else {
            co[0] = c2[0]; ho[0] = h2[0];
        }
        if (p.a_next) {
            unsigned short *o = p.a_next + (long long)r * p.a_pitch + p.off_next + d;
            if constexpr (kW == 4) store_pieces4<kPieces>(h2, p.next_scale, o, p.K_next);
            else store_pieces1<kPieces>(h2[0], p.next_scale, o, p.K_next);
        }
    }
}

// GRU step with the gates in four D-wide blocks [r | z | n_x | n_h] (one GEMM chain per layer, like the LSTM: the
// weight rows of n_x carry only W_in, those of n_h only W_hn, so the two n-gate products stay apart)
struct GruCellParams {
    const float *gates; long long gates_pitch; const float *bias; const float *table; const long long *tok;
    const float *h_prev; const long long *idx; int n, D;
    float *h_new; unsigned short *a_next; long long a_pitch; int K_next, off_next;
    float gate_scale, next_scale;        // kPieces == 2: as in CellParams
};

// ATen's GRU cell order (nn.GRU on the CPU): n = tanh(z_nx + r * z_nh), h' = (h - n) * u + n, every op rounded
__device__ __forceinline__ float gru_unit(const float (&g)[4], const float (&b)[4], const float *tb, float h)
{
    float z[4];
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        z[q] = __fadd_rn(g[q], b[q]);
        if (tb) z[q] = __fadd_rn(tb[q], z[q]);              // + layer-0 input projection
    }
    const float r = sigmoid_f32(z[0]), u = sigmoid_f32(z[1]);
    const float nn = tanhf(__fadd_rn(z[2], __fmul_rn(r, z[3])));
    return __fadd_rn(__fmul_rn(__fsub_rn(h, nn), u), nn);
}

// one thread per (row, kW consecutive hidden units); the sibling of lstm_cell_kernel without the c state
template <int kW, int kPieces>
__global__ void __launch_bounds__(256)
gru_cell_kernel(const GruCellParams p)
{
    const int r = blockIdx.y;
    const float *g = p.gates + (long long)r * p.gates_pitch;
    const float *tb = p.table ? p.table + p.tok[r] * (long long)(4 * p.D) : nullptr;
    const long long prow = p.idx ? p.idx[r] : r;
    const float *hp = p.h_prev + prow * p.D;
    for (int d = (blockIdx.x * blockDim.x + threadIdx.x) * kW; d < p.D; d += gridDim.x * blockDim.x * kW) {
        float gv[4][kW], bv[4][kW], tv[4][kW], hv[kW];
        if (kW == 4) {
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const float4 a = __ldg(reinterpret_cast<const float4 *>(g + q * p.D + d));
                const float4 b = __ldg(reinterpret_cast<const float4 *>(p.bias + q * p.D + d));
                gv[q][0] = a.x; gv[q][1] = a.y; gv[q][2] = a.z; gv[q][3] = a.w;
                bv[q][0] = b.x; bv[q][1] = b.y; bv[q][2] = b.z; bv[q][3] = b.w;
                if (tb) {
                    const float4 t = __ldg(reinterpret_cast<const float4 *>(tb + q * p.D + d));
                    tv[q][0] = t.x; tv[q][1] = t.y; tv[q][2] = t.z; tv[q][3] = t.w;
                }
            }
            const float4 h = __ldg(reinterpret_cast<const float4 *>(hp + d));
            hv[0] = h.x; hv[1] = h.y; hv[2] = h.z; hv[3] = h.w;
        } else {
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                gv[q][0] = __ldg(g + q * p.D + d);
                bv[q][0] = __ldg(p.bias + q * p.D + d);
                if (tb) tv[q][0] = __ldg(tb + q * p.D + d);
            }
            hv[0] = __ldg(hp + d);
        }
        float h2[kW];
#pragma unroll
        for (int i = 0; i < kW; ++i) {
            if (kPieces == 2) {
#pragma unroll
                for (int q = 0; q < 4; ++q) gv[q][i] = __fmul_rn(gv[q][i], p.gate_scale);
            }
            const float gi[4] = {gv[0][i], gv[1][i], gv[2][i], gv[3][i]};
            const float bi[4] = {bv[0][i], bv[1][i], bv[2][i], bv[3][i]};
            const float ti[4] = {tb ? tv[0][i] : 0.0f, tb ? tv[1][i] : 0.0f, tb ? tv[2][i] : 0.0f, tb ? tv[3][i] : 0.0f};
            h2[i] = gru_unit(gi, bi, tb ? ti : nullptr, hv[i]);
        }
        float *ho = p.h_new + (long long)r * p.D + d;
        if (kW == 4) *reinterpret_cast<float4 *>(ho) = make_float4(h2[0], h2[1], h2[2], h2[3]);
        else ho[0] = h2[0];
        if (p.a_next) {
            unsigned short *o = p.a_next + (long long)r * p.a_pitch + p.off_next + d;
            if constexpr (kW == 4) store_pieces4<kPieces>(h2, p.next_scale, o, p.K_next);
            else store_pieces1<kPieces>(h2[0], p.next_scale, o, p.K_next);
        }
    }
}

}  // namespace e2e

namespace {

using namespace e2e;

// a power of two in a range where s*x and the fp32 GEMM accumulators cannot overflow
bool valid_scale(float s)
{
    int e = 0;
    return s > 0.0f && std::frexp(s, &e) == 0.5f && e >= -60 && e <= 60;
}

int split_rows_impl(const char *name, int pieces, float scale, const float *src, long long src_pitch, const long long *row_idx,
                    int n, int w, void *dst16, long long dst_pitch, int K, int off, void *stream)
{
    if (!src || !dst16) return set_error(E2E_ERR_ARG, "%s: null pointer", name);
    if (n <= 0 || w <= 0 || K <= 0 || off < 0 || off + w > K || dst_pitch < (long long)pieces * K || src_pitch < w)
        return set_error(E2E_ERR_ARG, "%s: bad size", name);
    if (pieces == 2 && !valid_scale(scale)) return set_error(E2E_ERR_ARG, "%s: scale must be a power of two", name);
    if (n > 65535 * 16) return set_error(E2E_ERR_UNSUPPORTED, "%s: too many rows", name);
    const bool vec = (w % 4 == 0) && (src_pitch % 4 == 0) && (dst_pitch % 4 == 0) && (K % 4 == 0) && (off % 4 == 0) &&
                     !(reinterpret_cast<uintptr_t>(src) & 15) && !(reinterpret_cast<uintptr_t>(dst16) & 7);
    const int per_thread = vec ? 4 : 1;
    const int bx = (w + 256 * per_thread - 1) / (256 * per_thread);
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    unsigned short *dst = static_cast<unsigned short *>(dst16);
    for (int r0 = 0; r0 < n; r0 += 65535) {          // gridDim.y limit
        const int rows = n - r0 < 65535 ? n - r0 : 65535;
        const dim3 grid(bx, rows);
        const float *s0 = src + (row_idx ? 0 : (long long)r0 * src_pitch);
        const long long *i0 = row_idx ? row_idx + r0 : nullptr;
        unsigned short *d0 = dst + (long long)r0 * dst_pitch;
        if (pieces == 3) {
            if (vec) lstm_split_rows_kernel<true, 3><<<grid, 256, 0, st>>>(s0, src_pitch, i0, rows, w, d0, dst_pitch, K, off, 1.0f);
            else lstm_split_rows_kernel<false, 3><<<grid, 256, 0, st>>>(s0, src_pitch, i0, rows, w, d0, dst_pitch, K, off, 1.0f);
        } else {
            if (vec) lstm_split_rows_kernel<true, 2><<<grid, 256, 0, st>>>(s0, src_pitch, i0, rows, w, d0, dst_pitch, K, off, scale);
            else lstm_split_rows_kernel<false, 2><<<grid, 256, 0, st>>>(s0, src_pitch, i0, rows, w, d0, dst_pitch, K, off, scale);
        }
        count_launch();
    }
    return check_launch(name);
}

int split_rows_multi_impl(const char *name, int pieces, float scale, int n_src, const float *const *srcs, const long long *src_pitches,
                          const int *widths, void *const *dsts16, const long long *dst_pitches, const int *Ks, const int *offs,
                          const long long *row_idx, int n, void *stream)
{
    if (!srcs || !src_pitches || !widths || !dsts16 || !dst_pitches || !Ks || !offs) return set_error(E2E_ERR_ARG, "%s: null pointer", name);
    if (n_src <= 0 || n_src > kMaxSplitSrc || n <= 0) return set_error(E2E_ERR_ARG, "%s: bad size", name);
    if (pieces == 2 && !valid_scale(scale)) return set_error(E2E_ERR_ARG, "%s: scale must be a power of two", name);
    SplitMulti p;
    p.scale = scale;
    int wmax = 0;
    for (int i = 0; i < n_src; ++i) {
        if (!srcs[i] || !dsts16[i]) return set_error(E2E_ERR_ARG, "%s: null pointer", name);
        const bool vec = (widths[i] % 4 == 0) && (src_pitches[i] % 4 == 0) && (dst_pitches[i] % 4 == 0) && (Ks[i] % 4 == 0) &&
                         (offs[i] % 4 == 0) && !(reinterpret_cast<uintptr_t>(srcs[i]) & 15) && !(reinterpret_cast<uintptr_t>(dsts16[i]) & 7);
        if (!vec) return set_error(E2E_ERR_UNSUPPORTED, "%s: source %d is not 16-byte vectorisable", name, i);
        if (widths[i] <= 0 || offs[i] < 0 || offs[i] + widths[i] > Ks[i] || dst_pitches[i] < (long long)pieces * Ks[i] || src_pitches[i] < widths[i])
            return set_error(E2E_ERR_ARG, "%s: bad geometry of source %d", name, i);
        p.src[i] = srcs[i]; p.src_pitch[i] = src_pitches[i]; p.w[i] = widths[i];
        p.dst[i] = static_cast<unsigned short *>(dsts16[i]); p.dst_pitch[i] = dst_pitches[i]; p.K[i] = Ks[i]; p.off[i] = offs[i];
        wmax = widths[i] > wmax ? widths[i] : wmax;
    }
    const int bx = (wmax + 1023) / 1024;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    for (int r0 = 0; r0 < n; r0 += 65535) {
        const int rows = n - r0 < 65535 ? n - r0 : 65535;
        SplitMulti q = p;
        q.n = rows;
        q.idx = row_idx ? row_idx + r0 : nullptr;
        for (int i = 0; i < n_src; ++i) {
            if (!row_idx) q.src[i] = p.src[i] + (long long)r0 * p.src_pitch[i];
            q.dst[i] = p.dst[i] + (long long)r0 * p.dst_pitch[i];
        }
        if (pieces == 3) lstm_split_rows_multi_kernel<3><<<dim3(bx, rows, n_src), 256, 0, st>>>(q);
        else lstm_split_rows_multi_kernel<2><<<dim3(bx, rows, n_src), 256, 0, st>>>(q);
        count_launch();
    }
    return check_launch(name);
}

// the LSTM cell (c_new given) or the GRU cell (c_new == nullptr, s_prev = h_prev) over n rows
int cell_impl(const char *name, bool gru, int pieces, float gate_scale, float next_scale, const float *gates, long long gates_pitch,
              const float *bias, const float *table, const long long *tok, const float *s_prev, const long long *row_idx, int n, int D,
              float *c_new, float *h_new, void *a_next16, long long a_pitch, int K_next, int off_next, void *stream)
{
    if (!gates || !bias || !s_prev || (!gru && !c_new) || !h_new || (table && !tok)) return set_error(E2E_ERR_ARG, "%s: null pointer", name);
    if (n <= 0 || D <= 0 || gates_pitch < 4LL * D) return set_error(E2E_ERR_ARG, "%s: bad size", name);
    if (a_next16 && (K_next <= 0 || off_next < 0 || off_next + D > K_next || a_pitch < (long long)pieces * K_next))
        return set_error(E2E_ERR_ARG, "%s: bad next-layer operand geometry", name);
    if (pieces == 2 && (!valid_scale(gate_scale) || (a_next16 && !valid_scale(next_scale))))
        return set_error(E2E_ERR_ARG, "%s: scales must be powers of two", name);
    CellParams p;
    p.gates = gates; p.gates_pitch = gates_pitch; p.bias = bias; p.table = table; p.tok = tok;
    p.c_prev = s_prev; p.idx = row_idx; p.D = D; p.a_pitch = a_pitch; p.K_next = K_next; p.off_next = off_next;
    p.gate_scale = gate_scale; p.next_scale = next_scale;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const bool vec = (D % 4 == 0) && (gates_pitch % 4 == 0) && !(reinterpret_cast<uintptr_t>(gates) & 15) &&
                     !(reinterpret_cast<uintptr_t>(bias) & 15) && !(reinterpret_cast<uintptr_t>(table) & 15) &&
                     !(reinterpret_cast<uintptr_t>(s_prev) & 15) && !(reinterpret_cast<uintptr_t>(c_new) & 15) &&
                     !(reinterpret_cast<uintptr_t>(h_new) & 15) &&
                     (!a_next16 || ((a_pitch % 4 == 0) && (K_next % 4 == 0) && (off_next % 4 == 0) && !(reinterpret_cast<uintptr_t>(a_next16) & 7)));
    const int per_thread = vec ? 4 : 1;
    const int threads = D / per_thread >= 256 ? 256 : ((D / per_thread + 31) / 32 * 32);
    const int bx = (D + threads * per_thread - 1) / (threads * per_thread);
    for (int r0 = 0; r0 < n; r0 += 65535) {
        const int rows = n - r0 < 65535 ? n - r0 : 65535;
        p.n = rows;
        p.gates = gates + (long long)r0 * gates_pitch;
        p.tok = tok ? tok + r0 : nullptr;
        p.idx = row_idx ? row_idx + r0 : nullptr;
        p.c_prev = row_idx ? s_prev : s_prev + (long long)r0 * D;
        p.c_new = gru ? nullptr : c_new + (long long)r0 * D;
        p.h_new = h_new + (long long)r0 * D;
        p.a_next = a_next16 ? static_cast<unsigned short *>(a_next16) + (long long)r0 * a_pitch : nullptr;
        const dim3 grid(bx, rows);
        if (gru) {
            const GruCellParams q{p.gates, p.gates_pitch, p.bias, p.table, p.tok, p.c_prev, p.idx, p.n, p.D,
                                  p.h_new, p.a_next, p.a_pitch, p.K_next, p.off_next, p.gate_scale, p.next_scale};
            if (pieces == 3) {
                if (vec) gru_cell_kernel<4, 3><<<grid, threads, 0, st>>>(q);
                else gru_cell_kernel<1, 3><<<grid, threads, 0, st>>>(q);
            } else {
                if (vec) gru_cell_kernel<4, 2><<<grid, threads, 0, st>>>(q);
                else gru_cell_kernel<1, 2><<<grid, threads, 0, st>>>(q);
            }
        } else if (pieces == 3) {
            if (vec) lstm_cell_kernel<4, 3><<<grid, threads, 0, st>>>(p);
            else lstm_cell_kernel<1, 3><<<grid, threads, 0, st>>>(p);
        } else {
            if (vec) lstm_cell_kernel<4, 2><<<grid, threads, 0, st>>>(p);
            else lstm_cell_kernel<1, 2><<<grid, threads, 0, st>>>(p);
        }
        count_launch();
    }
    return check_launch(name);
}

}  // namespace

extern "C" int e2e_lstm_split_rows(const float *src, long long src_pitch, const long long *row_idx, int n, int w,
                                   void *dst_bf16, long long dst_pitch, int K, int off, void *stream)
{
    return split_rows_impl("e2e_lstm_split_rows", 3, 1.0f, src, src_pitch, row_idx, n, w, dst_bf16, dst_pitch, K, off, stream);
}

extern "C" int e2e_lstm_split_rows_f16x2(const float *src, long long src_pitch, const long long *row_idx, int n, int w,
                                         void *dst_f16, long long dst_pitch, int K, int off, float scale, void *stream)
{
    return split_rows_impl("e2e_lstm_split_rows_f16x2", 2, scale, src, src_pitch, row_idx, n, w, dst_f16, dst_pitch, K, off, stream);
}

extern "C" int e2e_lstm_split_rows_multi(int n_src, const float *const *srcs, const long long *src_pitches, const int *widths,
                                         void *const *dsts_bf16, const long long *dst_pitches, const int *Ks, const int *offs,
                                         const long long *row_idx, int n, void *stream)
{
    return split_rows_multi_impl("e2e_lstm_split_rows_multi", 3, 1.0f, n_src, srcs, src_pitches, widths, dsts_bf16, dst_pitches,
                                 Ks, offs, row_idx, n, stream);
}

extern "C" int e2e_lstm_split_rows_multi_f16x2(int n_src, const float *const *srcs, const long long *src_pitches, const int *widths,
                                               void *const *dsts_f16, const long long *dst_pitches, const int *Ks, const int *offs,
                                               const long long *row_idx, int n, float scale, void *stream)
{
    return split_rows_multi_impl("e2e_lstm_split_rows_multi_f16x2", 2, scale, n_src, srcs, src_pitches, widths, dsts_f16,
                                 dst_pitches, Ks, offs, row_idx, n, stream);
}

extern "C" int e2e_lstm_cell(const float *gates, long long gates_pitch, const float *bias, const float *table, const long long *tok,
                             const float *c_prev, const long long *row_idx, int n, int D,
                             float *c_new, float *h_new, void *a_next_bf16, long long a_pitch, int K_next, int off_next,
                             void *stream)
{
    return cell_impl("e2e_lstm_cell", false, 3, 1.0f, 1.0f, gates, gates_pitch, bias, table, tok, c_prev, row_idx, n, D, c_new, h_new,
                     a_next_bf16, a_pitch, K_next, off_next, stream);
}

extern "C" int e2e_lstm_cell_f16x2(const float *gates, long long gates_pitch, float gate_scale, const float *bias, const float *table,
                                   const long long *tok, const float *c_prev, const long long *row_idx, int n, int D,
                                   float *c_new, float *h_new, void *a_next_f16, long long a_pitch, int K_next, int off_next,
                                   float next_scale, void *stream)
{
    return cell_impl("e2e_lstm_cell_f16x2", false, 2, gate_scale, next_scale, gates, gates_pitch, bias, table, tok, c_prev, row_idx, n, D,
                     c_new, h_new, a_next_f16, a_pitch, K_next, off_next, stream);
}

extern "C" int e2e_gru_cell(const float *gates, long long gates_pitch, const float *bias, const float *table, const long long *tok,
                            const float *h_prev, const long long *row_idx, int n, int D,
                            float *h_new, void *a_next_bf16, long long a_pitch, int K_next, int off_next, void *stream)
{
    return cell_impl("e2e_gru_cell", true, 3, 1.0f, 1.0f, gates, gates_pitch, bias, table, tok, h_prev, row_idx, n, D, nullptr, h_new,
                     a_next_bf16, a_pitch, K_next, off_next, stream);
}

extern "C" int e2e_gru_cell_f16x2(const float *gates, long long gates_pitch, float gate_scale, const float *bias, const float *table,
                                  const long long *tok, const float *h_prev, const long long *row_idx, int n, int D,
                                  float *h_new, void *a_next_f16, long long a_pitch, int K_next, int off_next, float next_scale,
                                  void *stream)
{
    return cell_impl("e2e_gru_cell_f16x2", true, 2, gate_scale, next_scale, gates, gates_pitch, bias, table, tok, h_prev, row_idx, n, D,
                     nullptr, h_new, a_next_f16, a_pitch, K_next, off_next, stream);
}
