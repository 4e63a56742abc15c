// Whole-sequence (B)LSTM recurrence of the encoder (SURVEY.md §8f row f-4; RNNLayer, src/module.py:1003-1081:
// nn.LSTM over the utterance, one direction per call of this kernel's grid row).
// cuDNN runs this as two tiny launches per time step per direction (70 k launches per pass over the
// bench workload, each latency bound).  Here the input projections of ALL frames are one tensor-core
// GEMM (library, split-bf16, see stepper.SplitLinear) and the recurrence is one persistent launch per
// layer: a CTA owns a group of R utterances x one direction and walks their frames; thread u owns
// hidden unit u — its four gate columns for the R utterances live in registers (4R accumulators), the
// recurrent weights stream from L2 in a [k][unit][gate] layout (one coalesced 16-byte load per unit per k), the previous
// hidden states are shared-memory broadcasts ([k][R], one LDS.128 per four utterances), and the cell
// update happens in the same thread with no exchange but the one __syncthreads per time step that
// publishes h.  Utterances are PACKED (frame_off[n] + t): no padding is computed or stored, the
// backward direction simply walks t = len-1 .. 0, and long utterances are put in smaller groups so
// that the longest sequence does not set the run time.  Bound: fp32 FMA issue (R x 4H x H per step)
// against the L2 stream of W_hh (4H x H x 4 bytes per step).
//
// The GRU form (gru_seq_kernel, nn.GRU) is the same body with three gate blocks [r | z | n] per gates row: W_hh is laid
// out [k][unit][4] = (W_hr, W_hz, W_hn, 0), so the recurrence keeps one 16-byte load per unit per k and runs 3R
// accumulators (r, z and the n_h product, which starts at b_hn); the input half of the n gate is held apart (one value
// per utterance) and the cell is ATen's order n = tanh(n_x + r * n_h), h' = (h - n) * u + n.
#include "common.cuh"

namespace e2e {

constexpr int kSeqMaxThreads = 384;     // hidden sizes up to 384 (the register file then allows ~170 registers per thread)

struct SeqDir {
    const float *bias;      // [4H] b_ih + b_hh (may be null); GRU: [b_ir + b_hr | b_iz + b_hz | b_in | b_hn]
    const float *w_t;       // [H][H][4]: w_t[k][u][g] = w_hh[g*H + u][k]  (one 16-byte load per unit per k; GRU: g < 3, lane 3 zero)
    int gate_off;           // column of this direction's 4H (GRU: 3H) block inside a gates row
    int out_off;            // column of this direction's H block inside an output row
    int reverse;            // 0: t = 0..len-1, 1: t = len-1..0
};

struct SeqParams {
    const float *gates; long long gates_pitch;      // [frames][pitch]: x_t W_ih^T of every packed frame
    float *out; long long out_pitch;                // [frames][pitch]
    const int *frame_off, *lens;                    // [N] first packed frame / frame count of utterance n
    const int *group_first, *group_rows;            // [n_groups] rows first .. first+rows-1 (rows in {4, 8, 16})
    int N, H, n_groups;
    SeqDir dir[2];
};

__device__ __forceinline__ float seq_sigmoid(float x) { return __fdiv_rn(1.0f, __fadd_rn(1.0f, expf(-x))); }

template <bool kGru, int R>
__device__ __forceinline__ void lstm_seq_body(const SeqParams &p, const SeqDir &d, int first, int rows, float *smem)
{
    const int H = p.H, u = threadIdx.x;
    const bool unit = u < H;
    float *hs = smem;                                  // [2][H][R]
    int *s_len = reinterpret_cast<int *>(smem + 2 * H * R);
    int *s_off = s_len + R;
    if (u < R) {
        const bool ok = u < rows;
        s_len[u] = ok ? p.lens[first + u] : 0;
        s_off[u] = ok ? p.frame_off[first + u] : 0;
    }
    for (int i = u; i < 2 * H * R; i += blockDim.x) hs[i] = 0.0f;
    __syncthreads();
    int max_len = 0;
#pragma unroll
    for (int r = 0; r < R; ++r) max_len = max(max_len, s_len[r]);
    float c[R];
#pragma unroll
    for (int r = 0; r < R; ++r) c[r] = 0.0f;
    float b[4] = {0.0f, 0.0f, 0.0f, 0.0f};
    if (unit && d.bias)
#pragma unroll
        for (int g = 0; g < 4; ++g) b[g] = __ldg(d.bias + g * H + u);
    const float4 *wu = reinterpret_cast<const float4 *>(d.w_t) + u;

    for (int s = 0; s < max_len; ++s) {
        const float *hc = hs + (size_t)(s & 1) * H * R;
        float *hn = hs + (size_t)((s + 1) & 1) * H * R;
        constexpr int kAcc = kGru ? 3 : 4;                 // GRU: r, z, n_h; the input part of n waits in nx
        float acc[kAcc][R], nx[kGru ? R : 1];
        int row[R];
#pragma unroll
        for (int r = 0; r < R; ++r) {
            const int len = s_len[r];
            const bool on = s < len;
            row[r] = on ? s_off[r] + (d.reverse ? len - 1 - s : s) : -1;
            if constexpr (kGru) {
                const float *gr = p.gates + (long long)row[r] * p.gates_pitch + d.gate_off + u;
                const bool ld = on && unit;
                acc[0][r] = ld ? __fadd_rn(__ldg(gr), b[0]) : 0.0f;
                acc[1][r] = ld ? __fadd_rn(__ldg(gr + H), b[1]) : 0.0f;
                nx[r] = ld ? __fadd_rn(__ldg(gr + 2 * H), b[2]) : 0.0f;
                acc[2][r] = b[3];                            // b_hn + W_hn h
            } else {
#pragma unroll
                for (int g = 0; g < 4; ++g)
                    acc[g][r] = (on && unit) ? __fadd_rn(__ldg(p.gates + (long long)row[r] * p.gates_pitch + d.gate_off + g * H + u), b[g]) : 0.0f;
            }
        }
        if (unit) {
#pragma unroll 4
            for (int k = 0; k < H; ++k) {
                const float4 w4 = __ldg(wu + (size_t)k * H);
                const float w[4] = {w4.x, w4.y, w4.z, w4.w};
                float hv[R];
#pragma unroll
                for (int q = 0; q < R / 4; ++q) {
                    const float4 h4 = *reinterpret_cast<const float4 *>(hc + k * R + 4 * q);
                    hv[4 * q] = h4.x; hv[4 * q + 1] = h4.y; hv[4 * q + 2] = h4.z; hv[4 * q + 3] = h4.w;
                }
#pragma unroll
                for (int g = 0; g < kAcc; ++g)
#pragma unroll
                    for (int r = 0; r < R; ++r) acc[g][r] = fmaf(w[g], hv[r], acc[g][r]);
            }
            float hout[R];
#pragma unroll
            for (int r = 0; r < R; ++r) {
                if (kGru && row[r] >= 0) {                           // gate order r, z, n (torch.nn.GRU)
                    const float rg = seq_sigmoid(acc[0][r]), ug = seq_sigmoid(acc[1][r]);
                    const float ng = tanhf(__fadd_rn(nx[r], __fmul_rn(rg, acc[2][r])));
                    const float h2 = __fadd_rn(__fmul_rn(__fsub_rn(hc[u * R + r], ng), ug), ng);
                    hout[r] = h2;
                    p.out[(long long)row[r] * p.out_pitch + d.out_off + u] = h2;
                } else if (!kGru && row[r] >= 0) {                   // gate order i, f, g, o (torch.nn.LSTM)
                    const float c2 = __fadd_rn(__fmul_rn(seq_sigmoid(acc[1][r]), c[r]), __fmul_rn(seq_sigmoid(acc[0][r]), tanhf(acc[2][r])));
                    const float h2 = __fmul_rn(seq_sigmoid(acc[kAcc - 1][r]), tanhf(c2));
                    c[r] = c2;
                    hout[r] = h2;
                    p.out[(long long)row[r] * p.out_pitch + d.out_off + u] = h2;
                } else {
                    hout[r] = hc[u * R + r];                         // finished (or absent) utterance: state frozen
                }
            }
#pragma unroll
            for (int q = 0; q < R / 4; ++q)
                *reinterpret_cast<float4 *>(hn + u * R + 4 * q) = make_float4(hout[4 * q], hout[4 * q + 1], hout[4 * q + 2], hout[4 * q + 3]);
        }
        __syncthreads();
    }
}

__global__ void __launch_bounds__(kSeqMaxThreads, 1)
lstm_seq_kernel(const SeqParams p)
{
    extern __shared__ __align__(16) float seq_smem[];
    const int grp = blockIdx.x;
    const SeqDir &d = p.dir[blockIdx.y];
    const int first = p.group_first[grp], rows = p.group_rows[grp];
    if (rows <= 4) lstm_seq_body<false, 4>(p, d, first, rows, seq_smem);
    else if (rows <= 8) lstm_seq_body<false, 8>(p, d, first, rows, seq_smem);
    else lstm_seq_body<false, 16>(p, d, first, rows, seq_smem);
}

__global__ void __launch_bounds__(kSeqMaxThreads, 1)
gru_seq_kernel(const SeqParams p)
{
    extern __shared__ __align__(16) float seq_smem[];
    const int grp = blockIdx.x;
    const SeqDir &d = p.dir[blockIdx.y];
    const int first = p.group_first[grp], rows = p.group_rows[grp];
    if (rows <= 4) lstm_seq_body<true, 4>(p, d, first, rows, seq_smem);
    else if (rows <= 8) lstm_seq_body<true, 8>(p, d, first, rows, seq_smem);
    else lstm_seq_body<true, 16>(p, d, first, rows, seq_smem);
}

}  // namespace e2e

namespace {

int sequence_impl(const char *name, bool gru, const float *gates, long long gates_pitch, float *out, long long out_pitch,
                  const int *frame_off, const int *lens, const int *group_first, const int *group_rows,
                  int N, int H, int n_groups, int n_dirs,
                  const float *bias_fw, const float *w_t_fw, int gate_off_fw, int out_off_fw,
                  const float *bias_bw, const float *w_t_bw, int gate_off_bw, int out_off_bw, void *stream)
{
    using namespace e2e;
    const int n_gates = gru ? 3 : 4;
    if (!gates || !out || !frame_off || !lens || !group_first || !group_rows || !w_t_fw || (n_dirs == 2 && !w_t_bw))
        return set_error(E2E_ERR_ARG, "%s: null pointer", name);
    if (N <= 0 || H <= 0 || n_groups <= 0 || (n_dirs != 1 && n_dirs != 2) || gates_pitch < (long long)n_gates * H || out_pitch < H)
        return set_error(E2E_ERR_ARG, "%s: bad size", name);
    if (H > kSeqMaxThreads) return set_error(E2E_ERR_UNSUPPORTED, "%s: hidden size %d > %d", name, H, kSeqMaxThreads);
    SeqParams p;
    p.gates = gates; p.gates_pitch = gates_pitch; p.out = out; p.out_pitch = out_pitch;
    p.frame_off = frame_off; p.lens = lens; p.group_first = group_first; p.group_rows = group_rows;
    p.N = N; p.H = H; p.n_groups = n_groups;
    p.dir[0] = SeqDir{bias_fw, w_t_fw, gate_off_fw, out_off_fw, 0};
    p.dir[1] = SeqDir{bias_bw, w_t_bw, gate_off_bw, out_off_bw, 1};
    const int threads = (H + 31) / 32 * 32;
    const size_t smem = ((size_t)2 * H * 16 + 2 * 16) * 4;
    if (smem > 200 * 1024) return set_error(E2E_ERR_UNSUPPORTED, "%s: %zu bytes of shared memory needed", name, smem);
    const auto kernel = gru ? gru_seq_kernel : lstm_seq_kernel;
    if (smem > 48 * 1024) {
        cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return set_error(E2E_ERR_LAUNCH, "cudaFuncSetAttribute: %s", cudaGetErrorString(e));
    }
    kernel<<<dim3(n_groups, n_dirs), threads, smem, static_cast<cudaStream_t>(stream)>>>(p);
    count_launch();
    return check_launch(name);
}

}  // namespace

extern "C" int e2e_lstm_sequence(const float *gates, long long gates_pitch, float *out, long long out_pitch,
                                 const int *frame_off, const int *lens, const int *group_first, const int *group_rows,
                                 int N, int H, int n_groups, int n_dirs,
                                 const float *bias_fw, const float *w_t_fw, int gate_off_fw, int out_off_fw,
                                 const float *bias_bw, const float *w_t_bw, int gate_off_bw, int out_off_bw,
                                 void *stream)
{
    return sequence_impl("e2e_lstm_sequence", false, gates, gates_pitch, out, out_pitch, frame_off, lens, group_first, group_rows,
                         N, H, n_groups, n_dirs, bias_fw, w_t_fw, gate_off_fw, out_off_fw, bias_bw, w_t_bw, gate_off_bw, out_off_bw,
                         stream);
}

extern "C" int e2e_gru_sequence(const float *gates, long long gates_pitch, float *out, long long out_pitch,
                                const int *frame_off, const int *lens, const int *group_first, const int *group_rows,
                                int N, int H, int n_groups, int n_dirs,
                                const float *bias_fw, const float *w_t_fw, int gate_off_fw, int out_off_fw,
                                const float *bias_bw, const float *w_t_bw, int gate_off_bw, int out_off_bw,
                                void *stream)
{
    return sequence_impl("e2e_gru_sequence", true, gates, gates_pitch, out, out_pitch, frame_off, lens, group_first, group_rows,
                         N, H, n_groups, n_dirs, bias_fw, w_t_fw, gate_off_fw, out_off_fw, bias_bw, w_t_bw, gate_off_bw, out_off_bw,
                         stream);
}
