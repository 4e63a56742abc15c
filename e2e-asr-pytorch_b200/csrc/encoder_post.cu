// Post-processing of an encoder layer's packed recurrence output (RNNLayer, src/module.py:1003-1081, in the order of
// RecurrentLayer._post): LayerNorm over each full output row, then frame sub-sampling by dropping (keep t = 0, r, 2r, ..)
// or by concatenating r consecutive frames into one row.  Both are a gather of source rows, so one kernel does either,
// with or without the LayerNorm:
//   out[out_off[n] + j][s*W : (s+1)*W] = LN(in[in_off[n] + j*stride + s])      for j < out_len[n], s < g
// drop: stride r, g = 1;  concat: stride r, g = r;  LayerNorm alone: stride 1, g = 1.
// One warp per source row: the mean, then the biased variance around it (two passes, as nn.LayerNorm), then the
// normalised row.  The row (at most 2 x 1024 floats) is read three times; the second and third reads hit L1.  Memory
// bound, no tensor cores.
#include "common.cuh"

namespace e2e {

constexpr int kPostWarps = 8;

struct PostParams {
    const float *in; long long in_pitch;
    float *out; long long out_pitch;
    const int *in_off, *out_off, *out_len;
    const float *w, *b;
    int N, W, stride, g;
    float eps;
};

__global__ void __launch_bounds__(kPostWarps * 32)
packed_subsample_ln_kernel(const PostParams p)
{
    const int n = blockIdx.x, lane = threadIdx.x & 31;
    const long long rows = (long long)__ldg(p.out_len + n) * p.g;     // (output row, slot) pairs of utterance n
    const long long src0 = __ldg(p.in_off + n), dst0 = __ldg(p.out_off + n);
    const int W = p.W;
    for (long long q = (long long)blockIdx.y * kPostWarps + (threadIdx.x >> 5); q < rows; q += (long long)gridDim.y * kPostWarps) {
        const long long j = q / p.g;
        const int s = (int)(q - j * p.g);
        const float *src = p.in + (src0 + j * p.stride + s) * p.in_pitch;
        float *dst = p.out + (dst0 + j) * p.out_pitch + (long long)s * W;
        if (!p.w) {
            for (int i = lane; i < W; i += 32) dst[i] = src[i];
            continue;
        }
        float sum = 0.0f;
        for (int i = lane; i < W; i += 32) sum += src[i];
        const float mean = warp_sum(sum) / (float)W;
        float sq = 0.0f;
        for (int i = lane; i < W; i += 32) {
            const float d = src[i] - mean;
            sq = fmaf(d, d, sq);
        }
        const float rstd = __frsqrt_rn(warp_sum(sq) / (float)W + p.eps);
        for (int i = lane; i < W; i += 32)
            dst[i] = fmaf((src[i] - mean) * rstd, __ldg(p.w + i), p.b ? __ldg(p.b + i) : 0.0f);
    }
}

}  // namespace e2e

extern "C" int e2e_packed_subsample_ln(const float *in, long long in_pitch, float *out, long long out_pitch,
                                       const int *in_off, const int *out_off, const int *out_len, int N, int W,
                                       int stride, int g, const float *ln_weight, const float *ln_bias, float eps,
                                       void *stream)
{
    using namespace e2e;
    const char *name = "e2e_packed_subsample_ln";
    if (!in || !out || !in_off || !out_off || !out_len || (!ln_weight && ln_bias))
        return set_error(E2E_ERR_ARG, "%s: null pointer", name);
    if (N <= 0 || W <= 0 || stride <= 0 || (g != 1 && g != stride))
        return set_error(E2E_ERR_ARG, "%s: bad size (N %d, W %d, stride %d, g %d)", name, N, W, stride, g);
    if (in_pitch < W || out_pitch < (long long)g * W)
        return set_error(E2E_ERR_ARG, "%s: bad pitch (in %lld, out %lld for W %d, g %d)", name, in_pitch, out_pitch, W, g);
    if (ln_weight && !(eps > 0.0f)) return set_error(E2E_ERR_ARG, "%s: eps must be > 0", name);
    PostParams p;
    p.in = in; p.in_pitch = in_pitch; p.out = out; p.out_pitch = out_pitch;
    p.in_off = in_off; p.out_off = out_off; p.out_len = out_len;
    p.w = ln_weight; p.b = ln_bias;
    p.N = N; p.W = W; p.stride = stride; p.g = g; p.eps = eps;
    // about 32 resident warps per SM over all utterances; each warp strides over its utterance's rows
    const int per_utt = (148 * 4 + N - 1) / N;
    packed_subsample_ln_kernel<<<dim3(N, per_utt), kPostWarps * 32, 0, static_cast<cudaStream_t>(stream)>>>(p);
    count_launch();
    return check_launch(name);
}
