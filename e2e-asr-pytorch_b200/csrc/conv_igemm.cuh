// Interface between the host entry points of the implicit-GEMM convolution (conv_igemm_host.cu, in
// libe2e_asr_b200.so) and its tcgen05 kernel (conv_igemm.cu, in libe2e_asr_b200_tc.so).  The tensor-core kernel is built
// into a library of its own, which the main library links against: libe2e_asr_b200.so itself holds no tensor-core
// contraction (tests/test_abi.py), and the launcher below is self-contained so that the kernel library needs nothing
// from it.
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>

namespace e2e {

constexpr int kIgemmBM = 128;                 // pixels per CTA = TMEM lanes
constexpr int kIgemmBN = 128;                 // output channels per CTA = columns of one accumulator
constexpr int kIgemmBK = 64;                  // K per stage: one 128-byte swizzle row of bf16

enum { kEpiRaw = 0, kEpiRelu = 1, kEpiPool = 2 };

struct IgemmArgs {
    const float *in;          // [N][H][W][C] fp32
    const int *valid;         // [N]
    const float *bias;        // [Cout]
    float *out;               // raw / relu: [N*H*W][Cout]; pool: [N][ceil(H/2)][ceil(W/2)][Cout]
    int N, H, W, C, Cout, epi;
};

}  // namespace e2e

// Launches conv3x3_igemm_kernel on `stream` over `tiles` pixel tiles x Cout / 128 channel blocks; `wmap` is the
// tensor map of the weight pieces (bf16 [3][Cout][9C], box 64 x 128, 128-byte swizzle).  Returns the cudaError_t of
// the launch (the kernel library's own runtime state).
extern "C" int e2e_tc_conv3x3_igemm_launch(const CUtensorMap *wmap, const e2e::IgemmArgs *args, unsigned tiles, void *stream);
