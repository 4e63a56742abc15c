// C entry points of the 3x3 convolution as one tcgen05 implicit split GEMM: argument checks, the shape query and the
// weight tensor map.  The kernel itself is in conv_igemm.cu, built into libe2e_asr_b200_tc.so (see conv_igemm.cuh).
#include "common.cuh"
#include "conv_igemm.cuh"

namespace e2e {

typedef CUresult (*EncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *, const cuuint64_t *,
                                  const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
EncodeTiledFn tensor_map_encoder();   // prefix_score.cu

namespace {

bool igemm_shape_ok(int C, int Cout)
{
    return (C == 128 || C == 256) && (Cout == 128 || Cout == 256);
}

}  // namespace
}  // namespace e2e

using namespace e2e;

extern "C" int e2e_conv3x3_igemm_supported(int C, int Cout)
{
    return igemm_shape_ok(C, Cout) ? 1 : 0;
}

extern "C" int e2e_conv3x3_igemm(const float *in_nhwc, const int *valid_rows, int N, int H, int W, int C,
                                 const void *w_split_bf16, const float *bias, int Cout, int epilogue, float *out, void *stream)
{
    const char *name = "e2e_conv3x3_igemm";
    if (!in_nhwc || !valid_rows || !w_split_bf16 || !out || (epilogue != kEpiRaw && !bias))
        return set_error(E2E_ERR_ARG, "%s: null pointer", name);
    if (N <= 0 || H <= 0 || W <= 0 || epilogue < kEpiRaw || epilogue > kEpiPool)
        return set_error(E2E_ERR_ARG, "%s: bad size or epilogue", name);
    if (!igemm_shape_ok(C, Cout)) return set_error(E2E_ERR_UNSUPPORTED, "%s: C = %d, Cout = %d not supported", name, C, Cout);
    if ((reinterpret_cast<uintptr_t>(in_nhwc) & 15) || (reinterpret_cast<uintptr_t>(w_split_bf16) & 15) ||
        (reinterpret_cast<uintptr_t>(out) & 15) || (reinterpret_cast<uintptr_t>(bias) & 15))
        return set_error(E2E_ERR_ARG, "%s: misaligned buffer", name);
    const long long rows_out = epilogue == kEpiPool ? (long long)N * ((H + 1) / 2) * ((W + 1) / 2) : (long long)N * H * W;
    const long long tiles = epilogue == kEpiPool ? (rows_out + kIgemmBM / 4 - 1) / (kIgemmBM / 4) : (rows_out + kIgemmBM - 1) / kIgemmBM;
    if (tiles > 0x7fffffffLL) return set_error(E2E_ERR_ARG, "%s: too many pixels", name);

    EncodeTiledFn enc = tensor_map_encoder();
    if (!enc) return set_error(E2E_ERR_LAUNCH, "%s: cuTensorMapEncodeTiled is not available from this driver", name);
    CUtensorMap map;
    const cuuint64_t dims[2] = {(cuuint64_t)9 * C, (cuuint64_t)3 * Cout};                 // [3][Cout][9C] bf16, K innermost
    const cuuint64_t strides[1] = {(cuuint64_t)9 * C * 2};
    const cuuint32_t box[2] = {(cuuint32_t)kIgemmBK, (cuuint32_t)kIgemmBN};
    const cuuint32_t estr[2] = {1u, 1u};
    const CUresult cr = enc(&map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void *>(w_split_bf16), dims, strides, box, estr,
                            CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                            CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (cr != CUDA_SUCCESS) return set_error(E2E_ERR_LAUNCH, "%s: cuTensorMapEncodeTiled failed (CUresult %d)", name, (int)cr);

    const IgemmArgs a = {in_nhwc, valid_rows, bias, out, N, H, W, C, Cout, epilogue};
    const int e = e2e_tc_conv3x3_igemm_launch(&map, &a, (unsigned)tiles, stream);
    count_launch();
    if (e != (int)cudaSuccess) return set_error(E2E_ERR_LAUNCH, "%s: %s", name, cudaGetErrorString((cudaError_t)e));
    return check_launch(name);
}
