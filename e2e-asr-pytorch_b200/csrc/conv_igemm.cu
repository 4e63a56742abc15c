// 3x3 "same" convolution of the VGG front end as ONE implicit split GEMM on the tcgen05 tensor cores
// (SURVEY.md §8f row f-4; DESIGN.md §4).  The arithmetic is that of the unfold path (conv_split.cu +
// three library GEMMs + bias_relu_mask(_pool)_kernel), bit for bit:
//     y[p][co] = sum_k A[p][k] * Wmat[k][co],   k = (dy*3 + dx)*C + c,   A = a1 + a2 + a3 (exact bf16 split)
// with the six partial products grouped by magnitude into three fp32 accumulators, each summed in the K order
// the library GEMMs sum it (stepper.SplitLinear):
//     acc0 = a1.w1                     (addmm #2:   a1 @ w1)
//     acc1 = a1.w2 , a2.w1             (addmm #1:  [a1|a2] @ [w2;w1])
//     acc2 = a1.w3 , a2.w2 , a3.w1     (mm:        [a1|a2|a3] @ [w3;w2;w1])
//     y    = acc0 + (acc1 + acc2)      (the C round trips of mm -> addmm -> addmm)
// followed by the epilogue of the unfold path: relu(y + bias) on rows h < valid[n], 0 elsewhere, and the 2x2
// ceil-mode max pool where the layer has one.  The K loop runs in piece phases — a1 against w1, w2, w3, then a2
// against w1, w2, then a3 against w1 — so every accumulator sees its products in the library's order and each A
// piece is produced once.  Nothing but the NHWC fp32 output is written: no unfolded operand, no C round trips.
//
// CTA = 128 pixels x 128 output channels, three TMEM accumulators (384 of 512 columns), 14 warps:
//   warp 0      TMA of the weight pieces (bf16 [3][Cout][9C], 128-byte swizzle), owns the TMEM allocation
//   warp 1      one thread issues tcgen05.mma (M 128, N 128, K 16) and tcgen05.commit
//   warps 2-13  A producers in three groups of four: fp32 NHWC loads of one (tap, 64-channel) slice per stage, split
//               to the phase's bf16 piece, stored in the 128-byte swizzled K-major layout the MMA reads; then the
//               epilogue (tcgen05.ld 32x32b: thread <-> pixel row, registers <-> channels, a group per 32 columns).
// Pooled layers order the tile's rows window-major (row m = 4*j + 2*dy + dx for pooled pixel j), so the four
// pixels of a window are four adjacent lanes of one warp.
//
// Built into libe2e_asr_b200_tc.so (see conv_igemm.cuh); the C entry points are in conv_igemm_host.cu.
#include "common.cuh"
#include "conv_igemm.cuh"
#include <cuda_bf16.h>

namespace e2e {
namespace {

constexpr int kBM = kIgemmBM, kBN = kIgemmBN, kBK = kIgemmBK;
constexpr int kTile = kBM * kBK * 2;          // 16 KB; A and B tiles alike
constexpr int kBStages = 6;
constexpr int kBarBytes = 256;                // mbarriers + the TMEM address word
// kGroups groups of 4 producer warps fill the A stages round robin (stage s always by group s % kGroups), so that
// kGroups stages are loaded and split at once.  Measured on the B200 (tools/bench_vgg_igemm.py, 128->128 layer):
// 1 group 324, 2 groups 477, 3 groups 602 TFLOP/s of bf16 work; loading a group's next stage ahead of splitting the
// current one gained nothing (336 / 461), so the producers are bound by their L2 traffic, not by load latency.
constexpr int kGroups = 3;
constexpr int kAStages = 2 * kGroups;
constexpr int kThreads = 64 + 128 * kGroups;
constexpr int kSmemBytes = 1024 + (kAStages + kBStages) * kTile + kBarBytes + kBM * 16;   // + alignment slack, row table

static_assert((2 * (kAStages + kBStages) + 1) * 8 + 4 <= kBarBytes, "barrier block");

// the fields of the tcgen05 instruction descriptor (kind::f16): fp32 D, bf16 A and B, both K-major, M 128, N 128
constexpr uint32_t kIdesc = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(kBN >> 3) << 17) | ((uint32_t)(kBM >> 4) << 24);

// shared-memory matrix descriptor: K-major, 128-byte swizzle, 8-row core groups 1024 bytes apart (SBO), version 1
__device__ __forceinline__ uint64_t sw128_desc(uint32_t saddr)
{
    return (uint64_t)((saddr >> 4) & 0x3fffu) | ((uint64_t)1 << 16) | ((uint64_t)(1024 >> 4) << 32) | ((uint64_t)1 << 46) |
           ((uint64_t)2 << 61);
}

__device__ __forceinline__ void mbar_arrive(uint64_t *bar)
{
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}

__device__ __forceinline__ void tma_load_2d(void *dst, const CUtensorMap *map, int c0, int c1, uint64_t *bar)
{
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
                 ::"r"(smem_u32(dst)), "l"(map), "r"(c0), "r"(c1), "r"(smem_u32(bar))
                 : "memory");
}

__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }

__device__ __forceinline__ void tc_mma(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t accumulate)
{
    asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
                 "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
                 ::"r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(kIdesc), "r"(accumulate));
}

// arrives on `bar` once every tcgen05.mma this thread issued before has completed
__device__ __forceinline__ void tc_commit(uint64_t *bar)
{
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}

__device__ __forceinline__ void tmem_ld32(uint32_t taddr, float (&v)[32])
{
    uint32_t *r = reinterpret_cast<uint32_t *>(v);
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
                 "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
                   "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
                   "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
                   "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
                 : "r"(taddr));
}

// piece `pp` (0: a1, 1: a2, 2: a3) of the exact 3-piece bf16 split (conv_split3) of x0 and x1, packed (x0 low)
__device__ __forceinline__ uint32_t split_piece2(float x0, float x1, int pp)
{
    __nv_bfloat162 p = __floats2bfloat162_rn(x0, x1);
    if (pp > 0) {
        const float2 a = __bfloat1622float2(p);
        x0 = __fsub_rn(x0, a.x);
        x1 = __fsub_rn(x1, a.y);
        p = __floats2bfloat162_rn(x0, x1);
        if (pp > 1) {
            const float2 b = __bfloat1622float2(p);
            p = __floats2bfloat162_rn(__fsub_rn(x0, b.x), __fsub_rn(x1, b.y));
        }
    }
    return *reinterpret_cast<uint32_t *>(&p);
}

// one row of the tile: its pixel and which of its nine taps read input (in the image, source row < valid[n])
struct alignas(16) IgemmRow {
    const float *pix;         // the pixel's own channels in the input
    uint32_t flags;           // bit t = dy*3 + dx: tap t reads; kRowLive: h < valid[n]; kRowPixel: the row is a pixel
    uint32_t pad;
};
constexpr uint32_t kRowLive = 1u << 9, kRowPixel = 1u << 10;

__global__ void __launch_bounds__(kThreads, 1)
conv3x3_igemm_kernel(const __grid_constant__ CUtensorMap wmap, const IgemmArgs args)
{
    extern __shared__ uint8_t igemm_smem_raw[];
    uint8_t *smem = reinterpret_cast<uint8_t *>((reinterpret_cast<uintptr_t>(igemm_smem_raw) + 1023) & ~(uintptr_t)1023);
    uint8_t *a_ring = smem;
    uint8_t *b_ring = smem + kAStages * kTile;
    uint64_t *bars = reinterpret_cast<uint64_t *>(b_ring + kBStages * kTile);
    uint64_t *a_full = bars, *a_empty = bars + kAStages;
    uint64_t *b_full = bars + 2 * kAStages, *b_empty = b_full + kBStages;
    uint64_t *acc_full = b_empty + kBStages;
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(acc_full + 1);
    IgemmRow *rows = reinterpret_cast<IgemmRow *>(reinterpret_cast<uint8_t *>(bars) + kBarBytes);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int H = args.H, W = args.W, C = args.C;
    const bool pool = args.epi == kEpiPool;
    const int n0 = blockIdx.y * kBN;
    const int KB = 9 * C / kBK;                                    // K blocks per piece

    if (threadIdx.x == 0) {
        for (int i = 0; i < kAStages; ++i) { mbar_init(a_full + i, 128); mbar_init(a_empty + i, 1); }
        for (int i = 0; i < kBStages; ++i) { mbar_init(b_full + i, 1); mbar_init(b_empty + i, 1); }
        mbar_init(acc_full, 1);
        mbar_fence_init();
    }
    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 512;" ::"r"(smem_u32(tmem_slot)) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    if (threadIdx.x >= 64 && threadIdx.x < 64 + kBM) {
        const int m = threadIdx.x - 64;
        int h = 0, w = 0, n = -1;
        if (pool) {
            const int H2 = (H + 1) >> 1, W2 = (W + 1) >> 1;
            const long long q = (long long)blockIdx.x * (kBM / 4) + (m >> 2);
            if (q < (long long)args.N * H2 * W2) {
                const int w2 = (int)(q % W2);
                const long long t = q / W2;
                h = 2 * (int)(t % H2) + ((m >> 1) & 1);
                w = 2 * w2 + (m & 1);
                if (h < H && w < W) n = (int)(t / H2);
            }
        } else {
            const long long p = (long long)blockIdx.x * kBM + m;
            if (p < (long long)args.N * H * W) {
                const long long t = p / W;
                w = (int)(p % W);
                h = (int)(t % H);
                n = (int)(t / H);
            }
        }
        IgemmRow r = {args.in, 0u, 0u};
        if (n >= 0) {
            const int vr = __ldg(args.valid + n);
            r.pix = args.in + (((long long)n * H + h) * W + w) * C;
            r.flags = kRowPixel | (h < vr ? kRowLive : 0u);
            for (int t = 0; t < 9; ++t) {
                const int hs = h + t / 3 - 1, ws = w + t % 3 - 1;
                if (hs >= 0 && hs < H && hs < vr && ws >= 0 && ws < W) r.flags |= 1u << t;
            }
        }
        rows[m] = r;
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = *tmem_slot;

    if (warp == 0) {
        // ---- weight tiles: the same (phase, K block, piece) sequence the MMA thread consumes
        if (lane == 0) {
            int stage = 0;
            uint32_t phase = 0;
            for (int pp = 0; pp < 3; ++pp)
                for (int kb = 0; kb < KB; ++kb)
                    for (int j = 0; j < 3 - pp; ++j) {
                        mbar_wait(b_empty + stage, phase ^ 1u);
                        mbar_arrive_expect_tx(b_full + stage, kTile);
                        tma_load_2d(b_ring + stage * kTile, &wmap, kb * kBK, j * args.Cout + n0, b_full + stage);
                        if (++stage == kBStages) { stage = 0; phase ^= 1u; }
                    }
        }
    } else if (warp == 1) {
        // ---- MMA issue: accumulator pp + j gets A piece pp times weight piece j
        if (lane == 0) {
            int as = 0, bs = 0;
            uint32_t aph = 0, bph = 0;
            for (int pp = 0; pp < 3; ++pp)
                for (int kb = 0; kb < KB; ++kb) {
                    mbar_wait(a_full + as, aph);
                    tc_fence_after();
                    const uint64_t adesc = sw128_desc(smem_u32(a_ring + as * kTile));
                    for (int j = 0; j < 3 - pp; ++j) {
                        mbar_wait(b_full + bs, bph);
                        tc_fence_after();
                        const uint64_t bdesc = sw128_desc(smem_u32(b_ring + bs * kTile));
#pragma unroll
                        for (int k16 = 0; k16 < kBK / 16; ++k16)         // +32 bytes inside the swizzle row per K step
                            tc_mma(tmem + (uint32_t)((pp + j) * kBN), adesc + 2 * k16, bdesc + 2 * k16,
                                   (pp > 0 || kb > 0 || k16 > 0) ? 1u : 0u);
                        tc_commit(b_empty + bs);
                        if (++bs == kBStages) { bs = 0; bph ^= 1u; }
                    }
                    tc_commit(a_empty + as);
                    if (++as == kAStages) { as = 0; aph ^= 1u; }
                }
            tc_commit(acc_full);
        }
    } else {
        // ---- A producers: 16 lanes per pixel row (4 channels each), 8 rows per pass, 16 passes per stage
        const int grp = (threadIdx.x - 64) >> 7, pt = (threadIdx.x - 64) & 127;
        const int c16 = pt & 15, rsub = pt >> 4;
        const int cpb = C / kBK;                                   // K blocks per tap
        // this group's stages: sequence numbers seq = grp, grp + kGroups, .. of the (piece, K block) order
        int as = grp;
        uint32_t aph = 0;
        for (int seq = grp; seq < 3 * KB; seq += kGroups) {
            const int pp = seq / KB, kb = seq - pp * KB, tap = kb / cpb, cb = kb - tap * cpb;
            const long long tap_off = ((long long)(tap / 3 - 1) * W + (tap % 3 - 1)) * C + cb * kBK + c16 * 4;
            float4 v[kBM / 8];
#pragma unroll
            for (int i = 0; i < kBM / 8; ++i) {
                const IgemmRow r = rows[i * 8 + rsub];
                v[i] = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
                if ((r.flags >> tap) & 1u) v[i] = __ldg(reinterpret_cast<const float4 *>(r.pix + tap_off));
            }
            mbar_wait(a_empty + as, aph ^ 1u);
            uint8_t *tile = a_ring + as * kTile;
#pragma unroll
            for (int i = 0; i < kBM / 8; ++i) {
                const int row = i * 8 + rsub;
                const uint32_t lo = split_piece2(v[i].x, v[i].y, pp), hi = split_piece2(v[i].z, v[i].w, pp);
                const int chunk = (c16 >> 1) ^ (row & 7);                                 // 128-byte swizzle
                *reinterpret_cast<uint2 *>(tile + row * 128 + chunk * 16 + (c16 & 1) * 8) = make_uint2(lo, hi);
            }
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");                 // generic writes -> MMA reads
            mbar_arrive(a_full + as);
            as += kGroups;
            if (as >= kAStages) { as -= kAStages; aph ^= 1u; }
        }

        // ---- epilogue: warp w reads TMEM lanes 32*(w % 4) ..; this thread holds tile row m; the groups share the
        //      32-column chunks
        const int m = (warp & 3) * 32 + lane;
        const uint32_t flags = rows[m].flags;
        mbar_wait(acc_full, 0);
        tc_fence_after();
        const uint32_t lane_addr = tmem + ((uint32_t)((warp & 3) * 32) << 16);
        const long long H2W2 = (long long)((H + 1) >> 1) * ((W + 1) >> 1);
        const bool live = (flags & kRowLive) != 0u, pixel = (flags & kRowPixel) != 0u;
        for (int c = grp; c < kBN / 32; c += kGroups) {
            float y0[32], y1[32], y2[32];
            tmem_ld32(lane_addr + c * 32, y0);
            tmem_ld32(lane_addr + kBN + c * 32, y1);
            tmem_ld32(lane_addr + 2 * kBN + c * 32, y2);
            asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
            float y[32];
#pragma unroll
            for (int i = 0; i < 32; ++i) y[i] = __fadd_rn(y0[i], __fadd_rn(y1[i], y2[i]));
            const int col = n0 + c * 32;
            if (args.epi == kEpiRaw) {
                if (pixel) {
                    float4 *dst = reinterpret_cast<float4 *>(args.out + ((long long)blockIdx.x * kBM + m) * args.Cout + col);
#pragma unroll
                    for (int i = 0; i < 8; ++i) dst[i] = make_float4(y[4 * i], y[4 * i + 1], y[4 * i + 2], y[4 * i + 3]);
                }
            } else if (!pool) {
                if (pixel) {
                    float4 *dst = reinterpret_cast<float4 *>(args.out + ((long long)blockIdx.x * kBM + m) * args.Cout + col);
#pragma unroll
                    for (int i = 0; i < 8; ++i) {
                        float4 o = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
                        if (live) {
                            const float4 b = __ldg(reinterpret_cast<const float4 *>(args.bias + col) + i);
                            o.x = fmaxf(__fadd_rn(y[4 * i], b.x), 0.0f); o.y = fmaxf(__fadd_rn(y[4 * i + 1], b.y), 0.0f);
                            o.z = fmaxf(__fadd_rn(y[4 * i + 2], b.z), 0.0f); o.w = fmaxf(__fadd_rn(y[4 * i + 3], b.w), 0.0f);
                        }
                        dst[i] = o;
                    }
                }
            } else {
                // window pixel s = m & 3 (dy*2 + dx); the maximum runs from 0 over the live pixels in (dy, dx) order,
                // as bias_relu_mask_pool_kernel does; lane s of the window writes channels 8s .. 8s+7 of the chunk
                const int s = m & 3, base = lane & ~3;
                float t[32];
#pragma unroll
                for (int i = 0; i < 32; ++i) t[i] = live ? __fadd_rn(y[i], __ldg(args.bias + col + i)) : -INFINITY;
                float res[8];
#pragma unroll
                for (int i = 0; i < 32; ++i) {
                    float acc = 0.0f;
#pragma unroll
                    for (int k = 0; k < 4; ++k) acc = fmaxf(acc, __shfl_sync(E2E_FULL_MASK, t[i], base + k));
                    if ((i >> 3) == s) res[i & 7] = acc;
                }
                const long long q = (long long)blockIdx.x * (kBM / 4) + (m >> 2);
                if (q < (long long)args.N * H2W2) {
                    float4 *dst = reinterpret_cast<float4 *>(args.out + q * args.Cout + col + 8 * s);
                    dst[0] = make_float4(res[0], res[1], res[2], res[3]);
                    dst[1] = make_float4(res[4], res[5], res[6], res[7]);
                }
            }
        }
        tc_fence_before();
    }
    __syncthreads();
    if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 512;" ::"r"(tmem) : "memory");
}

}  // namespace
}  // namespace e2e

extern "C" int e2e_tc_conv3x3_igemm_launch(const CUtensorMap *wmap, const e2e::IgemmArgs *args, unsigned tiles, void *stream)
{
    using namespace e2e;
    static bool attr_set = false;
    if (!attr_set) {
        const cudaError_t e = cudaFuncSetAttribute(conv3x3_igemm_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemBytes);
        if (e != cudaSuccess) return (int)e;
        attr_set = true;
    }
    conv3x3_igemm_kernel<<<dim3(tiles, (unsigned)(args->Cout / kBN)), kThreads, kSmemBytes, static_cast<cudaStream_t>(stream)>>>(*wmap, *args);
    return (int)cudaGetLastError();
}
