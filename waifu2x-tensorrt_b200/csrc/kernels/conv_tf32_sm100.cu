// tf32 convolutions (--precision tf32): fp32 NHWC activations, fp32 K-major weights, tcgen05.mma kind::tf32, fp32 accumulate,
// fp32 epilogues.  The numerics the reference's TF32 TensorRT engine promises (SURVEY q13): fp32 storage range (activations above
// 65504, weights below 6e-8 survive), TF32 products, fp32 sums.
//
//   conv_tf32_kernel   implicit GEMM over the same 5-D view and tap list as the fp16 igemm_kernel (conv_igemm_sm100.cu):
//                      D[128 pixels, N] (fp32, TMEM) += A[128 pixels, K] (fp32 smem) x B[N, K] (fp32 smem), both K-major, 128B swizzle.
//                      One K chunk is 32 floats = one 128-byte swizzled row; a UMMA K step is 8 tf32 elements = 32 bytes, the same
//                      byte stride as 16 fp16 elements, so the descriptor stepping of the fp16 kernel carries over unchanged.
//                      Persistent CTAs; warp 0 = TMA producer (5-D activation box + weight tile per K chunk), warp 1 = TMEM allocator
//                      + single-thread MMA issuer, warps 2..9 = epilogue (tcgen05.ld -> bias / activation / skip -> direct fp32 stores).
//                      Two TMEM accumulators, an mbarrier ring between TMA and MMA.  SE layers produce their squeeze sums in the
//                      epilogue, exact int64 fixed-point like the fp16 kernels (kSeFixedScale).
//   conv_first_f32     the RGB first layers (cin = 4 -> 32): a 16-byte tap is less than one UMMA K step, so they run on the CUDA
//                      cores in fp32 FMA (about 1 % of the model's FLOPs).
#include <cuda.h>
#include <cuda_runtime.h>

#include <algorithm>
#include <cstdio>
#include <string>

#include "../hostutil.h"
#include "../model_pack.h"
#include "conv_params.h"
#include "launch.h"
#include "sm100_common.cuh"

namespace w2x {

using namespace sm100;

struct Tf32Args {
    CUtensorMap tmA;  // activation view (c, x, z, y, img), box (32, bw, 1, bh, 1)
    CUtensorMap tmB;  // weights (k, n, img), box (32, bn, 1)
    ConvParamsF32 p;
    int bn, bw, bh, bwShift;
    int tilesX, tilesY, tilesN, totalTiles;
    int stages, cchunks, kblocks;
    uint32_t idesc, tmemCols, bytesA, bytesB, descHi;
};

struct Tf32Plan {
    Tf32Args args;
    int grid = 0;
    size_t smem = 0;
};

namespace {

constexpr int kKC = 32;                          // K chunk in elements (128 bytes of fp32)
constexpr int kEpiWarps = 8;                     // two warps per TMEM lane quarter, splitting the columns
constexpr int kThreads = 64 + 32 * kEpiWarps;
constexpr int kMaxStages = 8;
constexpr uint32_t kOffFull = 0, kOffEmpty = 64, kOffTFull = 128, kOffTEmpty = 144, kOffSlot = 160, kHeaderBytes = 1024;
constexpr size_t kSmemLimit = 227 * 1024;

struct Float8 { float4 a, b; };

// fp32 twin of conv_epilogue8 for the four CUNet epilogues; v = 8 raw fp32 accumulators of columns [j0, j0 + 8) of pixel (img, y, x)
__device__ __forceinline__ void conv_epilogue8_f32(const ConvParamsF32& p, int img, int y, int x, int j0, const float* v) {
    float r[8];
    if (p.mode == EPI_STORE) {
        if (j0 >= p.cout) return;
#pragma unroll
        for (int i = 0; i < 8; ++i) r[i] = lrelu(v[i] + __ldg(p.bias + j0 + i), p.slope);
        float* o = p.out + (((long long)img * p.out_h + y) * p.out_w + x) * p.out_c + j0;
        reinterpret_cast<float4*>(o)[0] = make_float4(r[0], r[1], r[2], r[3]);
        if (p.cout - j0 >= 8) reinterpret_cast<float4*>(o)[1] = make_float4(r[4], r[5], r[6], r[7]);
    } else if (p.mode == EPI_D2S) {
        const int q = j0 / p.cout, co = j0 - q * p.cout;
        const int oy = 2 * y + (q >> 1), ox = 2 * x + (q & 1);
#pragma unroll
        for (int i = 0; i < 8; ++i) r[i] = lrelu(v[i] + __ldg(p.bias + j0 + i), p.slope);
        if (p.skip) {
            const Float8 sv = *reinterpret_cast<const Float8*>(p.skip + (((long long)img * p.skip_h + oy + p.skip_off) * p.skip_w + ox + p.skip_off) * p.skip_c + co);
            float f[8] = {sv.a.x, sv.a.y, sv.a.z, sv.a.w, sv.b.x, sv.b.y, sv.b.z, sv.b.w};
            if (p.skip_scale) {
#pragma unroll
                for (int i = 0; i < 8; ++i) f[i] *= __ldg(p.skip_scale + (long long)img * p.skip_c + co + i);
            }
#pragma unroll
            for (int i = 0; i < 8; ++i) r[i] += f[i];
        }
        float* o = p.out + (((long long)img * p.out_h + oy) * p.out_w + ox) * p.out_c + co;
        reinterpret_cast<float4*>(o)[0] = make_float4(r[0], r[1], r[2], r[3]);
        reinterpret_cast<float4*>(o)[1] = make_float4(r[4], r[5], r[6], r[7]);
    } else if (p.mode == EPI_UP4) {
        if (j0 >= 16) return;
#pragma unroll
        for (int hsel = 0; hsel < 2; ++hsel) {
            const int q = (j0 >> 2) + hsel;
            const int oy = 2 * y - 1 + (q >> 1), ox = 2 * x - 1 + (q & 1);
            if (oy < 0 || ox < 0 || oy >= p.out_h || ox >= p.out_w) continue;
            const float* vv = v + 4 * hsel;
            const float* bb = p.bias + j0 + 4 * hsel;
            *reinterpret_cast<float4*>(p.out + (((long long)img * p.out_h + oy) * p.out_w + ox) * p.out_c) =
                make_float4(vv[0] + __ldg(bb + 0), vv[1] + __ldg(bb + 1), vv[2] + __ldg(bb + 2), vv[3] + __ldg(bb + 3));
        }
    } else {  // EPI_FINAL
        if (j0 != 0) return;
        const float4 s = *reinterpret_cast<const float4*>(p.skip + (((long long)img * p.skip_h + y + p.skip_off) * p.skip_w + x + p.skip_off) * p.skip_c);
        *reinterpret_cast<float4*>(p.out + (((long long)img * p.out_h + y) * p.out_w + x) * p.out_c) =
            make_float4(fminf(fmaxf(v[0] + __ldg(p.bias + 0) + s.x, 0.f), 1.f), fminf(fmaxf(v[1] + __ldg(p.bias + 1) + s.y, 0.f), 1.f),
                        fminf(fmaxf(v[2] + __ldg(p.bias + 2) + s.z, 0.f), 1.f), 0.f);
    }
}

struct TileCoord { int img, y0, x0, n0; };

__device__ __forceinline__ TileCoord tileCoord(const Tf32Args& a, int t) {
    const int tn = t % a.tilesN;
    t /= a.tilesN;
    const int tx = t % a.tilesX;
    t /= a.tilesX;
    const int ty = t % a.tilesY;
    return TileCoord{t / a.tilesY, ty * a.bh, tx * a.bw, tn * a.bn};
}

// NCOL accumulator columns [c0, c0 + NCOL) of this lane's pixel: TMEM -> epilogue -> global; SE layers also produce their squeeze sums:
// the exact sum over the warp's 32 pixels of round(output * 2^10) per column, in int64 (fp32 outputs can exceed the fp16 range that keeps
// the fp16 kernels' int32 warp sums safe), one integer atomic per column and tile
template <int NCOL>
__device__ __forceinline__ void epilogueChunk(const ConvParamsF32& p, uint32_t taddr, const TileCoord& tc, int c0, int y, int x, bool valid, int lane) {
    uint32_t r[32];
    if (NCOL == 32) tmemLd32(taddr + (uint32_t)c0, r);
    else tmemLd16(taddr + (uint32_t)c0, r);
    tmemLdWait();
    const float* v = reinterpret_cast<const float*>(r);
    if (valid) {
#pragma unroll
        for (int q = 0; q < NCOL / 8; ++q) conv_epilogue8_f32(p, tc.img, y, x, tc.n0 + c0 + 8 * q, v + 8 * q);
    }
    if (p.se_sum) {
        long long mine = 0;
#pragma unroll
        for (int i = 0; i < NCOL; ++i) {
            long long s = valid ? __float2ll_rn(lrelu(v[i] + __ldg(p.bias + tc.n0 + c0 + i), p.slope) * kSeFixedScale) : 0ll;
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
            if (lane == i) mine = s;
        }
        if (lane < NCOL && mine != 0)
            atomicAdd(reinterpret_cast<unsigned long long*>(p.se_sum + (size_t)tc.img * p.npad + tc.n0 + c0 + lane), (unsigned long long)mine);
    }
}

__global__ void __launch_bounds__(kThreads, 1) conv_tf32_kernel(const __grid_constant__ Tf32Args a) {
    extern __shared__ uint8_t smemRaw[];
    const uint32_t rawAddr = smemU32(smemRaw);
    const uint32_t base = (rawAddr + 1023u) & ~1023u;
    uint8_t* sm = smemRaw + (base - rawAddr);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t barFull = base + kOffFull, barEmpty = base + kOffEmpty, barTFull = base + kOffTFull, barTEmpty = base + kOffTEmpty;
    if (threadIdx.x == 0) {
        for (int s = 0; s < kMaxStages; ++s) {
            mbarInit(barFull + 8u * s, 1);
            mbarInit(barEmpty + 8u * s, 1);
        }
        for (int i = 0; i < 2; ++i) {
            mbarInit(barTFull + 8u * i, 1);
            mbarInit(barTEmpty + 8u * i, kEpiWarps);
        }
        mbarInitFence();
        tmaPrefetchDesc(&a.tmA);
        tmaPrefetchDesc(&a.tmB);
    }
    if (warp == 1) tmemAlloc(smemU32(sm + kOffSlot), a.tmemCols);
    tcFenceBefore();
    __syncthreads();
    tcFenceAfter();
    const uint32_t tmemBase = *reinterpret_cast<volatile uint32_t*>(sm + kOffSlot);
    const uint32_t stage0 = base + kHeaderBytes;
    const uint32_t stageBytes = a.bytesA + a.bytesB;
    const int first = blockIdx.x, step = gridDim.x;
    pdlLaunchDependents();
    pdlWait();  // activations and SE-scaled weights come from earlier kernels

    if (warp == 0) {
        if (lane == 0) {
            int stage = 0;
            uint32_t phase = 0;
            for (int t = first; t < a.totalTiles; t += step) {
                const TileCoord tc = tileCoord(a, t);
                for (int tap = 0; tap < a.p.ntaps; ++tap) {
                    const ConvTap tp = a.p.tap[tap];
                    for (int cc = 0; cc < a.cchunks; ++cc) {
                        mbarWait(barEmpty + 8u * stage, phase ^ 1u);
                        const uint32_t full = barFull + 8u * stage;
                        const uint32_t dstA = stage0 + stage * stageBytes;
                        mbarExpectTx(full, stageBytes);
                        tmaLoad5d(dstA, &a.tmA, full, tp.c0 + cc * kKC, tc.x0 + tp.dx, tp.dz, tc.y0 + tp.dy, tc.img);
                        tmaLoad3d(dstA + a.bytesA, &a.tmB, full, tap * a.p.cin + cc * kKC, tc.n0, a.p.w_img_stride ? tc.img : 0);
                        if (++stage == a.stages) { stage = 0; phase ^= 1u; }
                    }
                }
            }
        }
    } else if (warp == 1) {
        int stage = 0, acc = 0;
        uint32_t phase = 0, accPhase = 0;
        for (int t = first; t < a.totalTiles; t += step) {
            mbarWait(barTEmpty + 8u * acc, accPhase ^ 1u);
            tcFenceAfter();
            const uint32_t tmemD = tmemBase + (uint32_t)(acc * a.bn);
            for (int kb = 0; kb < a.kblocks; ++kb) {
                mbarWait(barFull + 8u * stage, phase);
                tcFenceAfter();
                if (electOne()) {
                    const uint32_t aLo = descLo(stage0 + stage * stageBytes), bLo = descLo(stage0 + stage * stageBytes + a.bytesA);
#pragma unroll
                    for (int ks = 0; ks < kKC / 8; ++ks)
                        ummaTf32LoHi(tmemD, aLo + 2u * ks, a.descHi, bLo + 2u * ks, a.descHi, a.idesc, (kb | ks) != 0 ? 1u : 0u);
                    tcCommit(barEmpty + 8u * stage);
                    if (kb == a.kblocks - 1) tcCommit(barTFull + 8u * acc);
                }
                __syncwarp();
                if (++stage == a.stages) { stage = 0; phase ^= 1u; }
            }
            if (++acc == 2) { acc = 0; accPhase ^= 1u; }
        }
    } else {
        // warp w reads TMEM lanes 32*(w%4)..+31 (one output pixel per lane); the two warps of a lane quarter split the columns
        const int quarter = warp & 3, half = (warp - 2) >> 2;
        const int m = quarter * 32 + lane;
        const int yy = m >> a.bwShift, xx = m & (a.bw - 1);
        const bool split = a.bn >= 64;
        const int colsPerWarp = split ? a.bn >> 1 : a.bn;
        const int colBegin = split ? half * colsPerWarp : 0;
        const bool active = split || half == 0;
        int acc = 0;
        uint32_t accPhase = 0;
        for (int t = first; t < a.totalTiles; t += step) {
            const TileCoord tc = tileCoord(a, t);
            const int y = tc.y0 + yy, x = tc.x0 + xx;
            const bool valid = y < a.p.gy && x < a.p.gx;
            mbarWait(barTFull + 8u * acc, accPhase);
            tcFenceAfter();
            const uint32_t taddr = tmemBase + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(acc * a.bn);
            if (active) {
                for (int c0 = colBegin; c0 < colBegin + colsPerWarp; c0 += 32) {
                    if (colBegin + colsPerWarp - c0 >= 32) epilogueChunk<32>(a.p, taddr, tc, c0, y, x, valid, lane);
                    else epilogueChunk<16>(a.p, taddr, tc, c0, y, x, valid, lane);
                }
            }
            tcFenceBefore();
            __syncwarp();
            if (lane == 0) mbarArrive(barTEmpty + 8u * acc);
            if (++acc == 2) { acc = 0; accPhase ^= 1u; }
        }
    }

    tcFenceBefore();
    __syncthreads();
    if (warp == 1) {
        tcFenceAfter();
        tmemDealloc(tmemBase, a.tmemCols);
    }
}

// ---- RGB first layer: out[img][y][x][0..32) = lrelu(bias + sum_{tap, c < 4} in[img][y+ky][x+kx][c] * w[n][tap*4 + c]) -------------
// one output pixel per thread, the 32 x 36 weights in shared memory (broadcast reads)
__global__ void __launch_bounds__(128) conv_first_f32_kernel(const __grid_constant__ ConvParamsF32 p) {
    __shared__ float ws[32 * 36];
    __shared__ float bs[32];
    for (int i = threadIdx.x; i < 32 * 36; i += blockDim.x) ws[i] = p.w[i];
    if (threadIdx.x < 32) bs[threadIdx.x] = p.bias[threadIdx.x];
    __syncthreads();
    const int img = blockIdx.y;
    const int pix = blockIdx.x * blockDim.x + threadIdx.x;
    if (pix >= p.gx * p.gy) return;
    const int y = pix / p.gx, x = pix - y * p.gx;
    float acc[32];
#pragma unroll
    for (int n = 0; n < 32; ++n) acc[n] = bs[n];
#pragma unroll
    for (int tap = 0; tap < 9; ++tap) {
        const ConvTap tp = p.tap[tap];
        const float4 v = *reinterpret_cast<const float4*>(p.in + img * p.sn + (long long)(y + tp.dy) * p.sy + (long long)(x + tp.dx) * p.sx + tp.c0);
#pragma unroll
        for (int n = 0; n < 32; ++n) {
            const float* wr = ws + n * 36 + tap * 4;
            acc[n] = fmaf(v.x, wr[0], fmaf(v.y, wr[1], fmaf(v.z, wr[2], fmaf(v.w, wr[3], acc[n]))));
        }
    }
    float4* o = reinterpret_cast<float4*>(p.out + (((long long)img * p.out_h + y) * p.out_w + x) * p.out_c);
#pragma unroll
    for (int q = 0; q < 8; ++q)
        o[q] = make_float4(lrelu(acc[4 * q], p.slope), lrelu(acc[4 * q + 1], p.slope), lrelu(acc[4 * q + 2], p.slope), lrelu(acc[4 * q + 3], p.slope));
}

// ---- host side -------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

// fp32 tensor map, 128-byte swizzle; strides in elements
void encodeF32(CUtensorMap* tm, int rank, const void* ptr, const long long* dims, const long long* stridesElems, const int* box, const char* what) {
    static EncodeTiledFn fn = [] {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess || !p)
            throw Error("cuTensorMapEncodeTiled is not available from the CUDA driver");
        return (EncodeTiledFn)p;
    }();
    cuuint64_t d[5], s[4];
    cuuint32_t b[5], es[5] = {1, 1, 1, 1, 1};
    for (int i = 0; i < rank; ++i) { d[i] = (cuuint64_t)dims[i]; b[i] = (cuuint32_t)box[i]; }
    for (int i = 0; i + 1 < rank; ++i) s[i] = (cuuint64_t)stridesElems[i] * 4;
    const CUresult r = fn(tm, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, (cuuint32_t)rank, const_cast<void*>(ptr), d, s, b, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
                          CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) throw Error(std::string("cuTensorMapEncodeTiled(") + what + ", fp32) failed with code " + std::to_string((int)r));
}

void checkCuda(cudaError_t e) {
    if (e != cudaSuccess) throw Error(std::string("cuda: ") + cudaGetErrorString(e));
}

// N tile: the largest divisor of npad that is a multiple of 32 and <= 256 (16-wide heads stay 16)
int pickBn(int npad) {
    if (npad <= 32) return npad;
    for (int bn = 256; bn >= 32; bn -= 32)
        if (npad % bn == 0) return bn;
    return 0;
}

}  // namespace

bool tf32Supported(const ConvParamsF32& p) {
    if (p.cin % kKC != 0 || p.npad % 16 != 0 || p.npad > 1024 || (p.npad > 32 && p.npad % 32 != 0)) return false;
    if (p.ntaps < 1 || p.ntaps > 9) return false;
    if (p.mode != EPI_STORE && p.mode != EPI_D2S && p.mode != EPI_UP4 && p.mode != EPI_FINAL) return false;
    if (p.mode == EPI_STORE && (p.act != ACT_LRELU || p.skip || !(p.cout == 4 || p.cout % 8 == 0))) return false;
    if (p.mode == EPI_D2S && p.cout % 8 != 0) return false;
    if (p.se_sum && (p.mode != EPI_STORE || p.cout != p.npad)) return false;
    return true;
}

Tf32Plan* tf32CreatePlan(const ConvParamsF32& p) {
    if (!tf32Supported(p)) throw Error("tf32 conv: unsupported layer shape");
    Tf32Plan* plan = new Tf32Plan();
    Tf32Args& a = plan->args;
    a = Tf32Args{};
    a.p = p;
    a.bn = pickBn(p.npad);
    a.cchunks = p.cin / kKC;
    a.kblocks = p.ntaps * a.cchunks;
    long long best = -1;
    for (int bw = 8; bw <= 128; bw *= 2) {  // 128-pixel tile with the least padding
        const int bh = 128 / bw;
        const long long cover = (long long)((p.gx + bw - 1) / bw) * bw * ((p.gy + bh - 1) / bh) * bh;
        if (best < 0 || cover < best) { best = cover; a.bw = bw; a.bh = bh; }
    }
    while ((1 << a.bwShift) < a.bw) ++a.bwShift;
    a.tilesX = (p.gx + a.bw - 1) / a.bw;
    a.tilesY = (p.gy + a.bh - 1) / a.bh;
    a.tilesN = p.npad / a.bn;
    a.totalTiles = a.tilesX * a.tilesY * a.tilesN * p.gn;
    a.bytesA = 128u * kKC * 4u;
    a.bytesB = (uint32_t)a.bn * kKC * 4u;
    const size_t stageBytes = a.bytesA + a.bytesB;
    const size_t avail = kSmemLimit - 1024 - kHeaderBytes;
    a.stages = (int)std::min<size_t>(kMaxStages, avail / stageBytes);
    if (a.stages < 2) { delete plan; throw Error("tf32 conv: tile does not fit in shared memory"); }
    uint32_t cols = 32;
    while (cols < (uint32_t)(2 * a.bn)) cols *= 2;
    a.tmemCols = cols;
    a.idesc = instrDescTf32(128, a.bn);
    a.descHi = (1024u >> 4) | (1u << 14) | (2u << 29);  // SBO = 8 rows x 128 B, version 1, 128-byte swizzle
    try {
        {
            const long long dims[5] = {p.dimc, p.dimx, p.dimz, p.dimy, p.gn};
            const long long st[4] = {p.sx, p.sz, p.sy, p.sn};
            const int box[5] = {kKC, a.bw, 1, a.bh, 1};
            encodeF32(&a.tmA, 5, p.in, dims, st, box, "A");
        }
        {
            const bool perImage = p.w_img_stride != 0;  // SE scale folded into per-image weights
            const long long dims[3] = {p.ktot, p.npad, perImage ? p.gn : 1};
            const long long st[2] = {p.ktot, perImage ? p.w_img_stride : (long long)p.npad * p.ktot};
            const int box[3] = {kKC, a.bn, 1};
            encodeF32(&a.tmB, 3, p.w, dims, st, box, "weights");
        }
        static bool attrSet[64] = {};  // per device
        int dev = 0;
        cudaGetDevice(&dev);
        if (dev < 0 || dev >= 64) dev = 0;
        if (!attrSet[dev]) {
            checkCuda(cudaFuncSetAttribute(conv_tf32_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSmemLimit));
            attrSet[dev] = true;
        }
        int sms = 0;
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
        plan->grid = std::min(a.totalTiles, std::max(sms, 1));
    } catch (...) {
        delete plan;
        throw;
    }
    plan->smem = 1024 + kHeaderBytes + (size_t)a.stages * stageBytes;
    return plan;
}

void tf32DestroyPlan(Tf32Plan* plan) { delete plan; }

const char* tf32Describe(const Tf32Plan* plan, char* buf, int cap) {
    const Tf32Args& a = plan->args;
    std::snprintf(buf, cap, "igemm-tf32 bn=%d kc=%d tile=%dx%d stages=%d grid=%d smem=%zu", a.bn, kKC, a.bh, a.bw, a.stages, plan->grid, plan->smem);
    return buf;
}

void tf32Launch(const Tf32Plan* plan, cudaStream_t s, float* outOverride, int nImages) {
    if (plan->grid <= 0) return;
    const bool fewer = nImages > 0 && nImages < plan->args.p.gn;  // last, partially filled batch: skip the padding slots
    const bool redirect = outOverride && outOverride != plan->args.p.out;
    if (!fewer && !redirect) {
        checkCuda(launchPdl(conv_tf32_kernel, dim3(plan->grid), dim3(kThreads), plan->smem, s, plan->args));
        return;
    }
    Tf32Args local = plan->args;  // only the epilogue's destination / the image count change; the tensor maps stay valid
    if (redirect) local.p.out = outOverride;
    if (fewer) {
        local.totalTiles = local.totalTiles / local.p.gn * nImages;
        local.p.gn = nImages;
    }
    checkCuda(launchPdl(conv_tf32_kernel, dim3(std::min(plan->grid, std::max(local.totalTiles, 1))), dim3(kThreads), plan->smem, s, local));
}

void launchConvFirstF32(const ConvParamsF32& p, cudaStream_t s) {
    if (p.cin != 4 || p.ktot != 36 || p.npad != 32 || p.ntaps != 9 || p.mode != EPI_STORE || p.out_c != 32 || p.sx != 4 || p.w_img_stride)
        throw Error("fp32 first layer: unsupported layer shape");
    if (p.gn <= 0) return;
    dim3 grid((p.gx * p.gy + 127) / 128, p.gn);
    conv_first_f32_kernel<<<grid, 128, 0, s>>>(p);
}

}  // namespace w2x
