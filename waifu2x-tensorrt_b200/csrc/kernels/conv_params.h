// Shared description of one implicit-GEMM convolution launch (host + device), and the fused epilogues.
//
// Every dense layer of the model hot path (SURVEY 2.2 / 8a row a17) is expressed as
//     D[pixel, n] = sum_{tap, c} A(pixel + tap, c) * B[n, tap*cin + c]
// over a 5-D strided view (c, x, z, y, img) of an NHWC fp16 activation, followed by one of four epilogues that
// fuse bias + LeakyReLU(0.1), depth-to-space (ConvTranspose), the cropped skip-add, and the final add + clamp.
#pragma once
#include <cuda_fp16.h>
#include <cstdint>
#include <vector>

namespace w2x {

enum EpiMode : int {
    EPI_STORE = 0,  // out[img][y][x][0..cout) = lrelu(acc + bias)
    EPI_D2S = 1,    // ConvTranspose 2x2 s2: column (q*cout+co) -> out[img][2y+q/2][2x+q%2][co] = lrelu(acc+bias) + skip
    EPI_UP4 = 2,    // ConvTranspose 4x4 s2 p3 head: column (q*4+co) -> out[img][2y-1+q/2][2x-1+q%2][co] = acc + bias
    EPI_FINAL = 3,  // image head: out[img][y][x][0..4) = clamp(acc + bias + skip[img][y+off][x+off], 0, 1)
    EPI_TOIMG = 4,  // SwinUNet ToImage: column (q*4+c) -> out[img][s*y+q/s][s*x+q%s][c] = clamp(acc + bias, 0, 1), s = cout (1|2|4)
};
enum ActKind : int { ACT_LRELU = 0, ACT_GELU = 1 };  // ACT_LRELU with slope 1 == identity

struct ConvTap {
    int c0, dx, dz, dy;  // offsets along (c, x, z, y) of the 5-D view
};

// T is the activation / weight element type: __half for the fp16 kernels, float for the tf32 kernel (conv_tf32_sm100.cu)
template <typename T>
struct ConvParamsT {
    // A operand view (element strides; c is contiguous)
    const T* in;
    long long sx, sz, sy, sn;
    int dimc, dimx, dimz, dimy;  // view extents (for the TMA map)
    int cin;                     // channels per tap
    int ntaps;
    ConvTap tap[9];
    int is3x3;                   // plain 3x3 stride-1 valid conv on an NHWC view (eligible for the patch kernel)
    // GEMM extents
    int gx, gy, gn;  // pixel grid per image (x, y) and image count
    int npad, ktot;
    const T* w;         // B: [npad][ktot], K-major
    long long w_img_stride;  // elements between per-image copies of B (SE scale folded into the weights), 0 = shared
    const float* bias;  // [npad]
    // epilogue
    int mode;
    float slope;  // LeakyReLU negative slope; 1.0f = linear
    int act;      // ActKind (EPI_STORE only)
    T* out;
    int out_h, out_w, out_c;
    int cout;  // EPI_STORE: channels stored (4 or a multiple of 8); EPI_D2S: channels per phase
    const T* skip;
    int skip_h, skip_w, skip_c, skip_off;
    const float* skip_scale;  // optional per-(img, channel) multiplier applied to skip (SE fold), or nullptr
    long long* se_sum;        // optional [gn][npad] int64: fused SE squeeze = sum over the image of round(activation * 2^10) (kSeFixedScale),
                              // accumulated with integer atomics (exact, so the result does not depend on which CTA saw which
                              // tile or on the image's batch slot); the buffer must be zeroed before the launch
    int se_slots;             // unused (kept for ABI stability of the struct inside this library)
};
using ConvParams = ConvParamsT<__half>;
using ConvParamsF32 = ConvParamsT<float>;

#ifdef __CUDACC__

__device__ __forceinline__ float lrelu(float v, float slope) { return v > 0.f ? v : v * slope; }
// nn.GELU() (erf form): gelu(v) = v * Phi(v).  Phi(v) - 1/2 = v * Q(v^2) with a degree-9 polynomial Q fitted on |v| <= 4 (Chebyshev
// nodes; |error of gelu| <= 1.3e-5 there, fp32 Horner included); outside, v * Phi(+-4) -- a relative error of 3.3e-5 for v > 4 and an
// absolute error <= 1.3e-4 where the true value is within 1.3e-4 of zero -- all far below the fp16 resolution of the stored result.
// No MUFU: the rcp + ex2 of the Abramowitz-Stegun form made the Linear epilogues and the fused MLP kernel bound by the XU pipe
// (99.8 % busy in profiles/r02_ncu_swin_mlp.txt); this form is 14 FMA-pipe instructions.
__device__ __forceinline__ float geluErf(float v) {
    const float vn = fmaxf(v, -4.f);
    const float vc = fminf(vn, 4.f);
    const float u = vc * vc;
    float q = -4.407132645e-12f;
    q = fmaf(q, u, 4.129891984e-10f);
    q = fmaf(q, u, -1.754582968e-08f);
    q = fmaf(q, u, 4.542657450e-07f);
    q = fmaf(q, u, -8.172721209e-06f);
    q = fmaf(q, u, 1.105528936e-04f);
    q = fmaf(q, u, -1.176239806e-03f);
    q = fmaf(q, u, 9.960514493e-03f);
    q = fmaf(q, u, -6.648434699e-02f);
    q = fmaf(q, u, 3.989418149e-01f);
    return vn * fmaf(vc, q, 0.5f);
}

struct alignas(16) Half8 { __half2 a, b, c, d; };
struct alignas(8) Half4 { __half2 a, b; };

// Epilogue for 8 consecutive GEMM columns [j0, j0+8) of pixel (img, y, x); v = raw fp32 accumulators.
// The caller guarantees y < gy, x < gx, img < gn and j0 % 8 == 0.
__device__ __forceinline__ void conv_epilogue8(const ConvParams& p, int img, int y, int x, int j0, const float* v, const Half4* preSkip = nullptr) {
    float r[8];
    if (p.mode == EPI_STORE) {
        if (j0 >= p.cout) return;
        if (p.act == ACT_GELU) {
#pragma unroll
            for (int i = 0; i < 8; ++i) r[i] = geluErf(v[i] + __ldg(p.bias + j0 + i));
        } else {
#pragma unroll
            for (int i = 0; i < 8; ++i) r[i] = lrelu(v[i] + __ldg(p.bias + j0 + i), p.slope);
        }
        if (p.skip && p.cout - j0 >= 8) {  // residual add (token-wise Linear + skip of the same geometry)
            const Half8 sv = *reinterpret_cast<const Half8*>(
                p.skip + (((long long)img * p.skip_h + y + p.skip_off) * p.skip_w + x + p.skip_off) * p.skip_c + j0);
            float2 t;
            t = __half22float2(sv.a); r[0] += t.x; r[1] += t.y;
            t = __half22float2(sv.b); r[2] += t.x; r[3] += t.y;
            t = __half22float2(sv.c); r[4] += t.x; r[5] += t.y;
            t = __half22float2(sv.d); r[6] += t.x; r[7] += t.y;
        }
        __half* o = p.out + (((long long)img * p.out_h + y) * p.out_w + x) * p.out_c + j0;
        if (p.cout - j0 >= 8) {
            Half8 h{__floats2half2_rn(r[0], r[1]), __floats2half2_rn(r[2], r[3]), __floats2half2_rn(r[4], r[5]),
                    __floats2half2_rn(r[6], r[7])};
            *reinterpret_cast<Half8*>(o) = h;
        } else {
            Half4 h{__floats2half2_rn(r[0], r[1]), __floats2half2_rn(r[2], r[3])};
            *reinterpret_cast<Half4*>(o) = h;
        }
    } else if (p.mode == EPI_D2S) {
        const int q = j0 / p.cout, co = j0 - q * p.cout;
        const int oy = 2 * y + (q >> 1), ox = 2 * x + (q & 1);
#pragma unroll
        for (int i = 0; i < 8; ++i) r[i] = lrelu(v[i] + __ldg(p.bias + j0 + i), p.slope);
        if (p.skip) {
            const __half* s = p.skip + (((long long)img * p.skip_h + oy + p.skip_off) * p.skip_w + ox + p.skip_off) * p.skip_c + co;
            const Half8 sv = *reinterpret_cast<const Half8*>(s);
            float f[8];
            float2 t;
            t = __half22float2(sv.a); f[0] = t.x; f[1] = t.y;
            t = __half22float2(sv.b); f[2] = t.x; f[3] = t.y;
            t = __half22float2(sv.c); f[4] = t.x; f[5] = t.y;
            t = __half22float2(sv.d); f[6] = t.x; f[7] = t.y;
            if (p.skip_scale) {
#pragma unroll
                for (int i = 0; i < 8; ++i) f[i] *= __ldg(p.skip_scale + (long long)img * p.skip_c + co + i);
            }
#pragma unroll
            for (int i = 0; i < 8; ++i) r[i] += f[i];
        }
        __half* o = p.out + (((long long)img * p.out_h + oy) * p.out_w + ox) * p.out_c + co;
        Half8 h{__floats2half2_rn(r[0], r[1]), __floats2half2_rn(r[2], r[3]), __floats2half2_rn(r[4], r[5]),
                __floats2half2_rn(r[6], r[7])};
        *reinterpret_cast<Half8*>(o) = h;
    } else if (p.mode == EPI_UP4) {
        if (j0 >= 16) return;
#pragma unroll
        for (int hsel = 0; hsel < 2; ++hsel) {
            const int q = (j0 >> 2) + hsel;
            const int oy = 2 * y - 1 + (q >> 1), ox = 2 * x - 1 + (q & 1);
            if (oy < 0 || ox < 0 || oy >= p.out_h || ox >= p.out_w) continue;
            const float* vv = v + 4 * hsel;
            const float* bb = p.bias + j0 + 4 * hsel;
            Half4 h{__floats2half2_rn(vv[0] + __ldg(bb + 0), vv[1] + __ldg(bb + 1)),
                    __floats2half2_rn(vv[2] + __ldg(bb + 2), vv[3] + __ldg(bb + 3))};
            *reinterpret_cast<Half4*>(p.out + (((long long)img * p.out_h + oy) * p.out_w + ox) * p.out_c) = h;
        }
    } else if (p.mode == EPI_TOIMG) {
        const int s = p.cout;  // pixel-shuffle factor
        if (j0 >= 4 * s * s) return;
#pragma unroll
        for (int hsel = 0; hsel < 2; ++hsel) {
            const int q = (j0 >> 2) + hsel;
            if (q >= s * s) continue;
            const int oy = s * y + q / s, ox = s * x + q % s;
            const float* vv = v + 4 * hsel;
            const float* bb = p.bias + j0 + 4 * hsel;
            Half4 h{__floats2half2_rn(fminf(fmaxf(vv[0] + __ldg(bb + 0), 0.f), 1.f), fminf(fmaxf(vv[1] + __ldg(bb + 1), 0.f), 1.f)),
                    __floats2half2_rn(fminf(fmaxf(vv[2] + __ldg(bb + 2), 0.f), 1.f), 0.f)};
            *reinterpret_cast<Half4*>(p.out + (((long long)img * p.out_h + oy) * p.out_w + ox) * p.out_c) = h;
        }
    } else {  // EPI_FINAL
        if (j0 != 0) return;
        const Half4 sv = preSkip ? *preSkip : *reinterpret_cast<const Half4*>(
            p.skip + (((long long)img * p.skip_h + y + p.skip_off) * p.skip_w + x + p.skip_off) * p.skip_c);
        const float2 s0 = __half22float2(sv.a), s1 = __half22float2(sv.b);
        r[0] = fminf(fmaxf(v[0] + __ldg(p.bias + 0) + s0.x, 0.f), 1.f);
        r[1] = fminf(fmaxf(v[1] + __ldg(p.bias + 1) + s0.y, 0.f), 1.f);
        r[2] = fminf(fmaxf(v[2] + __ldg(p.bias + 2) + s1.x, 0.f), 1.f);
        r[3] = 0.f;
        Half4 h{__floats2half2_rn(r[0], r[1]), __floats2half2_rn(r[2], r[3])};
        *reinterpret_cast<Half4*>(p.out + (((long long)img * p.out_h + y) * p.out_w + x) * p.out_c) = h;
    }
}

#endif  // __CUDACC__

// host-side launchers (kernels/*.cu)
void launchConvDirect(const ConvParams& p, cudaStream_t s);       // scalar CUDA-core reference (tests / self-check only)
void launchConvFirst(const ConvParams& p, cudaStream_t s);        // cin=4 -> 32 first layer (mma.sync column strips)
struct HeadPlan;                                                  // image head (kernels/conv_head.cu): params + input tensor map
bool convHeadSupported(const ConvParams& p);                      // 3x3, 64 -> 3 channels, EPI_FINAL
HeadPlan* convHeadCreatePlan(const ConvParams& p);
void convHeadDestroyPlan(HeadPlan* plan);
void launchConvHead(const HeadPlan* plan, cudaStream_t s, __half* outOverride = nullptr, int nImages = 0);
void encodeActivationMap5d(void* tensorMap, const ConvParams& p, int boxX, int boxY);  // conv_igemm_sm100.cu
void encodeMatrixMap2d(void* tensorMap, const void* ptr, long long k, long long rows, int boxK, int boxRows, bool sw128);  // conv_igemm_sm100.cu
struct SwinMlpPlan;                                               // fused LN + fc1 + GELU + fc2 + residual (kernels/swin_mlp_sm100.cu)
bool swinMlpSupported(int c, int hidden);
SwinMlpPlan* swinMlpCreatePlan(__half* x, int c, const float* gamma, const float* beta, float eps, const __half* w1, const float* b1, const __half* w2, const float* b2,
                               int variant = 0);  // variant 1: stream the weights even where they would fit
void swinMlpDestroyPlan(SwinMlpPlan* plan);
void swinMlpLaunch(const SwinMlpPlan* plan, cudaStream_t s, long long tokens);
const char* swinMlpDescribe(const SwinMlpPlan* plan, char* buf, int cap);
struct SwinAttnPlan;                                              // fused LN + QKV + window attention + proj + residual (kernels/swin_attn_sm100.cu)
bool swinAttnSupported(int c, int heads, int window, int h, int w);
void swinAttnPrepare(const uint16_t* wqkv, const float* bqkv, const float* relpos, int c, int heads, std::vector<uint16_t>& wOut, std::vector<float>& bOut,
                     std::vector<float>& relOut);
bool swinAttnFusesProj(int c);                                    // c = 96: proj + residual inside the kernel (x in place); c = 192: attention output to `out`
SwinAttnPlan* swinAttnCreatePlan(__half* x, int n, int h, int w, int c, int heads, int window, int shift, const float* gamma, const float* beta, float eps,
                                 const __half* wqkvR, const float* bqkvR, const __half* wproj, const float* bproj, const float* relposR, __half* out);
void swinAttnDestroyPlan(SwinAttnPlan* plan);
void swinAttnLaunch(const SwinAttnPlan* plan, cudaStream_t s, int nImages);
const char* swinAttnDescribe(const SwinAttnPlan* plan, char* buf, int cap);
struct IgemmPlan;                                                 // opaque: tensor maps + launch geometry
IgemmPlan* igemmCreatePlan(const ConvParams& p);                  // throws w2x::Error when unsupported
void igemmDestroyPlan(IgemmPlan* plan);
bool igemmFusedFirstSupported(const ConvParams& second, const ConvParams& first);  // conv(4->32)+lrelu computed inside conv(32->64)
IgemmPlan* igemmCreatePlanFusedFirst(const ConvParams& second, const ConvParams& first);
void igemmLaunch(const IgemmPlan* plan, cudaStream_t s, __half* outOverride = nullptr, int nImages = 0, const __half* inOverride = nullptr);
void igemmSetFusedFrameInput(IgemmPlan* plan, const __half* base, long long images);
bool igemmSupported(const ConvParams& p);
const char* igemmDescribe(const IgemmPlan* plan, char* buf, int cap);
bool igemmSeFusable(const IgemmPlan* plan);  // can this layer's epilogue produce ConvParams::se_sum?
int probeUmma(int mode, int pitch, float* err9);
float probeMmaRate(int n, int iters, int sboA);
float probeMmaTiles(int tiles, int mode);  // the patch kernel's MMA schedule in isolation: cycles per MMA
int probeMmaRateStream(int n, int iters, int streamBytes, float* res);  // UMMA rate with concurrent async smem writes
float probeHmmaRate(int warps, int chains, int iters);
float probeL2Stream(int bytes, int iters);               // L2 -> SM ingest rate of a shared, L2-resident buffer (conv_direct.cu)  // legacy mma.sync issue rate (conv_direct.cu)

// SwinUNet token kernels (kernels/swin.cu)
void launchLayerNorm(const __half* x, __half* y, long long tokens, int c, const float* gamma, const float* beta, float eps, cudaStream_t s);
void launchWindowAttention(const __half* qkv, __half* out, int n, int h, int w, int c, int heads, int window, int shift,
                           const float* relpos, cudaStream_t s);

// tf32 path (kernels/conv_tf32_sm100.cu): fp32 NHWC activations and fp32 K-major weights, tcgen05 kind::tf32 MMAs, fp32 epilogues
struct Tf32Plan;                                                  // opaque: tensor maps + launch geometry
bool tf32Supported(const ConvParamsF32& p);
Tf32Plan* tf32CreatePlan(const ConvParamsF32& p);                 // throws w2x::Error when unsupported
void tf32DestroyPlan(Tf32Plan* plan);
void tf32Launch(const Tf32Plan* plan, cudaStream_t s, float* outOverride = nullptr, int nImages = 0);
const char* tf32Describe(const Tf32Plan* plan, char* buf, int cap);
void launchConvFirstF32(const ConvParamsF32& p, cudaStream_t s);  // cin=4 -> 32 first layer on the CUDA cores (fp32 FMA)
void launchScaleWeightsF32(const float* w, float* wOut, const float* scale, int nimg, int npad, int ktot, int cin, cudaStream_t s);

// squeeze/excite
constexpr float kSeFixedScale = 1024.f;  // 2^10 fixed-point resolution of the squeeze sums: 32 fp16-range values cannot overflow int32
void launchSeSqueeze(const __half* x, int n, int h, int w, int c, long long* sums, cudaStream_t s);  // sums must be zeroed
void launchSeExcite(const long long* sums, int n, int c, int r, int hw, const float* w1, const float* b1,
                    const float* w2, const float* b2, float* scale, cudaStream_t s);
void launchSeScale(__half* x, int n, int h, int w, int c, const float* scale, cudaStream_t s);
// W'[img][n][k] = W[n][k] * scale[img][k % cin]: folds an SE channel scale into the CONSUMER's weights (one copy per image)
void launchScaleWeights(const __half* w, __half* wOut, const float* scale, int nimg, int npad, int ktot, int cin, cudaStream_t s);

// tiling (kernels/tiling.cu)
// input rect origin, D4 op, valid: 0 = zero dummy slot (img2img_render.cpp:281), 1 = the frame's B, G, R bytes, kSlotAlpha = the
// alpha byte of a BGRA frame as R = G = B (the alpha pass of a Bgra8 render)
struct TileSlot { int x, y, aug, valid; };
constexpr int kSlotAlpha = 2;
// The pixel layout of a frame in and out: packed B, G, R (, A) u8 samples, or native-endian u16 B, G, R samples (2-byte aligned frame
// and pitch)
enum class PixelFormat { Bgr8, Bgra8, Bgr16 };
constexpr int bytesPerPixel(PixelFormat f) { return f == PixelFormat::Bgr8 ? 3 : f == PixelFormat::Bgra8 ? 4 : 6; }
void launchUnpack(const uint8_t* frame, int w, int h, size_t pitch, const TileSlot* slots, int nslots, int tile,
                  __half* out, cudaStream_t s, PixelFormat format);
void launchUnpack(const uint8_t* frame, int w, int h, size_t pitch, const TileSlot* slots, int nslots, int tile,
                  float* out, cudaStream_t s, PixelFormat format);  // tf32 engines: the reference's convertTo(CV_32F, 1/255) blob exactly
struct StitchParams {
    const void* tiles;   // [count][outT][outT][4] fp16 or f32
    int f32;             // element type of tiles
    int outT, nx, ny, ovx, ovy, cw, ch;
    const float* rampx;  // [ovx]
    const float* rampy;  // [ovy]
    uint8_t* dst;
    size_t pitch;
    // row-band mode (one image sharded over GPUs by tile rows): only output rows [y_begin, y_end) are produced, and tile
    // (i, j) lives at slot tile_map[i * ny + j] of `tiles` (nullptr = identity, the reference's column-major order)
    int y_begin, y_end;
    const int* tile_map;
    // the canvas: Bgr16 packs saturate(rint(65535 v)) per sample.  Bgra8 with alpha_off > 0: the alpha pass's tile of reference tile t
    // is at slot(t) + alpha_off, else alpha = 255
    PixelFormat format;
    int alpha_off;
};
// A StitchParams of the tile grid (output tile size, tile counts, blend overlaps, canvas size, blend ramps); the rest is zero: fp16
// tiles in the reference's order, a Bgr8 canvas, the whole canvas
inline StitchParams stitchGrid(int outT, int nx, int ny, int ovx, int ovy, int cw, int ch, const float* rampx, const float* rampy) {
    StitchParams p{};
    p.outT = outT; p.nx = nx; p.ny = ny; p.ovx = ovx; p.ovy = ovy;
    p.cw = cw; p.ch = ch;
    p.rampx = rampx; p.rampy = rampy;
    return p;
}
void launchStitch(const StitchParams& p, cudaStream_t s);
// BGRA frames (kernels/alpha.cu), packed w x h x 4 bytes on the device.
// flags[0] = 1 if some alpha < 255, flags[1] = 1 if some alpha == 0; flags must be zeroed
void launchAlphaScan(const uint8_t* bgra, size_t pixels, int* flags, cudaStream_t s);
// One Jacobi round of the colour bleed: a pixel is known when its alpha byte is > 0; a known pixel keeps B, G, R, an unknown one with
// n > 0 known 8-neighbours takes their per-channel mean (2 sum + n) / 2n (grow != 0) and becomes known, any other is (0, 0, 0).  The
// output alpha byte is 255 / 0 for known / unknown, or, when alphaOf != nullptr (last round), alphaOf's alpha byte.
void launchAlphaBleedRound(const uint8_t* in, uint8_t* out, int w, int h, int grow, const uint8_t* alphaOf, cudaStream_t s);
// Antialiased bicubic reduction (kernels/resample.cu): one axis table on the device, laid out as hostutil.h's ResampleAxis
struct ResampleTable {
    const int* first;    // [n_out] first input index
    const int* count;    // [n_out] taps
    const float* w;      // [n_out][taps] weights
    int taps;
};
// horizontal pass: canvas rows [y0, y1) of a u8 BGR canvas -> rows [y0, y1) of tmp, f32 [rows][dstW][3]
void launchResampleH(const uint8_t* canvas, size_t pitch, int y0, int y1, const ResampleTable& tx, int dstW, float* tmp, cudaStream_t s);
// vertical pass: output rows [i0, i1) from tmp -> u8 BGR rows of dst, rint + clamp to [0, 255]
void launchResampleV(const float* tmp, int dstW, const ResampleTable& ty, int i0, int i1, uint8_t* dst, size_t pitch, cudaStream_t s);
void launchTtaReduce(const __half* outs, int tiles, int outT, float* mean, cudaStream_t s);
void launchTtaReduce(const float* outs, int tiles, int outT, float* mean, cudaStream_t s);
// NCHW f32 <-> NHWC4 fp16 / f32 (Img2Img::infer host entry, tests)
void launchNchwToNhwc4(const float* in, int n, int t, __half* out, cudaStream_t s);
void launchNhwc4ToNchw(const __half* in, int n, int t, float* out, cudaStream_t s);
void launchNchwToNhwc4(const float* in, int n, int t, float* out, cudaStream_t s);
void launchNhwc4ToNchw(const float* in, int n, int t, float* out, cudaStream_t s);

}  // namespace w2x
