// ONNX import + kernel-native weight packing ("build" in the B200 engine).
// Replaces nvonnxparser::parseFromFile + buildSerializedNetwork (/root/reference/src/tensorrt/img2img_build.cpp:87-147):
// instead of a TensorRT plan the artefact is a flat file of fp16 (tf32 packs: fp32) GEMM-operand matrices laid out exactly as
// the tcgen05 implicit-GEMM kernels consume them.
#pragma once
#include <cstdint>
#include <cstring>
#include <string>
#include <vector>

namespace w2x {

// ---- minimal ONNX view -----------------------------------------------------------------------------
struct OnnxTensor {
    std::string name;
    std::vector<int64_t> dims;
    std::vector<float> data;  // FLOAT / FLOAT16 / DOUBLE initialisers widened to f32; INT64 left empty
    std::vector<int64_t> idata;
};
struct OnnxNode {
    std::string op, name;
    std::vector<std::string> inputs, outputs;
    std::vector<int64_t> kernel_shape, strides, pads, dilations, axes;
    int64_t group = 1, transA = 0, transB = 0;
    std::string auto_pad;
    float epsilon = 1e-5f;  // LayerNormalization
    float alpha = 0.01f;    // LeakyRelu (ONNX default) / Gemm
    bool hasMin = false, hasMax = false;  // Clip (opset < 11 carries the bounds as attributes)
    float minv = 0.f, maxv = 0.f;
};
struct OnnxGraph {
    std::vector<OnnxNode> nodes;
    std::vector<OnnxTensor> initializers;
    const OnnxTensor* find(const std::string& name) const;
};
OnnxGraph parseOnnx(const std::vector<uint8_t>& blob);

// ---- packed model ----------------------------------------------------------------------------------
enum LayerKind : uint32_t {
    L_CONV3 = 0,  // 3x3 valid stride-1 conv:            B[npad][9*cin],  k = (ky*3+kx)*cin + ci
    L_DOWN2 = 1,  // 2x2 stride-2 conv:                  B[npad][4*cin],  k = (dy*2+dx)*cin + ci
    L_UP2 = 2,    // ConvTranspose 2x2 stride 2:         B[4*cout][cin],  n = (dy*2+dx)*cout + co
    L_UP4 = 3,    // ConvTranspose 4x4 stride 2 pad 3 as a 2x2 window conv with 4 output phases:
                  //                                     B[16][4*cin],    n = (py*2+px)*4 + co,  k = (wy*2+wx)*cin + ci,
                  //                                     tap (ky,kx) = (2+py-2*wy, 2+px-2*wx)
    // SwinUNet records
    L_LINEAR = 4,  // token-wise Linear (ONNX MatMul [K,N] + Add):  B[N][K], bias[N]
    L_LN = 5,      // LayerNorm over channels: gamma / beta (fp32), eps
    L_ATTN = 6,    // window attention: relative position bias relpos[heads][n][n] (fp32), n = window^2
    L_UPLIN = 7,   // PatchUp = Linear(cin -> 4*cout) + pixel_shuffle(2): rows permuted to n = (i*2+j)*cout + c
    L_TOIMG = 8,   // ToImage = Linear(cin -> 3*s*s) + pixel_shuffle(s): B[16][cin], n = (i*2+j)*4 + c  (s = 1: n = c)
};

enum Arch : uint32_t { ARCH_CUNET = 1, ARCH_UPCUNET = 2, ARCH_SWINUNET = 3 };

struct PackedLayer {
    std::string name;
    uint32_t kind = 0;
    uint32_t cin = 0;    // channels per tap as stored (3 padded to 4)
    uint32_t cout = 0;   // real output channels
    uint32_t npad = 0;   // GEMM N (rows of B)
    uint32_t ktot = 0;   // GEMM K (= taps * cin)
    uint32_t taps = 0;
    uint32_t se_r = 0;   // squeeze/excite hidden width (0 = no SE after this layer)
    std::vector<uint16_t> w;     // fp16 bits, [npad][ktot] K-major (fp16 packs)
    std::vector<float> wf;       // the same as fp32 rounded to nearest TF32 (tf32 packs; w is then empty)
    std::vector<float> bias;     // [npad]
    std::vector<float> se_w1, se_b1, se_w2, se_b2;  // [r][c], [r], [c][r], [c]
    // SwinUNet
    uint32_t heads = 0, window = 0, upscale = 0;     // L_ATTN: heads, window; L_TOIMG: pixel-shuffle factor
    float eps = 0.f;                                 // L_LN
    std::vector<float> gamma, beta, relpos;          // L_LN: [c], [c];  L_ATTN: [heads][n][n]
    size_t weightCount() const { return w.empty() ? wf.size() : w.size(); }
};

struct PackedModel {
    uint32_t arch = 0, scale = 0, offset = 0, precision = 1;
    uint32_t dim = 0;  // SwinUNet base width C
    std::vector<PackedLayer> layers;
};

bool isSwinGraph(const OnnxGraph& g);
PackedModel packFromOnnx(const OnnxGraph& g, int precision);  // precision W2X_PRECISION_TF32: fp32 weights (PackedLayer::wf), cunet only
// PatchUp (L_UPLIN: rows q0 * cout + c, q0 = dy * 2 + dx) followed by ToImage with pixel shuffle 2 (L_TOIMG: rows q1 * 4 + c3) and nothing in
// between is one linear map with a pixel shuffle of 4: w [64][K] fp16 bits (row (oy * 4 + ox) * 4 + c3, oy = 2 dy + ey, ox = 2 dx + ex; rows with
// c3 = 3 are zero), b [64].  Composed in double precision from the packed fp16 weights, rounded to fp16 once.
void composeUpToImage(const PackedLayer& up, const PackedLayer& toImage, std::vector<uint16_t>& w, std::vector<float>& b);
std::vector<uint8_t> serializePack(const PackedModel& m);
PackedModel deserializePack(const std::vector<uint8_t>& blob);

uint16_t floatToHalfBits(float f);
float halfBitsToFloat(uint16_t h);

#ifdef __CUDACC__
#define W2X_HOST_DEVICE __host__ __device__
#else
#define W2X_HOST_DEVICE
#endif
// round to nearest even TF32 (8-bit exponent, 10-bit mantissa: the low 13 bits of the fp32 pattern cleared); inf / nan unchanged
inline W2X_HOST_DEVICE float roundToTf32(float f) {
#ifdef __CUDA_ARCH__
    uint32_t u = __float_as_uint(f);
#else
    uint32_t u;
    std::memcpy(&u, &f, 4);
#endif
    if ((u & 0x7f800000u) != 0x7f800000u) u = (u + 0xfffu + ((u >> 13) & 1u)) & 0xffffe000u;
#ifdef __CUDA_ARCH__
    return __uint_as_float(u);
#else
    std::memcpy(&f, &u, 4);
    return f;
#endif
}

}  // namespace w2x
