// Engine: the B200-native replacement for trt::Img2Img (/root/reference/src/tensorrt/img2img.h:14-50).
// Owns the packed model in HBM, all activation/tile workspaces, streams and events.
#pragma once
#include <cuda_fp16.h>
#include <cuda_runtime.h>

#include <cstring>
#include <string>
#include <vector>

#include "hostutil.h"
#include "kernels/conv_params.h"
#include "model_pack.h"

namespace w2x {

#define W2X_CUDA(expr)                                                                                  \
    do {                                                                                                \
        cudaError_t _e = (expr);                                                                        \
        if (_e != cudaSuccess) throw ::w2x::Error(std::string(#expr) + ": " + cudaGetErrorString(_e)); \
    } while (0)

// Activation tensor NHWC [n][h][w][c].  Its elements are the engine's (Engine::elemBytes): fp16, or fp32 in a tf32 engine, where the
// pointer (like every activation / weight pointer of the plan and of ConvParams) is nominal and the kernels read it as float (asF32).
struct Act {
    __half* p = nullptr;
    int n = 0, h = 0, w = 0, c = 0;
    size_t elems() const { return (size_t)n * h * w * c; }
};

enum ConvImpl { IMPL_DIRECT = 0, IMPL_FIRST = 1, IMPL_IGEMM = 2, IMPL_LAYERNORM = 3, IMPL_ATTENTION = 4, IMPL_HEAD = 5, IMPL_SKIP = 6, IMPL_SWIN_MLP = 7, IMPL_SWIN_ATTN = 8,
                IMPL_TF32 = 9, IMPL_FIRST_F32 = 10 };

// the plan's ConvParams of a tf32 engine, as the fp32 kernels take them (same layout; the pointers address fp32 data)
inline ConvParamsF32 asF32(const ConvParams& p) {
    static_assert(sizeof(ConvParams) == sizeof(ConvParamsF32), "ConvParamsT layouts differ");
    ConvParamsF32 q;
    std::memcpy(static_cast<void*>(&q), &p, sizeof q);
    return q;
}

struct LayerExec {
    std::string name;
    ConvParams p{};
    int impl = IMPL_DIRECT;
    IgemmPlan* plan = nullptr;
    Tf32Plan* tf32 = nullptr;  // IMPL_TF32
    HeadPlan* head = nullptr;  // IMPL_HEAD
    SwinMlpPlan* mlp = nullptr;  // IMPL_SWIN_MLP: LayerNorm + fc1 + GELU + fc2 + residual in one kernel (the two preceding layers are IMPL_SKIP)
    SwinAttnPlan* attn = nullptr;  // IMPL_SWIN_ATTN: LayerNorm + QKV + window attention + proj + residual in one kernel (three preceding layers are IMPL_SKIP)
    double flops = 0;  // algorithmic 2*MAC for ONE tile
    bool isFinal = false;
    // squeeze/excite applied to p.out after the conv
    int seR = 0;
    const float *seW1 = nullptr, *seB1 = nullptr, *seW2 = nullptr, *seB2 = nullptr;
    long long* sePartial = nullptr;  // [batch][C] exact fixed-point channel sums (2^10 scale, kSeFixedScale)
    float* seScale = nullptr;
    int seBlocks = 0;
    struct FoldJob { const void* w; void* wOut; int npad, ktot, cin; };  // engine element type
    std::vector<FoldJob> foldJobs;  // consumers that take this layer's SE scale through per-image weights
    bool seFused = false;        // squeeze sums come from the conv epilogue (ConvParams::se_sum)
    size_t sePartialBytes = 0;
    // SwinUNet token ops (IMPL_LAYERNORM / IMPL_ATTENTION)
    const __half* tokIn = nullptr;
    __half* tokOut = nullptr;
    int tokN = 0, tokH = 0, tokW = 0, tokC = 0, heads = 0, window = 0, shift = 0;
    const float *gamma = nullptr, *beta = nullptr, *relpos = nullptr;
    float eps = 0.f;
};

// Builders for the implicit-GEMM views (shared with the self-test).
ConvParams makeConv3Params(const Act& in, const Act& out, const __half* w, const float* bias, int npad, int mode, float slope, int storeC);
ConvParams makeDown2Params(const Act& in, const Act& out, const __half* w, const float* bias, int npad, float slope);
ConvParams makeUp2Params(const Act& in, const Act& out, const __half* w, const float* bias, int cout, float slope, const Act* skip, int skipOff);
ConvParams makeUp4Params(const Act& in, const Act& out, const __half* w, const float* bias);

class Engine {
public:
    Engine();
    ~Engine();

    bool build(const std::string& onnxPath, const w2x_build_config& cfg);
    bool load(const std::string& onnxPath, const w2x_render_config& cfg);
    bool render(const uint8_t* src, int w, int h, size_t srcStride, uint8_t* dst, size_t dstStride);
    bool renderDevice(const uint8_t* dSrc, int w, int h, size_t srcStride, uint8_t* dDst, size_t dstStride);
    // BGRA host buffers (w x h, pitch >= 4w) -> BGRA (w*scale x h*scale, pitch >= 4*w*scale), synchronous like render: the B, G, R of
    // the colour-bled frame through the render pipeline, the alpha plane as a second model pass in the same batches (none when opaque)
    bool renderBgra(const uint8_t* src, int w, int h, size_t srcStride, uint8_t* dst, size_t dstStride);
    int submit(const uint8_t* src, int w, int h, size_t srcStride, uint8_t* dst, size_t dstStride);
    bool wait(int ticket);
    // one image sharded over several engines (one per GPU) by bands of tile rows, seam rows exchanged peer-to-peer
    static bool renderBanded(Engine* const* engines, int count, const uint8_t* src, int w, int h, size_t srcStride, uint8_t* dst, size_t dstStride);
    bool sync();
    bool infer(const float* inNchw, int n, float* outNchw);
    int profileLayers(int repeats, char (*names)[48], float* ms, double* flops, int cap);

    void setMessageCallback(w2x_message_cb cb, void* user) { msgCb = cb; msgUser = user; }
    void setProgressCallback(w2x_progress_cb cb, void* user) { progCb = cb; progUser = user; }
    const char* lastError() const { return lastErr.c_str(); }
    int outputTile() const { return outTile; }
    long long launchCount() const { return launches; }
    double flopsPerTile() const;
    int lastStageMs(float* out, int n);
    int layerKernel(int index, char* buf, int cap) const;
    bool timerMark(int idx, int which);
    float timerElapsedMs(int i0, int i1);
    int device() const { return cfg.deviceId; }
    bool loaded() const { return isLoaded; }

    void log(int severity, const std::string& msg, const char* func, int line);

private:
    void unload();
    void buildPlan();
    void uploadAsync(void* dst, const void* src, size_t bytes);
    void buildPlanCunet();
    void buildPlanSwin();
    void launchLayer(LayerExec& L, cudaStream_t s, void* outOverride, int nImages, const void* inOverride = nullptr);
    void runModel(cudaStream_t s, void* finalOut, int nImages = 0, const void* inTiles = nullptr);
    void launchSe(const LayerExec& L, int nImages, cudaStream_t s);  // squeeze (unless fused) -> excite -> scale or fold into the consumers
    bool tf32() const { return elemBytes == 4; }
    // element `i` of an activation / tile buffer of this engine's element type
    void* elemAt(void* base, size_t i) const { return static_cast<uint8_t*>(base) + i * elemBytes; }
    void unpackTiles(const uint8_t* src, int w, int h, size_t pitch, const TileSlot* slots, int n, void* out, cudaStream_t s, int pixelBytes = 3);
    void ttaReduce(const void* outs, int tiles, float* mean, cudaStream_t s);
    bool frameWideUnpack() const;
    // passes: 1 = the colour tiles, 2 = the colour tiles followed by the alpha tiles of a BGRA frame (renderBgra)
    void ensureFrameBuffers(int w, int h, int passes = 1);
    struct RowBand { int y0, y1, batch; };             // output rows [y0, y1) are final once batch `batch` has run (row-major tile order)
    struct BandDone { int y0, y1; cudaEvent_t ev; };   // ... and have been stitched when `ev` fires
    // bands != nullptr (and no TTA): stitch progressively, one launch per finished tile row, and report the bands instead of one stitch at the end
    // pixelBytes 4: packed BGRA frames (dSrcPitch = 4w): alpha scan, colour bleed and alpha pass as the frame needs them; no bands
    void renderOnStream(const uint8_t* dSrc, int w, int h, size_t srcPitch, uint8_t* dDst, size_t dstPitch, cudaStream_t s, bool timed,
                        std::vector<BandDone>* bands = nullptr, int pixelBytes = 3);
    void* dalloc(size_t bytes);
    Act allocAct(int h, int w, int c);

    w2x_message_cb msgCb = nullptr;
    void* msgUser = nullptr;
    w2x_progress_cb progCb = nullptr;
    void* progUser = nullptr;
    std::string lastErr;

    bool isLoaded = false;
    w2x_render_config cfg{};
    PackedModel model;
    int tile = 0, outTile = 0, scale = 1, batch = 1;
    size_t elemBytes = 2;            // activations, weights and model outputs: 2 (fp16) or 4 (fp32, --precision tf32)
    bool useDirect = false;
    bool debugSync = false;      // W2X_DEBUG_SYNC: synchronise + check after every layer (names the failing kernel)

    std::vector<void*> allocs;       // freed in unload()
    std::vector<__half*> dW;         // per layer (engine element type)
    std::vector<float*> dBias;
    std::vector<LayerExec> layers;
    Act actIn;                       // [batch][tile][tile][4]
    Act actOut;                      // final layer output view (pointer overridden per batch)
    cudaStream_t stream = nullptr, h2dStream = nullptr, d2hStream = nullptr;
    long long launches = 0;

    // frame-level state
    int frameW = 0, frameH = 0, framePasses = 1;
    TileGrid grid;
    int stepCount = 0, batchCount = 0;
    TileSlot* dSlots = nullptr;
    int* dTileMap = nullptr;                     // slot of reference tile ti (row-major processing order without TTA)
    size_t tileMapCap = 0;
    std::vector<RowBand> rowBands;
    std::vector<cudaEvent_t> bandEv;
    size_t slotCap = 0;
    void* dUnpacked = nullptr;       // [steps][tile][tile][4] engine elements: every tile of the frame, unpacked by one launch
    size_t unpackedCap = 0;
    void* dTileOut = nullptr;        // [steps][outT][outT][4] engine elements
    size_t tileOutCap = 0;
    float* dTtaMean = nullptr;       // [tiles][outT][outT][4] f32 (TTA only)
    size_t ttaCap = 0;
    float *dRampX = nullptr, *dRampY = nullptr;
    int rampXLen = -1, rampYLen = -1;
    // host-buffer paths
    uint8_t *dFrameIn = nullptr, *dFrameOut = nullptr;
    size_t frameInCap = 0, frameOutCap = 0;
    // BGRA frames: alpha-scan flags (2 ints) and the two ping-pong buffers of the colour bleed
    int* dAlphaFlags = nullptr;
    uint8_t* dBleed[2] = {nullptr, nullptr};
    size_t bleedCap = 0;
    // pipelined submit
    static constexpr int kSlots = 3;
    struct PipeSlot {
        uint8_t *dIn = nullptr, *dOut = nullptr;
        size_t inCap = 0, outCap = 0;
        cudaEvent_t evH2D = nullptr, evComp = nullptr, evDone = nullptr;
        bool busy = false;
    } pipe[kSlots];
    int nextTicket = 0;
    // stage timing
    std::vector<cudaEvent_t> evPool;
    int evUsed = 0;
    struct StageSpan { int kind, e0, e1; };
    std::vector<StageSpan> spans;
    cudaEvent_t nextEvent();
    cudaEvent_t timerEv[16] = {};
    // row-band mode
    void* dBandTiles = nullptr;
    size_t bandTilesCap = 0;
    int* dBandMap = nullptr;
    size_t bandMapCap = 0;
    TileSlot* dBandSlots = nullptr;
    size_t bandSlotCap = 0;
    cudaEvent_t evBandModel = nullptr;
    float* dBandMean = nullptr;                  // --tta in row-band mode: [own tiles + received seam row][outT][outT][4] f32
    size_t bandMeanCap = 0;
    std::vector<TileSlot> bandSlotsHost;         // staging of the asynchronous uploads (must outlive them)
    std::vector<int> bandMapHost;
};

// Single-layer test hooks, see include/w2x_dev.h.  impl: 0 = the kernel the planner picks, 1 = head kernel, 2 = scalar reference.
void runConvLayer(int device, int kind, int impl, int n, int h, int w, int cin, int cout, const uint16_t* in, const uint16_t* wPacked,
                  const float* bias, const uint16_t* skip, uint16_t* out);
// the same layer kinds through the tf32 kernel: fp32 NHWC tensors and fp32 packed weights
void runConvLayerF32(int device, int kind, int n, int h, int w, int cin, int cout, const float* in, const float* wPacked, const float* bias,
                     const float* skip, float* out);
double selftestConv(int device, int kind, int n, int h, int w, int cin, int cout, unsigned seed);

}  // namespace w2x
