// Engine: the B200-native replacement for trt::Img2Img (/root/reference/src/tensorrt/img2img.h:14-50).
// Owns the packed model in HBM, all activation/tile workspaces, streams and events.
#pragma once
#include <cuda_fp16.h>
#include <cuda_runtime.h>

#include <array>
#include <cstring>
#include <optional>
#include <string>
#include <utility>
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

// Device memory with one owner, freed with it.
class DeviceBuffer {
public:
    DeviceBuffer() = default;
    explicit DeviceBuffer(size_t bytes) { ensure(bytes); }
    DeviceBuffer(DeviceBuffer&& o) noexcept : p(std::exchange(o.p, nullptr)), cap(std::exchange(o.cap, 0)) {}
    DeviceBuffer& operator=(DeviceBuffer&& o) noexcept {
        if (this != &o) {
            release();
            p = std::exchange(o.p, nullptr);
            cap = std::exchange(o.cap, 0);
        }
        return *this;
    }
    ~DeviceBuffer() { release(); }

    // At least `bytes`; true when it reallocated (the contents are then undefined).  The old memory is released first, so a failed
    // allocation leaves the buffer empty rather than a stale capacity over a freed pointer.
    bool ensure(size_t bytes) {
        if (bytes <= cap) return false;
        release();
        W2X_CUDA(cudaMalloc(&p, bytes));
        cap = bytes;
        return true;
    }
    template <class T = void> T* get() const { return static_cast<T*>(p); }

private:
    void release() {
        if (p) cudaFree(p);
        p = nullptr;
        cap = 0;
    }
    void* p = nullptr;
    size_t cap = 0;
};

// A CUDA event with one owner, created with `flags` on first use and destroyed with it.
class CudaEvent {
public:
    CudaEvent() = default;
    explicit CudaEvent(unsigned flags) : flags(flags) {}
    CudaEvent(CudaEvent&& o) noexcept : e(std::exchange(o.e, nullptr)), flags(o.flags) {}
    CudaEvent& operator=(CudaEvent&& o) noexcept {
        if (this != &o) {
            if (e) cudaEventDestroy(e);
            e = std::exchange(o.e, nullptr);
            flags = o.flags;
        }
        return *this;
    }
    ~CudaEvent() {
        if (e) cudaEventDestroy(e);
    }

    cudaEvent_t get() {
        if (!e) W2X_CUDA(cudaEventCreateWithFlags(&e, flags));
        return e;
    }
    bool created() const { return e != nullptr; }

private:
    cudaEvent_t e = nullptr;
    unsigned flags = cudaEventDefault;
};

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

// One frame through the engine: src (w x h pixels of `format`) -> dst (the canvas, w*scale x h*scale, or `out` when set), strides in
// bytes, at least the pixel size times the row's width.  The formats (include/w2x.h):
//  - Bgr8: render's frames.  `out` reduces the canvas by an antialiased bicubic resample (w2x_render_resized), 1x1 .. the canvas; the
//    canvas size itself is render, byte for byte.
//  - Bgra8: the B, G, R of the colour-bled frame through the render pipeline, the alpha plane as a second model pass in the same
//    batches (none when opaque).  Synchronous host frames only.
//  - Bgr16: u16 samples, even strides and pointers; the input is scaled by f32(1/65535), the output is saturate(rint(65535 v)) of
//    render's fp32 canvas.  Tiles, batches and blending are render's.
// Engine::checkFrame decides which frames each entry point takes.
struct Frame {
    struct Size { int w, h; };
    PixelFormat format = PixelFormat::Bgr8;
    const void* src = nullptr;
    int w = 0, h = 0;
    size_t srcStride = 0;
    void* dst = nullptr;
    size_t dstStride = 0;
    std::optional<Size> out;   // the resized output size (Bgr8 only); unset: the canvas
};

class Engine {
public:
    Engine();
    ~Engine();
    Engine(const Engine&) = delete;
    Engine& operator=(const Engine&) = delete;

    bool build(const std::string& onnxPath, const w2x_build_config& cfg);
    bool load(const std::string& onnxPath, const w2x_render_config& cfg);
    // host frames, synchronous: dst is complete on return
    bool render(const Frame& f);
    // host frames through the copy / compute / copy pipeline (kSlots frames in flight): a ticket for wait, or -1
    int submit(const Frame& f);
    // device frames (Bgr8, canvas size) enqueued on the engine's stream, not synchronised
    bool renderDevice(const Frame& f);
    bool wait(int ticket);
    // one host frame (Bgr8, canvas size) sharded over several engines (one per GPU) by bands of tile rows, seam rows exchanged
    // peer-to-peer
    static bool renderBanded(Engine* const* engines, int count, const Frame& f);
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
    // test hook w2x_layer_tensor (include/w2x_dev.h): a read-only copy of one tensor of a CUNet plan layer
    long long layerTensor(int index, int which, void* dst, size_t cap, int* dims);
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
    void unpackTiles(const uint8_t* src, int w, int h, size_t pitch, const TileSlot* slots, int n, void* out, cudaStream_t s, PixelFormat format);
    void ttaReduce(const void* outs, int tiles, float* mean, cudaStream_t s);
    bool frameWideUnpack() const;
    // passes: 1 = the colour tiles, 2 = the colour tiles followed by the alpha tiles of a Bgra8 frame
    void ensureFrameBuffers(int w, int h, int passes = 1);
    struct RowBand { int y0, y1, batch; };             // output rows [y0, y1) are final once batch `batch` has run (row-major tile order)
    struct BandDone { int y0, y1; cudaEvent_t ev; };   // ... and have been stitched when `ev` fires
    // The entry points that take a frame, and every refusal they make (throws Error): no engine, null pointers, sizes, strides,
    // alignment, and the formats and output sizes each one takes.
    enum class FramePath { Render, Submit, Device, Banded };
    void checkFrame(const Frame& f, FramePath path) const;
    Frame::Size outputSize(const Frame& f) const { return f.out ? *f.out : Frame::Size{f.w * scale, f.h * scale}; }
    // d: a checked frame whose src and dst are on this device
    // bands != nullptr (and no TTA): stitch progressively, one launch per finished tile row, and report the bands instead of one stitch at the end
    // Bgra8: alpha scan, colour bleed and alpha pass as the frame needs them; no bands
    // d.out other than the canvas: stitch into resize.canvas, then resample into d.dst; with bands, the bands are output rows of d.dst
    // Bgr16: the tiles, batches and bands are those of Bgr8 frames
    void renderOnStream(const Frame& d, cudaStream_t s, bool timed, std::vector<BandDone>* bands = nullptr);
    void ensureResize(int cw, int ch, int dw, int dh);
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

    std::vector<DeviceBuffer> allocs;  // plan lifetime: weights, activations, SE scratch
    std::vector<__half*> dW;         // per layer (engine element type)
    std::vector<float*> dBias;
    std::vector<LayerExec> layers;
    Act actIn;                       // [batch][tile][tile][4]
    Act actOut;                      // final layer output view (pointer overridden per batch)
    cudaStream_t stream = nullptr, h2dStream = nullptr, d2hStream = nullptr;
    long long launches = 0;

    // Each group below is reset by one assignment in unload().
    // frame cache (ensureFrameBuffers), valid for the frame key w x h, passes; w == 0: no frame
    struct FrameCache {
        int w = 0, h = 0, passes = 1;
        TileGrid grid;
        int batchCount = 0;
        std::vector<RowBand> rowBands;
        std::vector<CudaEvent> bandEv;   // render's per-band events (cudaEventDisableTiming), reused frame after frame
        DeviceBuffer slots;              // TileSlot [steps]
        DeviceBuffer tileMap;            // int [tiles]: slot of reference tile ti (row-major processing order without TTA)
        DeviceBuffer unpacked;           // [steps][tile][tile][4] engine elements: every tile of the frame, unpacked by one launch
        DeviceBuffer tileOut;            // [steps][outT][outT][4] engine elements
        DeviceBuffer ttaMean;            // [tiles][outT][outT][4] f32 (TTA only)
        DeviceBuffer rampX, rampY;       // blend ramps of rampXLen / rampYLen entries
        int rampXLen = -1, rampYLen = -1;
    } fc;
    // host-buffer paths: the frame on the device (render, renderBanded), sized in bytes
    struct HostStaging { DeviceBuffer in, out; } staging;
    // BGRA frames: alpha-scan flags (2 ints) and the two ping-pong buffers of the colour bleed
    struct BgraScratch { DeviceBuffer flags, bleed[2]; } bgra;
    // resized frames (ensureResize), valid for the key canvas cw x ch -> dw x dh; cw == 0: none
    struct ResizeState {
        int cw = 0, ch = 0, dw = 0, dh = 0;
        DeviceBuffer canvas;             // u8 BGR [ch][cw][3], the stitched frame
        DeviceBuffer tmp;                // f32 [ch][dw][3], the horizontal pass
        DeviceBuffer tables[2];          // x, y: int first[n_out], int count[n_out], float w[n_out][taps]
        ResampleTable tx{}, ty{};
        std::vector<int> rowEnd;         // output row i reads canvas rows below rowEnd[i] (non-decreasing)
    } resize;
    // pipelined submit
    static constexpr int kSlots = 3;
    struct PipeSlot {
        DeviceBuffer in, out;            // bytes: u8 and u16 frames share them
        CudaEvent evH2D{cudaEventDisableTiming}, evComp{cudaEventDisableTiming}, evDone{cudaEventDisableTiming};
        bool busy = false;
    };
    std::array<PipeSlot, kSlots> pipe;
    int nextTicket = 0;
    // stage timing (renderOnStream's spans) and the caller's timer marks
    struct StageSpan { int kind, e0, e1; };
    struct Timing {
        std::vector<CudaEvent> pool;
        int used = 0;
        std::vector<StageSpan> spans;
        CudaEvent marks[16];
    } timing;
    cudaEvent_t nextEvent();
    // row-band mode
    struct BandState {
        DeviceBuffer tiles;              // engine elements: own model outputs (+ the received seam row without TTA)
        DeviceBuffer mean;               // --tta: [own tiles + received seam row][outT][outT][4] f32
        DeviceBuffer map;                // int [tiles]
        DeviceBuffer slots;              // TileSlot [steps]
        CudaEvent evModel{cudaEventDisableTiming};
        std::vector<TileSlot> slotsHost;  // staging of the asynchronous uploads (must outlive them)
        std::vector<int> mapHost;
    } band;
};

// Single-layer test hooks, see include/w2x_dev.h.  impl: 0 = the kernel the planner picks, 1 = head kernel, 2 = scalar reference.
void runConvLayer(int device, int kind, int impl, int n, int h, int w, int cin, int cout, const uint16_t* in, const uint16_t* wPacked,
                  const float* bias, const uint16_t* skip, uint16_t* out);
// the same layer kinds through the tf32 kernel: fp32 NHWC tensors and fp32 packed weights
void runConvLayerF32(int device, int kind, int n, int h, int w, int cin, int cout, const float* in, const float* wPacked, const float* bias,
                     const float* skip, float* out);
double selftestConv(int device, int kind, int n, int h, int w, int cin, int cout, unsigned seed);

}  // namespace w2x
