#include "engine.h"

#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <filesystem>
#include <memory>
#include <random>

namespace w2x {

namespace fs = std::filesystem;

// ------------------------------------------------------------------------------------------------
// implicit-GEMM views of the four layer kinds (see conv_params.h / model_pack.h)
// ------------------------------------------------------------------------------------------------
static void plainView(ConvParams& p, const Act& in) {
    p.in = in.p;
    p.dimc = in.c; p.dimx = in.w; p.dimz = 1; p.dimy = in.h;
    p.sx = in.c; p.sz = (long long)in.w * in.c; p.sy = (long long)in.w * in.c; p.sn = (long long)in.h * in.w * in.c;
    p.cin = in.c;
    p.gn = in.n;
}

static void setOut(ConvParams& p, const Act& out) {
    p.out = out.p; p.out_h = out.h; p.out_w = out.w; p.out_c = out.c;
}

ConvParams makeConv3Params(const Act& in, const Act& out, const __half* w, const float* bias, int npad, int mode, float slope, int storeC) {
    ConvParams p{};
    plainView(p, in);
    p.ntaps = 9;
    p.is3x3 = 1;
    for (int ky = 0; ky < 3; ++ky)
        for (int kx = 0; kx < 3; ++kx) p.tap[ky * 3 + kx] = {0, kx, 0, ky};
    p.gx = in.w - 2; p.gy = in.h - 2;
    p.npad = npad; p.ktot = 9 * in.c;
    p.w = w; p.bias = bias;
    p.mode = mode; p.slope = slope; p.cout = storeC;
    setOut(p, out);
    return p;
}

ConvParams makeDown2Params(const Act& in, const Act& out, const __half* w, const float* bias, int npad, float slope) {
    ConvParams p{};
    p.in = in.p;
    p.dimc = 2 * in.c; p.dimx = in.w / 2; p.dimz = 2; p.dimy = in.h / 2;
    p.sx = 2 * in.c; p.sz = (long long)in.w * in.c; p.sy = 2ll * in.w * in.c; p.sn = (long long)in.h * in.w * in.c;
    p.cin = in.c; p.gn = in.n;
    p.ntaps = 4;
    for (int dy = 0; dy < 2; ++dy)
        for (int dx = 0; dx < 2; ++dx) p.tap[dy * 2 + dx] = {dx * in.c, 0, dy, 0};
    p.gx = in.w / 2; p.gy = in.h / 2;
    p.npad = npad; p.ktot = 4 * in.c;
    p.w = w; p.bias = bias;
    p.mode = EPI_STORE; p.slope = slope; p.cout = npad;
    setOut(p, out);
    return p;
}

ConvParams makeUp2Params(const Act& in, const Act& out, const __half* w, const float* bias, int cout, float slope, const Act* skip, int skipOff) {
    ConvParams p{};
    plainView(p, in);
    p.ntaps = 1;
    p.tap[0] = {0, 0, 0, 0};
    p.gx = in.w; p.gy = in.h;
    p.npad = 4 * cout; p.ktot = in.c;
    p.w = w; p.bias = bias;
    p.mode = EPI_D2S; p.slope = slope; p.cout = cout;
    setOut(p, out);
    if (skip) { p.skip = skip->p; p.skip_h = skip->h; p.skip_w = skip->w; p.skip_c = skip->c; p.skip_off = skipOff; }
    return p;
}

ConvParams makeUp4Params(const Act& in, const Act& out, const __half* w, const float* bias) {
    ConvParams p{};
    plainView(p, in);
    p.ntaps = 4;
    for (int wy = 0; wy < 2; ++wy)
        for (int wx = 0; wx < 2; ++wx) p.tap[wy * 2 + wx] = {0, wx, 0, wy};
    p.gx = in.w - 1; p.gy = in.h - 1;
    p.npad = 16; p.ktot = 4 * in.c;
    p.w = w; p.bias = bias;
    p.mode = EPI_UP4; p.slope = 1.f; p.cout = 4;
    setOut(p, out);
    return p;
}

// ------------------------------------------------------------------------------------------------
Engine::Engine() {}

Engine::~Engine() {
    try { unload(); } catch (...) {}
}

void Engine::log(int severity, const std::string& msg, const char* func, int line) {
    // "[func@line] msg", /root/reference/src/tensorrt/logger.cpp:19-22
    std::string full = std::string("[") + func + "@" + std::to_string(line) + "] " + msg;
    if (severity <= W2X_ERROR) lastErr = full;
    if (msgCb) msgCb(severity, full.c_str(), msgUser);
}
#define ELOG(sev, msg) log(sev, msg, __FUNCTION__, __LINE__)

void* Engine::dalloc(size_t bytes) {
    allocs.emplace_back(bytes ? bytes : 16);
    return allocs.back().get();
}

Act Engine::allocAct(int h, int w, int c) {
    if (h <= 0 || w <= 0) throw Error("tile size too small for this model");
    Act a;
    a.n = batch; a.h = h; a.w = w; a.c = c;
    a.p = (__half*)dalloc(a.elems() * elemBytes + 256);
    return a;
}

cudaEvent_t Engine::nextEvent() {
    if (timing.used == (int)timing.pool.size()) timing.pool.emplace_back();
    return timing.pool[timing.used++].get();
}

void Engine::unload() {
    if (stream) cudaStreamSynchronize(stream);
    if (h2dStream) cudaStreamSynchronize(h2dStream);
    if (d2hStream) cudaStreamSynchronize(d2hStream);
    for (auto& L : layers) {
        if (L.plan) igemmDestroyPlan(L.plan);
        if (L.tf32) tf32DestroyPlan(L.tf32);
        if (L.head) convHeadDestroyPlan(L.head);
        if (L.mlp) swinMlpDestroyPlan(L.mlp);
        if (L.attn) swinAttnDestroyPlan(L.attn);
    }
    layers.clear();
    dW.clear(); dBias.clear();
    allocs.clear();
    fc = {};
    staging = {};
    bgra = {};
    resize = {};
    band = {};
    pipe = {};
    timing = {};
    if (stream) { cudaStreamDestroy(stream); stream = nullptr; }
    if (h2dStream) { cudaStreamDestroy(h2dStream); h2dStream = nullptr; }
    if (d2hStream) { cudaStreamDestroy(d2hStream); d2hStream = nullptr; }
    isLoaded = false;
}

// ------------------------------------------------------------------------------------------------
// build: ONNX -> packed weights + json sidecar, named like the reference's engine files
// (img2img_build.cpp:151-166)
// ------------------------------------------------------------------------------------------------
static std::string deviceNameOf(int id) {
    cudaDeviceProp prop{};
    W2X_CUDA(cudaGetDeviceProperties(&prop, id));
    return prop.name;
}

bool Engine::build(const std::string& onnxPath, const w2x_build_config& bc) {
    try {
        cudaError_t e = cudaSetDevice(bc.deviceId);
        if (e != cudaSuccess) {
            ELOG(W2X_ERROR, "Failed to set cuda device to device id " + std::to_string(bc.deviceId) + ": " + cudaGetErrorString(e) + ".");
            return false;
        }
        if (bc.precision != W2X_PRECISION_FP16 && bc.precision != W2X_PRECISION_TF32) {
            ELOG(W2X_ERROR, "Failed to set precision: unknown precision " + std::to_string(bc.precision) + ".");
            return false;
        }
        OnnxGraph g;
        try {
            g = parseOnnx(readFile(onnxPath));
        } catch (const std::exception& ex) {
            ELOG(W2X_ERROR, std::string("Failed to parse ONNX model: ") + ex.what() + ".");
            return false;
        }
        if (bc.precision == W2X_PRECISION_TF32 && isSwinGraph(g)) {
            ELOG(W2X_ERROR, "Failed to set precision: tf32 is not available for swin_unet models.");
            return false;
        }
        PackedModel pm = packFromOnnx(g, bc.precision);
        const std::string name = deviceNameOf(bc.deviceId);
        const std::string base = fs::path(onnxPath).replace_extension("").string() + "_" + configHash(name, bc).substr(0, 16);
        Sidecar sc;
        sc.deviceName = name;
        sc.cfg = bc;
        writeSidecar(base + ".json", sc);
        const std::vector<uint8_t> blob = serializePack(pm);
        writeFile(base + ".w2x", blob.data(), blob.size());
        ELOG(W2X_INFO, "Packed " + std::to_string(pm.layers.size()) + " layers into \"" + base + ".w2x\"");
        return true;
    } catch (const std::exception& ex) {
        ELOG(W2X_ERROR, std::string("Engine build failed unexpectedly: ") + ex.what() + ".");
        return false;
    }
}

// getEnginePath, img2img_load.cpp:79-114: the selection rules live in hostutil.cpp (selectEngine) so they can be tested without a
// GPU; here only the device name of the requested device is looked up.
static std::string findEngine(const std::string& modelPath, const w2x_render_config& rc) {
    cudaDeviceProp prop{};
    const std::string name = cudaGetDeviceProperties(&prop, rc.deviceId) == cudaSuccess ? prop.name : "";
    return selectEngine(modelPath, rc, name);
}

// ------------------------------------------------------------------------------------------------
// load: packed weights -> HBM, activation arena, execution plan, streams (img2img_load.cpp:117-291)
// ------------------------------------------------------------------------------------------------
bool Engine::load(const std::string& onnxPath, const w2x_render_config& rc) {
    try {
        if (rc.precision != W2X_PRECISION_FP16 && rc.precision != W2X_PRECISION_TF32) {
            ELOG(W2X_ERROR, "Failed to set precision: unknown precision " + std::to_string(rc.precision) + ".");
            return false;
        }
        if (rc.precision == W2X_PRECISION_TF32) {
            // no tf32 engine file can exist for a SwinUNet (build refuses it): say why rather than that none was found
            bool swin = false;
            try { swin = isSwinGraph(parseOnnx(readFile(onnxPath))); } catch (const std::exception&) {}
            if (swin) {
                ELOG(W2X_ERROR, "Failed to set precision: tf32 is not available for swin_unet models.");
                return false;
            }
        }
        std::string enginePath;
        try {
            enginePath = findEngine(onnxPath, rc);
        } catch (const std::exception& ex) {
            ELOG(W2X_ERROR, "Failed to find engine file for model \"" + onnxPath + "\": " + ex.what() + ".");
            return false;
        }
        cudaError_t e = cudaSetDevice(rc.deviceId);
        if (e != cudaSuccess) {
            ELOG(W2X_ERROR, "Failed to set cuda device to device id " + std::to_string(rc.deviceId) + ": " + cudaGetErrorString(e) + ".");
            return false;
        }
        if (rc.channels != 3 || rc.width != rc.height || rc.batchSize < 1) {
            ELOG(W2X_ERROR, "Failed to set input tensor shape.");
            return false;
        }
        unload();
        model = deserializePack(readFile(enginePath));
        if ((int)model.precision != rc.precision) {
            ELOG(W2X_ERROR, "Engine file \"" + enginePath + "\" was packed for another precision.");
            return false;
        }
        if (model.arch == ARCH_SWINUNET && model.precision == W2X_PRECISION_TF32) {
            ELOG(W2X_ERROR, "Failed to set precision: tf32 is not available for swin_unet models.");
            return false;
        }
        elemBytes = model.precision == W2X_PRECISION_TF32 ? 4 : 2;
        if ((int)model.scale != rc.scaling) {
            ELOG(W2X_ERROR, "Render scaling " + std::to_string(rc.scaling) + " does not match the model's scale " + std::to_string(model.scale) + ".");
            return false;
        }
        cfg = rc;
        tile = rc.width;
        batch = rc.batchSize;
        scale = (int)model.scale;
        const char* impl = devEnv("W2X_CONV_IMPL");
        useDirect = impl && std::string(impl) == "direct";
        debugSync = std::getenv("W2X_DEBUG_SYNC") != nullptr;
        W2X_CUDA(cudaStreamCreateWithFlags(&stream, cudaStreamNonBlocking));  // img2img_load.cpp:206
        W2X_CUDA(cudaStreamCreateWithFlags(&h2dStream, cudaStreamNonBlocking));
        W2X_CUDA(cudaStreamCreateWithFlags(&d2hStream, cudaStreamNonBlocking));
        buildPlan();
        isLoaded = true;
        return true;
    } catch (const std::exception& ex) {
        ELOG(W2X_ERROR, std::string("Engine load failed unexpectedly: ") + ex.what() + ".");
        try { unload(); } catch (...) {}
        return false;
    }
}

// Host -> device upload of constants, ordered on the engine's compute stream: the streams are cudaStreamNonBlocking, so a plain
// cudaMemcpy (legacy default stream) would not be ordered before the kernels that read the data.
void Engine::uploadAsync(void* dst, const void* src, size_t bytes) {
    if (bytes) W2X_CUDA(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, stream));
}

void Engine::buildPlan() {
    if (model.arch == ARCH_SWINUNET) buildPlanSwin();
    else if (model.arch == ARCH_CUNET || model.arch == ARCH_UPCUNET) buildPlanCunet();
    else throw Error("unknown model architecture in pack file");
    W2X_CUDA(cudaStreamSynchronize(stream));  // every weight / table upload has landed before load() returns
}

void Engine::buildPlanCunet() {
    const bool up = model.arch == ARCH_UPCUNET;
    {
        // the plan below indexes layers 0..21 of the (Up)CUNet template: refuse a short, reordered or foreign pack file
        static const uint32_t kinds[22] = {L_CONV3, L_CONV3, L_DOWN2, L_CONV3, L_CONV3, L_UP2, L_CONV3, L_UP4, L_CONV3, L_CONV3, L_DOWN2,
                                           L_CONV3, L_CONV3, L_DOWN2, L_CONV3, L_CONV3, L_UP2, L_CONV3, L_CONV3, L_UP2, L_CONV3, L_CONV3};
        if (model.layers.size() != 22) throw Error("pack file does not hold the 22 layers of a CUNet/UpCUNet (" + std::to_string(model.layers.size()) + ")");
        for (int i = 0; i < 22; ++i) {
            const uint32_t want = (i == 7 && !up) ? (uint32_t)L_CONV3 : kinds[i];
            const PackedLayer& L = model.layers[i];
            if (L.kind != want) throw Error("pack file layer " + std::to_string(i) + " ('" + L.name + "') has an unexpected kind");
            if (L.weightCount() != (size_t)L.npad * L.ktot || L.bias.size() != L.npad) throw Error("pack file layer '" + L.name + "' is truncated");
        }
    }
    // weights -> HBM
    for (const auto& L : model.layers) {
        const size_t wBytes = L.weightCount() * elemBytes;
        __half* w = (__half*)dalloc(wBytes);
        float* b = (float*)dalloc(L.bias.size() * 4);
        uploadAsync(w, tf32() ? (const void*)L.wf.data() : (const void*)L.w.data(), wBytes);
        uploadAsync(b, L.bias.data(), L.bias.size() * 4);
        dW.push_back(w);
        dBias.push_back(b);
    }
    auto upload = [&](const std::vector<float>& v) {
        float* d = (float*)dalloc(v.size() * 4);
        uploadAsync(d, v.data(), v.size() * 4);
        return d;
    };
    auto even = [](int v, const char* what) {
        if (v <= 0 || (v & 1)) throw Error(std::string("tile size is not supported by this model (") + what + " must be even and positive)");
        return v;
    };
    const float S = 0.1f;
    // fused squeeze: the conv epilogue accumulates exact fixed-point channel sums (int64 atomics) per image
    auto fuseSqueeze = [&](LayerExec& E, const PackedLayer& L) {
        E.sePartialBytes = (size_t)batch * L.npad * sizeof(long long);
        E.sePartial = (long long*)dalloc(E.sePartialBytes);
        E.p.se_sum = E.sePartial;
        E.seFused = true;
    };
    // The plan below is the same for both precisions; only the kernel behind each layer differs.
    auto push = [&](int li, const ConvParams& p, double flops, bool fin = false) {
        LayerExec E;
        const PackedLayer& L = model.layers[li];
        E.name = L.name;
        E.p = p;
        E.flops = flops;
        E.isFinal = fin;
        const bool rgbFirst = L.kind == L_CONV3 && L.cin == 4 && L.npad == 32 && p.mode == EPI_STORE;
        if (tf32() && rgbFirst) E.impl = IMPL_FIRST_F32;
        else if (tf32()) {
            E.impl = IMPL_TF32;
            if (L.se_r) fuseSqueeze(E, L);
            E.tf32 = tf32CreatePlan(asF32(E.p));
        }
        else if (useDirect) E.impl = IMPL_DIRECT;
        else if (rgbFirst) E.impl = IMPL_FIRST;
        else if (convHeadSupported(p) && !devEnv("W2X_NO_HEAD_KERNEL")) { E.impl = IMPL_HEAD; E.head = convHeadCreatePlan(p); }
        else if (igemmSupported(p)) {
            E.impl = IMPL_IGEMM;
            if (L.se_r) fuseSqueeze(E, L);
            // a UNet's second convolution computes its RGB first layer on the fly (fusedFirstProducer): the 32-channel tensor
            // between them never touches HBM and the first layer's launch disappears
            static const bool noFuse = devEnv("W2X_NO_FUSE_FIRST") != nullptr;
            if (!noFuse && !layers.empty() && layers.back().impl == IMPL_FIRST && !L.se_r && igemmFusedFirstSupported(E.p, layers.back().p)) {
                E.plan = igemmCreatePlanFusedFirst(E.p, layers.back().p);
                layers.back().impl = IMPL_SKIP;
                E.flops += layers.back().flops;
                layers.back().flops = 0;
            } else {
                E.plan = igemmCreatePlan(E.p);
            }
        }
        else throw Error("no kernel for layer " + L.name);
        if (L.se_r) {
            E.seR = (int)L.se_r;
            E.seW1 = upload(L.se_w1); E.seB1 = upload(L.se_b1); E.seW2 = upload(L.se_w2); E.seB2 = upload(L.se_b2);
            if (!E.seFused) {
                E.sePartialBytes = (size_t)batch * L.cout * sizeof(long long);
                E.sePartial = (long long*)dalloc(E.sePartialBytes);
            }
            E.seScale = (float*)dalloc((size_t)batch * L.cout * 4);
        }
        layers.push_back(E);
    };
    auto conv3 = [&](int li, const Act& in, int cout, int mode = EPI_STORE, float slope = 0.1f, const Act* skip = nullptr, int skipOff = 0, bool fin = false) {
        const PackedLayer& L = model.layers[li];
        Act out = allocAct(in.h - 2, in.w - 2, cout < 8 ? 4 : cout);
        ConvParams p = makeConv3Params(in, out, dW[li], dBias[li], (int)L.npad, mode, slope, cout < 8 ? 4 : cout);
        if (skip) { p.skip = skip->p; p.skip_h = skip->h; p.skip_w = skip->w; p.skip_c = skip->c; p.skip_off = skipOff; }
        const int cinReal = L.cin == 4 ? 3 : (int)L.cin;
        push(li, p, 2.0 * p.gx * p.gy * (double)L.cout * 9 * cinReal, fin);
        return out;
    };
    // SE scale folding: when `in` is the (unscaled) output of an SE layer, the consumer multiplies by the SE scale through
    // per-image weights W'[img] = W * s[img] (written by the SE layer's excite step) instead of a separate in-place pass.
    auto foldInto = [&](int seLayerIdx, int li, ConvParams& p) {
        const PackedLayer& L = model.layers[li];
        LayerExec& prod = layers[seLayerIdx];
        if (!prod.seR) throw Error("internal: SE fold without an SE producer");
        __half* wImg = (__half*)dalloc((size_t)batch * L.weightCount() * elemBytes);
        prod.foldJobs.push_back({dW[li], wImg, (int)L.npad, (int)L.ktot, (int)L.cin});
        p.w = wImg;
        p.w_img_stride = (long long)L.weightCount();
    };
    auto down2 = [&](int li, const Act& in, int seProducer = -1) {
        const PackedLayer& L = model.layers[li];
        even(in.h, "down-sampled extent");
        Act out = allocAct(in.h / 2, in.w / 2, (int)L.cout);
        ConvParams p = makeDown2Params(in, out, dW[li], dBias[li], (int)L.npad, S);
        if (seProducer >= 0) foldInto(seProducer, li, p);
        push(li, p, 2.0 * p.gx * p.gy * (double)L.cout * 4 * L.cin);
        return out;
    };
    auto up2 = [&](int li, const Act& in, const Act& skip, int off, int seProducer = -1, int skipSeProducer = -1) {
        const PackedLayer& L = model.layers[li];
        Act out = allocAct(in.h * 2, in.w * 2, (int)L.cout);
        if (skip.h - 2 * off != out.h || skip.c != out.c) throw Error("tile size is not supported by this model (skip connection mismatch)");
        ConvParams p = makeUp2Params(in, out, dW[li], dBias[li], (int)L.cout, S, &skip, off);
        if (seProducer >= 0) foldInto(seProducer, li, p);
        if (skipSeProducer >= 0) p.skip_scale = layers[skipSeProducer].seScale;
        push(li, p, 2.0 * p.gx * p.gy * 4.0 * L.cout * L.cin);
        return out;
    };

    actIn = allocAct(tile, tile, 4);
    // ---- UNet1 ----
    Act a0 = conv3(0, actIn, 32);
    Act x1 = conv3(1, a0, 64);
    Act d1 = down2(2, x1);
    Act b0 = conv3(3, d1, 128);
    Act b1 = conv3(4, b0, 64);  // + SE (scale folded into conv2_up's weights)
    const int seB1 = (int)layers.size() - 1;
    Act u1 = up2(5, b1, x1, 4, seB1);
    Act c3 = conv3(6, u1, 64);
    Act z1;
    if (up) {
        const PackedLayer& L = model.layers[7];
        z1 = allocAct(2 * c3.h - 4, 2 * c3.w - 4, 4);
        ConvParams p = makeUp4Params(c3, z1, dW[7], dBias[7]);
        push(7, p, 2.0 * c3.h * c3.w * 16.0 * L.cout * L.cin);
    } else {
        z1 = conv3(7, c3, 3, EPI_STORE, 1.f);
    }
    // ---- UNet2 ----
    Act e0 = conv3(8, z1, 32);
    Act y1 = conv3(9, e0, 64);
    Act f1 = down2(10, y1);
    Act g0 = conv3(11, f1, 64);
    Act y2 = conv3(12, g0, 128);  // + SE (folded into conv2_down's weights and conv3_up's skip add)
    const int seY2 = (int)layers.size() - 1;
    Act f2 = down2(13, y2, seY2);
    Act h0 = conv3(14, f2, 256);
    Act h1 = conv3(15, h0, 128);  // + SE (folded into conv3_up's weights)
    const int seH1 = (int)layers.size() - 1;
    Act u3 = up2(16, h1, y2, 4, seH1, seY2);
    Act k0 = conv3(17, u3, 64);
    Act k1 = conv3(18, k0, 64);  // + SE (folded into conv4_up's weights)
    const int seK1 = (int)layers.size() - 1;
    Act u4 = up2(19, k1, y1, 16, seK1);
    Act c5 = conv3(20, u4, 64);
    if (z1.h - 40 != c5.h - 2) throw Error("tile size is not supported by this model (head crop mismatch)");
    actOut = conv3(21, c5, 3, EPI_FINAL, 1.f, &z1, 20, true);
    for (const auto& L : layers)  // the fp32 kernels take SE scales through the consumers' weights only (launchSeScale is fp16)
        if (tf32() && L.seR && (!L.seFused || L.foldJobs.empty())) throw Error("internal: tf32 SE layer '" + L.name + "' is not fused and folded");
    outTile = actOut.h;
    const int expect = up ? 2 * tile - 72 : tile - 56;
    if (outTile != expect) throw Error("internal: output tile size mismatch");
}

void Engine::launchLayer(LayerExec& L, cudaStream_t s, void* outp, int nImg, const void* inOverride) {
    switch (L.impl) {
        case IMPL_SKIP: break;  // computed inside the next layer's kernel
        case IMPL_IGEMM: igemmLaunch(L.plan, s, static_cast<__half*>(outp), nImg, static_cast<const __half*>(inOverride)); break;
        case IMPL_TF32: tf32Launch(L.tf32, s, static_cast<float*>(outp), nImg); break;
        case IMPL_FIRST_F32: {
            ConvParamsF32 p = asF32(L.p);
            p.gn = nImg;
            if (outp) p.out = static_cast<float*>(outp);
            if (inOverride) p.in = static_cast<const float*>(inOverride);
            launchConvFirstF32(p, s);
            break;
        }
        case IMPL_HEAD: launchConvHead(L.head, s, static_cast<__half*>(outp), nImg); break;
        case IMPL_SWIN_MLP: swinMlpLaunch(L.mlp, s, (long long)nImg * L.tokH * L.tokW); break;
        case IMPL_SWIN_ATTN: swinAttnLaunch(L.attn, s, nImg); break;
        case IMPL_LAYERNORM:
            launchLayerNorm(L.tokIn, L.tokOut, (long long)nImg * L.tokH * L.tokW, L.tokC, L.gamma, L.beta, L.eps, s);
            break;
        case IMPL_ATTENTION:
            launchWindowAttention(L.tokIn, L.tokOut, nImg, L.tokH, L.tokW, L.tokC, L.heads, L.window, L.shift, L.relpos, s);
            break;
        default: {
            ConvParams p = L.p;
            p.gn = nImg;
            if (outp) p.out = static_cast<__half*>(outp);
            if (inOverride) p.in = static_cast<const __half*>(inOverride);
            if (L.impl == IMPL_FIRST) launchConvFirst(p, s);
            else launchConvDirect(p, s);
        }
    }
}

// ------------------------------------------------------------------------------------------------
// SwinUNet execution plan (SURVEY 2.2): token tensors are NHWC fp16 [batch][h][w][C]; the residual stream is updated in
// place by the proj / fc2 epilogues (each thread reads exactly the element it then overwrites).
// ------------------------------------------------------------------------------------------------
void Engine::buildPlanSwin() {
    const int C = (int)model.dim, S = (int)model.scale;
    if (C != 96) throw Error("swin plan: only base_dim 96 (the released swin_unet models) is supported by the LayerNorm/attention kernels");
    if (C % 32 || tile < 64 || (tile - 16) % 48 != 0)
        throw Error("tile size is not supported by swin_unet ((tile - 16) must be a multiple of 48; SURVEY q10)");
    std::vector<float*> dAux0(model.layers.size(), nullptr), dAux1(model.layers.size(), nullptr);
    auto uploadF = [&](const std::vector<float>& v) {
        float* d = (float*)dalloc(std::max<size_t>(v.size(), 1) * 4);
        if (!v.empty()) uploadAsync(d, v.data(), v.size() * 4);
        return d;
    };
    for (size_t i = 0; i < model.layers.size(); ++i) {
        const auto& L = model.layers[i];
        __half* w = nullptr;
        float* b = nullptr;
        if (!L.w.empty()) {
            w = (__half*)dalloc(L.w.size() * 2);
            uploadAsync(w, L.w.data(), L.w.size() * 2);
            b = uploadF(L.bias);
        }
        dW.push_back(w);
        dBias.push_back(b);
        if (L.kind == L_LN) { dAux0[i] = uploadF(L.gamma); dAux1[i] = uploadF(L.beta); }
        if (L.kind == L_ATTN) {
            // relative-position bias as the attention kernel reads it: [head][48][40] (score tile padding), pre-multiplied by log2(e)
            // (the softmax runs on exp2), padded key columns pre-masked with -1e30 so the kernel needs no bounds tests
            if (L.window != 6 || L.relpos.size() != (size_t)L.heads * 36 * 36) throw Error("swin plan: window attention expects window 6 and a [heads][36][36] bias");
            std::vector<float> t((size_t)L.heads * 48 * 40, 0.f);
            for (uint32_t h = 0; h < L.heads; ++h)
                for (int r = 0; r < 48; ++r)
                    for (int c = 0; c < 40; ++c)
                        t[((size_t)h * 48 + r) * 40 + c] = c >= 36 ? -1e30f : (r < 36 ? L.relpos[((size_t)h * 36 + r) * 36 + c] * 1.4426950408889634f : 0.f);
            dAux0[i] = uploadF(t);
        }
    }
    size_t li = 0;
    auto next = [&](uint32_t kind) -> size_t {
        if (li >= model.layers.size() || model.layers[li].kind != kind) throw Error("swin plan: unexpected layer order in pack file");
        return li++;
    };
    auto pushConv = [&](size_t i, const ConvParams& p, double flops, bool fin = false) {
        LayerExec E;
        E.name = model.layers[i].name;
        E.p = p;
        E.flops = flops;
        E.isFinal = fin;
        if (useDirect) E.impl = IMPL_DIRECT;
        else if (model.layers[i].kind == L_CONV3 && model.layers[i].cin == 4) E.impl = IMPL_FIRST;
        else if (igemmSupported(p)) { E.impl = IMPL_IGEMM; E.plan = igemmCreatePlan(E.p); }
        else throw Error("no kernel for layer " + E.name);
        layers.push_back(E);
    };
    // ---- patch embedding: conv3x3(3->C/2) + lrelu, conv3x3(C/2->C) + lrelu, crop 6 ----
    actIn = allocAct(tile, tile, 4);
    const int T0 = tile - 16;  // token grid at level 1
    {
        const size_t i0 = next(L_CONV3);
        Act a0 = allocAct(tile - 2, tile - 2, 64);
        ConvParams p = makeConv3Params(actIn, a0, dW[i0], dBias[i0], 64, EPI_STORE, 0.1f, 64);
        pushConv(i0, p, 2.0 * p.gx * p.gy * (double)model.layers[i0].cout * 27);
        const size_t i1 = next(L_CONV3);
        // second conv computed directly on the cropped region: output (y, x) = full-conv output (y + 6, x + 6)
        Act view = a0;
        view.p = a0.p + ((size_t)6 * a0.w + 6) * a0.c;
        Act x1 = allocAct(T0, T0, C);
        ConvParams q = makeConv3Params(view, x1, dW[i1], dBias[i1], C, EPI_STORE, 0.1f, C);
        q.dimx = a0.w - 6; q.dimy = a0.h - 6;
        q.gx = T0; q.gy = T0;
        pushConv(i1, q, 2.0 * T0 * T0 * (double)C * 9 * model.layers[i1 - 1].cout);
        actOut = x1;
    }
    // scratch sized for level 1 (the largest token count)
    Act lnBuf = allocAct(T0, T0, C), qkvBuf = allocAct(T0, T0, 3 * C), attBuf = allocAct(T0, T0, C), hidBuf = allocAct(T0, T0, 2 * C);
    auto viewOf = [&](const Act& buf, int h, int w, int c) {
        Act v = buf;
        v.h = h; v.w = w; v.c = c;
        if (v.elems() > buf.elems()) throw Error("swin plan: scratch buffer too small");
        return v;
    };
    auto linear = [&](size_t i, const Act& in, const Act& out, int act, const Act* residual) {
        const PackedLayer& L = model.layers[i];
        ConvParams p{};
        p.in = in.p;
        p.dimc = in.c; p.dimx = in.w; p.dimz = 1; p.dimy = in.h;
        p.sx = in.c; p.sz = (long long)in.w * in.c; p.sy = (long long)in.w * in.c; p.sn = (long long)in.h * in.w * in.c;
        p.cin = in.c; p.gn = in.n;
        p.ntaps = 1; p.tap[0] = {0, 0, 0, 0};
        p.gx = in.w; p.gy = in.h;
        p.npad = (int)L.npad; p.ktot = (int)L.ktot;
        p.w = dW[i]; p.bias = dBias[i];
        p.mode = EPI_STORE; p.slope = 1.f; p.act = act; p.cout = (int)L.npad;
        p.out = out.p; p.out_h = out.h; p.out_w = out.w; p.out_c = out.c;
        if (residual) { p.skip = residual->p; p.skip_h = residual->h; p.skip_w = residual->w; p.skip_c = residual->c; p.skip_off = 0; }
        pushConv(i, p, 2.0 * in.h * in.w * (double)L.npad * L.ktot);
    };
    // regrouped / pre-scaled attention operands of the fused kernel: the host copies stay alive until the uploads have landed
    std::vector<std::vector<uint16_t>> keepW;
    std::vector<std::vector<float>> keepF;
    int blockIndex = 0;
    auto block = [&](Act& x) {
        const int h = x.h, w = x.w, c = x.c;
        const size_t n1 = next(L_LN), qk = next(L_LINEAR), at = next(L_ATTN), pj = next(L_LINEAR), n2 = next(L_LN), f1 = next(L_LINEAR), f2 = next(L_LINEAR);
        Act ln = viewOf(lnBuf, h, w, c), qkv = viewOf(qkvBuf, h, w, 3 * c), att = viewOf(attBuf, h, w, c), hid = viewOf(hidBuf, h, w, (int)model.layers[f1].npad);
        auto pushLn = [&](size_t i) {
            LayerExec E;
            E.name = model.layers[i].name; E.impl = IMPL_LAYERNORM;
            E.tokIn = x.p; E.tokOut = ln.p; E.tokN = x.n; E.tokH = h; E.tokW = w; E.tokC = c;
            E.gamma = dAux0[i]; E.beta = dAux1[i]; E.eps = model.layers[i].eps;
            layers.push_back(E);
        };
        const PackedLayer& QK = model.layers[qk];
        const PackedLayer &AT = model.layers[at], &PJ = model.layers[pj];
        const int blockShift = (blockIndex % 2) ? (int)AT.window / 2 : 0;
        const bool fuseAttn = !useDirect && !devEnv("W2X_NO_ATTN_FUSE") && swinAttnSupported(c, (int)AT.heads, (int)AT.window, h, w) && (int)QK.npad == 3 * c &&
                              (int)QK.ktot == c && (int)PJ.npad == c && (int)PJ.ktot == c && AT.relpos.size() == (size_t)AT.heads * 36 * 36;
        if (fuseAttn) {
            // c = 96: x += proj(window attention(LayerNorm(x))) in ONE kernel (normalised rows, Q / K / V, scores and probabilities stay on the
            // SM); c = 192: the same kernel up to the attention output, then the Linear kernel for proj + residual
            const bool fuseProj = swinAttnFusesProj(c);
            keepW.emplace_back();
            keepF.emplace_back();
            keepF.emplace_back();
            std::vector<uint16_t>& wR = keepW.back();
            std::vector<float>&bR = keepF[keepF.size() - 2], &relR = keepF.back();
            swinAttnPrepare(QK.w.data(), QK.bias.data(), AT.relpos.data(), c, (int)AT.heads, wR, bR, relR);
            __half* dWr = (__half*)dalloc(wR.size() * 2);
            uploadAsync(dWr, wR.data(), wR.size() * 2);
            float* dBr = uploadF(bR);
            float* dRel = uploadF(relR);
            for (size_t i : {n1, qk}) {
                LayerExec S;
                S.name = model.layers[i].name;
                S.impl = IMPL_SKIP;
                layers.push_back(S);
            }
            LayerExec E;
            E.impl = IMPL_SWIN_ATTN;
            E.tokN = x.n; E.tokH = h; E.tokW = w; E.tokC = c;
            E.heads = (int)AT.heads; E.window = (int)AT.window; E.shift = blockShift;
            const double flopsQkvAttn = 2.0 * h * w * (double)QK.npad * QK.ktot + 4.0 * (h / 6) * (w / 6) * 36.0 * 36.0 * c;
            E.attn = swinAttnCreatePlan(x.p, x.n, h, w, c, (int)AT.heads, (int)AT.window, blockShift, dAux0[n1], dAux1[n1], model.layers[n1].eps, dWr, dBr,
                                        fuseProj ? dW[pj] : nullptr, fuseProj ? dBias[pj] : nullptr, dRel, fuseProj ? nullptr : att.p);
            if (fuseProj) {
                LayerExec S;
                S.name = AT.name;
                S.impl = IMPL_SKIP;
                layers.push_back(S);
                E.name = PJ.name;
                E.flops = flopsQkvAttn + 2.0 * h * w * (double)PJ.npad * PJ.ktot;
                layers.push_back(E);
            } else {
                E.name = AT.name;
                E.flops = flopsQkvAttn;
                layers.push_back(E);
                linear(pj, att, x, ACT_LRELU, &x);   // x += proj(attn)
            }
        } else {
            pushLn(n1);
            linear(qk, ln, qkv, ACT_LRELU, nullptr);
        }
        if (!fuseAttn) {
            const PackedLayer& L = model.layers[at];
            if (L.window != 6 || (c / (int)L.heads != 16 && c / (int)L.heads != 32) || h % 6 || w % 6)
                throw Error("swin plan: unsupported attention geometry (window 6, head dim 16/32 only)");
            LayerExec E;
            E.name = L.name; E.impl = IMPL_ATTENTION;
            E.tokIn = qkv.p; E.tokOut = att.p; E.tokN = x.n; E.tokH = h; E.tokW = w; E.tokC = c;
            E.heads = (int)L.heads; E.window = (int)L.window; E.shift = (blockIndex % 2) ? (int)L.window / 2 : 0;
            E.relpos = dAux0[at];
            E.flops = 4.0 * (h / 6) * (w / 6) * 36.0 * 36.0 * c;
            layers.push_back(E);
            linear(pj, att, x, ACT_LRELU, &x);   // x += proj(attn)
        }
        const PackedLayer &F1 = model.layers[f1], &F2 = model.layers[f2];
        if (!useDirect && !devEnv("W2X_NO_MLP_FUSE") && swinMlpSupported(c, (int)F1.npad) && (int)F1.ktot == c && (int)F2.npad == c && F2.ktot == F1.npad) {
            // x += fc2(gelu(fc1(LayerNorm(x)))) in ONE kernel: the normalised rows and the hidden tensor stay in shared memory
            for (size_t i : {n2, f1}) {
                LayerExec S;
                S.name = model.layers[i].name;
                S.impl = IMPL_SKIP;
                layers.push_back(S);
            }
            LayerExec E;
            E.name = F2.name;
            E.impl = IMPL_SWIN_MLP;
            E.tokN = x.n; E.tokH = h; E.tokW = w; E.tokC = c;
            E.flops = 2.0 * h * w * ((double)F1.npad * F1.ktot + (double)F2.npad * F2.ktot);
            E.mlp = swinMlpCreatePlan(x.p, c, dAux0[n2], dAux1[n2], model.layers[n2].eps, dW[f1], dBias[f1], dW[f2], dBias[f2]);
            layers.push_back(E);
        } else {
            pushLn(n2);
            linear(f1, ln, hid, ACT_GELU, nullptr);
            linear(f2, hid, x, ACT_LRELU, &x);   // x += fc2(gelu(fc1(ln)))
        }
        ++blockIndex;
    };
    auto stage = [&](Act& x) {
        blockIndex = 0;  // shift alternates from 0 inside every stage
        while (li < model.layers.size() && model.layers[li].kind == L_LN) block(x);
    };
    auto down = [&](const Act& in) {
        const size_t i = next(L_DOWN2);
        const PackedLayer& L = model.layers[i];
        Act out = allocAct(in.h / 2, in.w / 2, (int)L.cout);
        ConvParams p = makeDown2Params(in, out, dW[i], dBias[i], (int)L.npad, 1.f);
        pushConv(i, p, 2.0 * p.gx * p.gy * (double)L.cout * 4 * L.cin);
        return out;
    };
    auto up = [&](const Act& in, const Act* skip) {
        const size_t i = next(L_UPLIN);
        const PackedLayer& L = model.layers[i];
        Act out = allocAct(in.h * 2, in.w * 2, (int)L.cout);
        if (skip && (skip->h != out.h || skip->c != out.c)) throw Error("swin plan: skip connection mismatch");
        ConvParams p = makeUp2Params(in, out, dW[i], dBias[i], (int)L.cout, 1.f, skip, 0);
        pushConv(i, p, 2.0 * p.gx * p.gy * 4.0 * L.cout * L.cin);
        return out;
    };
    Act x1 = actOut;
    stage(x1);
    Act x2 = down(x1);
    stage(x2);
    Act x3 = down(x2);
    stage(x3);
    Act y2 = up(x3, &x2);
    stage(y2);
    Act y1 = up(y2, &x1);
    stage(y1);
    Act top = y1;
    // 4x models end in PatchUp (Linear 96 -> 4 x 96, pixel shuffle 2) followed by ToImage (Linear 96 -> 4 x 3, pixel shuffle 2) with nothing in
    // between: one linear map 96 -> 16 x 3 with a pixel shuffle of 4.  Composed here in fp32 from the packed weights (then rounded to
    // fp16 once), the 4 x 96-wide intermediate tensor (177 MB per batch of four tiles) is neither written nor read.
    const bool composeHead = S == 4 && !useDirect && !devEnv("W2X_NO_HEAD_COMPOSE") && li + 2 == model.layers.size() && model.layers[li].kind == L_UPLIN &&
                             model.layers[li + 1].kind == L_TOIMG && model.layers[li + 1].upscale == 2 && model.layers[li + 1].ktot == model.layers[li].cout &&
                             model.layers[li].npad == 4 * model.layers[li].cout;
    if (S == 4 && !composeHead) top = up(y1, nullptr);
    {
        const size_t iu = composeHead ? next(L_UPLIN) : 0;
        const size_t i = next(L_TOIMG);
        const PackedLayer& L = model.layers[i];
        int s = (int)L.upscale, npad = 16;
        const __half* dWeights = dW[i];
        const float* dBiases = dBias[i];
        double flops = 2.0 * top.h * top.w * 3.0 * s * s * L.ktot;
        if (composeHead) {
            const PackedLayer& U = model.layers[iu];
            const int K = (int)U.ktot;
            keepW.emplace_back();
            keepF.emplace_back();
            std::vector<uint16_t>& wc = keepW.back();
            std::vector<float>& bc = keepF.back();
            composeUpToImage(U, L, wc, bc);
            __half* dWc = (__half*)dalloc(wc.size() * 2);
            uploadAsync(dWc, wc.data(), wc.size() * 2);
            dWeights = dWc;
            dBiases = uploadF(bc);
            s = 4;
            npad = 64;
            flops = 2.0 * top.h * top.w * 3.0 * s * s * K;
            LayerExec Sk;
            Sk.name = U.name;
            Sk.impl = IMPL_SKIP;
            layers.push_back(Sk);
        }
        Act out = allocAct(top.h * s, top.w * s, 4);
        ConvParams p{};
        p.in = top.p;
        p.dimc = top.c; p.dimx = top.w; p.dimz = 1; p.dimy = top.h;
        p.sx = top.c; p.sz = (long long)top.w * top.c; p.sy = (long long)top.w * top.c; p.sn = (long long)top.h * top.w * top.c;
        p.cin = top.c; p.gn = top.n;
        p.ntaps = 1; p.tap[0] = {0, 0, 0, 0};
        p.gx = top.w; p.gy = top.h;
        p.npad = npad; p.ktot = composeHead ? (int)model.layers[iu].ktot : (int)L.ktot;
        p.w = dWeights; p.bias = dBiases;
        p.mode = EPI_TOIMG; p.slope = 1.f; p.cout = s;
        p.out = out.p; p.out_h = out.h; p.out_w = out.w; p.out_c = 4;
        pushConv(i, p, flops, true);
        actOut = out;
    }
    if (li != model.layers.size()) throw Error("swin plan: trailing layers in pack file");
    outTile = actOut.h;
    if (outTile != (tile - 16) * S) throw Error("internal: swin output tile size mismatch");
    W2X_CUDA(cudaStreamSynchronize(stream));  // keepW / keepF are read by the uploads above
}

int Engine::layerKernel(int index, char* buf, int cap) const {
    if (index < 0 || index >= (int)layers.size()) return 0;
    const LayerExec& L = layers[index];
    if (L.plan) igemmDescribe(L.plan, buf, cap);
    else if (L.tf32) tf32Describe(L.tf32, buf, cap);
    else if (L.mlp) swinMlpDescribe(L.mlp, buf, cap);
    else if (L.attn) swinAttnDescribe(L.attn, buf, cap);
    else std::snprintf(buf, cap, "%s", L.impl == IMPL_FIRST ? "first-layer mma.sync" : L.impl == IMPL_FIRST_F32 ? "first-layer fp32 (CUDA cores)" :
                                       L.impl == IMPL_LAYERNORM ? "layernorm" :
                                       L.impl == IMPL_ATTENTION ? "window-attention mma.sync" :
                                       L.impl == IMPL_HEAD ? "head kernel, taps in N (tcgen05)" : L.impl == IMPL_SKIP ? "fused into the next layer" : "direct (reference kernel)");
    return 1;
}

// After the engine's work has finished: copy one tensor that the plan of layer `index` wrote or reads, as the last batch left it.
// It launches no kernel and changes no engine state.  dst == nullptr: report the size and the shape only.
long long Engine::layerTensor(int index, int which, void* dst, size_t cap, int* dims) {
    try {
        if (!isLoaded) throw Error("no engine loaded");
        if (model.arch != ARCH_CUNET && model.arch != ARCH_UPCUNET) throw Error("not a CUNet engine");
        if (which != 1 && (index < 0 || index >= (int)layers.size())) throw Error("layer index " + std::to_string(index) + " is out of range");
        const void* src = nullptr;
        size_t bytes = 0;
        int shape[4] = {batch, 1, 1, 1};
        if (which == 1) {
            src = actIn.p;
            bytes = actIn.elems() * elemBytes;
            shape[1] = actIn.h; shape[2] = actIn.w; shape[3] = actIn.c;
        } else {
            const LayerExec& L = layers[index];
            if (which == 0 && L.impl != IMPL_SKIP && !L.isFinal) {
                src = L.p.out;
                shape[1] = L.p.out_h; shape[2] = L.p.out_w; shape[3] = L.p.out_c;
                bytes = (size_t)batch * L.p.out_h * L.p.out_w * L.p.out_c * elemBytes;
            } else if (which == 2 && L.seR) {
                src = L.sePartial;
                bytes = L.sePartialBytes;
                shape[1] = (int)(bytes / ((size_t)batch * sizeof(long long)));
            } else if (which == 3 && L.seR) {
                src = L.seScale;
                shape[1] = L.p.out_c;
                bytes = (size_t)batch * L.p.out_c * sizeof(float);
            } else if (which == 4 && L.p.w_img_stride) {
                src = L.p.w;
                shape[1] = L.p.npad; shape[2] = (int)model.layers[index].ktot;
                bytes = (size_t)batch * L.p.w_img_stride * elemBytes;
            } else if (which < 0 || which > 4) {
                throw Error("unknown tensor " + std::to_string(which));
            }
        }
        if (dims) std::memcpy(dims, shape, sizeof shape);
        if (!src || !dst) return (long long)bytes;
        if (cap < bytes) throw Error("buffer of " + std::to_string(cap) + " bytes is too small for " + std::to_string(bytes));
        W2X_CUDA(cudaSetDevice(cfg.deviceId));
        W2X_CUDA(cudaStreamSynchronize(stream));
        W2X_CUDA(cudaStreamSynchronize(h2dStream));
        W2X_CUDA(cudaStreamSynchronize(d2hStream));
        W2X_CUDA(cudaMemcpy(dst, src, bytes, cudaMemcpyDeviceToHost));
        return (long long)bytes;
    } catch (const std::exception& ex) {
        ELOG(W2X_ERROR, std::string("Layer tensor copy failed: ") + ex.what() + ".");
        return -1;
    }
}

double Engine::flopsPerTile() const {
    double f = 0;
    for (const auto& L : layers) f += L.flops;
    return f;
}

// nImages < batch: the last, partially filled batch of a frame -- the padding slots (img2img_render.cpp:281) are not computed
// The layer that reads the model input can be pointed at another buffer when it is a direct / first-layer kernel (plain pointer) or
// the fused first layer (second tensor map); a first layer on the generic igemm path keeps the per-batch input tensor.
bool Engine::frameWideUnpack() const {
    if (layers.size() < 2) return false;
    const int impl = layers[0].impl;
    return impl == IMPL_FIRST || impl == IMPL_FIRST_F32 || impl == IMPL_DIRECT || (impl == IMPL_SKIP && layers[1].plan != nullptr);
}

// inTiles: this batch's unpacked tiles inside the frame-wide buffer (nullptr: the per-batch input tensor actIn)
void Engine::launchSe(const LayerExec& L, int n, cudaStream_t s) {
    if (!L.seFused) launchSeSqueeze(L.p.out, n, L.p.out_h, L.p.out_w, L.p.out_c, L.sePartial, s);
    launchSeExcite(L.sePartial, n, L.p.out_c, L.seR, L.p.out_h * L.p.out_w, L.seW1, L.seB1, L.seW2, L.seB2, L.seScale, s);
    if (L.foldJobs.empty()) launchSeScale(L.p.out, n, L.p.out_h, L.p.out_w, L.p.out_c, L.seScale, s);
    for (const auto& j : L.foldJobs) {
        if (tf32()) launchScaleWeightsF32(static_cast<const float*>(j.w), static_cast<float*>(j.wOut), L.seScale, n, j.npad, j.ktot, j.cin, s);
        else launchScaleWeights(static_cast<const __half*>(j.w), static_cast<__half*>(j.wOut), L.seScale, n, j.npad, j.ktot, j.cin, s);
    }
}

void Engine::runModel(cudaStream_t s, void* finalOut, int nImages, const void* inTiles) {
    const int n = (nImages > 0 && nImages < batch) ? nImages : batch;
    // SE accumulators are cleared up front so that the layer chain below is kernel -> kernel only (programmatic dependent launch)
    for (auto& L : layers)
        if (L.seR) W2X_CUDA(cudaMemsetAsync(L.sePartial, 0, L.sePartialBytes, s));
    for (size_t li = 0; li < layers.size(); ++li) {
        LayerExec& L = layers[li];
        void* outp = (L.isFinal && finalOut) ? finalOut : static_cast<void*>(L.p.out);
        // the layer that reads the model input: layer 0, or its fused consumer (layer 1) when layer 0 runs inside it
        const bool readsInput = inTiles && (li == 0 || (li == 1 && layers[0].impl == IMPL_SKIP));
        launchLayer(L, s, outp, n, readsInput ? inTiles : nullptr);
        if (L.impl != IMPL_SKIP) ++launches;
        if (debugSync) {
            cudaError_t de = cudaStreamSynchronize(s);
            if (de == cudaSuccess) de = cudaGetLastError();
            if (de != cudaSuccess) throw Error("layer '" + L.name + "': " + cudaGetErrorString(de));
        }
        if (L.seR) {
            launchSe(L, n, s);
            launches += (L.seFused ? 0 : 1) + 1 + (L.foldJobs.empty() ? 1 : (long long)L.foldJobs.size());
        }
    }
    W2X_CUDA(cudaGetLastError());
}

// ------------------------------------------------------------------------------------------------
// render (img2img_render.cpp:224-348)
// ------------------------------------------------------------------------------------------------
void Engine::ensureFrameBuffers(int w, int h, int passes) {
    if (w == fc.w && h == fc.h && passes == fc.passes) return;
    if (w <= 0 || h <= 0) throw Error("invalid frame size");
    W2X_CUDA(cudaStreamSynchronize(stream));
    // no frame matches the cache until every table below describes the new one: a frame refused here, or a failed allocation, must not
    // leave the previous key next to this frame's grid
    fc.w = fc.h = 0;
    TileGrid& grid = fc.grid;
    grid = calculateTiles(w, h, w * scale, h * scale, tile, tile, outTile, outTile, scale, cfg.overlapX, cfg.overlapY);
    if (grid.count <= 0) throw Error("frame is too small for the configured tile overlap");
    const int stepsPerTile = cfg.tta ? 8 : 1;
    // a BGRA frame with an alpha pass: the alpha steps follow the colour steps in the same order (alpha slot = colour slot +
    // count * stepsPerTile), and the batches are padded once per frame
    fc.batchCount = (int)std::lround(std::ceil((double)(grid.count * stepsPerTile * passes) / batch));  // render.cpp:249
    const int stepCount = fc.batchCount * batch;
    std::vector<RowBand>& rowBands = fc.rowBands;
    // Tile order.  The reference walks its column-major tile list (render.cpp:264-265).  A tile's result does not depend on its batch
    // or slot (exact integer SE sums), so without TTA the tiles are processed ROW by row instead: the output rows above the next tile row
    // are then final as soon as a tile row is done, which lets render() stitch and download them while later batches still compute.
    // rowBands[j] = {first output row, end row, batch after which they are final}; tileMapHost[ti] = slot of reference tile ti.
    rowBands.clear();
    std::vector<int> tileMapHost;
    std::vector<TileSlot> slots((size_t)stepCount);
    if (!cfg.tta) {
        tileMapHost.assign((size_t)grid.count, 0);
        for (int step = 0; step < stepCount; ++step) {
            if (step < grid.count * passes) {
                const int q = step % grid.count, j = q / grid.nx, i = q - j * grid.nx, ti = i * grid.ny + j;
                slots[step] = {grid.inRects[ti].x, grid.inRects[ti].y, 0, step < grid.count ? 1 : kSlotAlpha};
                if (step < grid.count) tileMapHost[ti] = step;
            } else {
                slots[step] = {0, 0, 0, 0};  // zero dummy tile, render.cpp:281
            }
        }
        int y0 = 0;
        for (int j = 0; j < grid.ny; ++j) {
            const int y1 = j + 1 < grid.ny ? grid.outRects[j + 1].y : h * scale;   // tile (0, j + 1): top of the next tile row
            if (y1 > y0) rowBands.push_back({y0, y1, ((j + 1) * grid.nx - 1) / batch});
            else if (!rowBands.empty()) rowBands.back().batch = ((j + 1) * grid.nx - 1) / batch;
            y0 = std::max(y0, y1);
        }
    } else {
        for (int step = 0; step < stepCount; ++step) {
            const int ti = step / stepsPerTile, aug = step % stepsPerTile;  // render.cpp:264-265
            if (ti < grid.count * passes) slots[step] = {grid.inRects[ti % grid.count].x, grid.inRects[ti % grid.count].y, aug, ti < grid.count ? 1 : kSlotAlpha};
            else slots[step] = {0, 0, 0, 0};  // zero dummy tile, render.cpp:281
        }
    }
    fc.slots.ensure(sizeof(TileSlot) * stepCount);
    uploadAsync(fc.slots.get(), slots.data(), sizeof(TileSlot) * stepCount);
    if (!tileMapHost.empty()) {
        fc.tileMap.ensure(sizeof(int) * tileMapHost.size());
        uploadAsync(fc.tileMap.get(), tileMapHost.data(), sizeof(int) * tileMapHost.size());
    }
    // a fused RGB first layer reads the frame-wide buffer through a tensor map of its own
    if (frameWideUnpack() && fc.unpacked.ensure((size_t)stepCount * tile * tile * 4 * elemBytes) && layers[0].impl == IMPL_SKIP)
        igemmSetFusedFrameInput(layers[1].plan, fc.unpacked.get<const __half>(), stepCount);
    const size_t tileElems = (size_t)outTile * outTile * 4;
    fc.tileOut.ensure((size_t)stepCount * tileElems * elemBytes);
    if (cfg.tta) fc.ttaMean.ensure((size_t)grid.count * passes * tileElems * sizeof(float));
    // a ramp drops its length while it is replaced, so that a failure leaves no length that its buffer does not hold
    auto ramp = [&](DeviceBuffer& buf, int& len, int overlap) {
        if (len == overlap) return;
        len = -1;
        const std::vector<float> r = blendRamp(overlap);
        buf.ensure(std::max<size_t>(r.size(), 1) * sizeof(float));
        uploadAsync(buf.get(), r.data(), r.size() * sizeof(float));
        len = overlap;
    };
    ramp(fc.rampX, fc.rampXLen, grid.outOvX);
    ramp(fc.rampY, fc.rampYLen, grid.outOvY);
    // the copies above are ordered on `stream` like every kernel that reads them; the sync keeps the staging vectors' lifetime trivial
    W2X_CUDA(cudaStreamSynchronize(stream));
    fc.w = w;
    fc.h = h;
    fc.passes = passes;
}

// Resized output: the tables and buffers of canvas cw x ch -> dw x dh.  Like ensureFrameBuffers, the key is cleared first and set only
// once every table has been uploaded.
void Engine::ensureResize(int cw, int ch, int dw, int dh) {
    if (cw == resize.cw && ch == resize.ch && dw == resize.dw && dh == resize.dh) return;
    W2X_CUDA(cudaStreamSynchronize(stream));
    resize.cw = resize.ch = resize.dw = resize.dh = 0;
    const ResampleAxis axes[2] = {resampleAxis(cw, dw), resampleAxis(ch, dh)};
    ResampleTable* tables[2] = {&resize.tx, &resize.ty};
    for (int a = 0; a < 2; ++a) {
        const ResampleAxis& ax = axes[a];
        const size_t intBytes = (size_t)ax.nOut * sizeof(int);
        resize.tables[a].ensure(2 * intBytes + ax.w.size() * sizeof(float));
        uint8_t* base = resize.tables[a].get<uint8_t>();
        uploadAsync(base, ax.first.data(), intBytes);
        uploadAsync(base + intBytes, ax.count.data(), intBytes);
        uploadAsync(base + 2 * intBytes, ax.w.data(), ax.w.size() * sizeof(float));
        *tables[a] = {reinterpret_cast<const int*>(base), reinterpret_cast<const int*>(base + intBytes), reinterpret_cast<const float*>(base + 2 * intBytes),
                      ax.taps};
    }
    resize.rowEnd.resize((size_t)dh);
    for (int i = 0; i < dh; ++i) resize.rowEnd[i] = axes[1].first[i] + axes[1].count[i];
    resize.canvas.ensure((size_t)cw * 3 * ch);
    resize.tmp.ensure((size_t)ch * dw * 3 * sizeof(float));
    W2X_CUDA(cudaStreamSynchronize(stream));   // the staging vectors above end with this call
    resize.cw = cw;
    resize.ch = ch;
    resize.dw = dw;
    resize.dh = dh;
}

void Engine::renderOnStream(const Frame& d, cudaStream_t s, bool timed, std::vector<BandDone>* bands) {
    const int w = d.w, h = d.h;
    const uint8_t* dSrc = static_cast<const uint8_t*>(d.src);
    uint8_t* dDst = static_cast<uint8_t*>(d.dst);
    if (timed) { timing.used = 0; timing.spans.clear(); }
    auto span = [&](int kind, auto&& fn) {
        if (!timed) { fn(); return; }
        cudaEvent_t e0 = nextEvent();
        const int i0 = timing.used - 1;
        W2X_CUDA(cudaEventRecord(e0, s));
        fn();
        cudaEvent_t e1 = nextEvent();
        W2X_CUDA(cudaEventRecord(e1, s));
        timing.spans.push_back({kind, i0, timing.used - 1});
    };
    int passes = 1;
    if (d.format == PixelFormat::Bgra8) {
        // The alpha plane decides the schedule: no alpha < 255, no alpha pass; some alpha == 0, the colour bleed first.  Both count as
        // unpack time.
        bgra.flags.ensure(2 * sizeof(int));
        int* dFlags = bgra.flags.get<int>();
        int flags[2] = {0, 0};
        span(0, [&] {
            W2X_CUDA(cudaMemsetAsync(dFlags, 0, 2 * sizeof(int), s));
            launchAlphaScan(dSrc, (size_t)w * h, dFlags, s);
            ++launches;
        });
        W2X_CUDA(cudaMemcpyAsync(flags, dFlags, sizeof flags, cudaMemcpyDeviceToHost, s));
        W2X_CUDA(cudaStreamSynchronize(s));
        passes = flags[0] ? 2 : 1;
        if (flags[1]) {
            for (DeviceBuffer& b : bgra.bleed) b.ensure((size_t)w * h * 4);
            // rounds = the model's input-side border (the halo of every tile): colour from farther away cannot reach an output pixel
            const int rounds = (int)(model.offset / std::max<uint32_t>(model.scale, 1));
            span(0, [&] {
                const uint8_t* in = dSrc;
                for (int r = 0; r < std::max(rounds, 1); ++r) {
                    uint8_t* out = bgra.bleed[r & 1].get<uint8_t>();
                    launchAlphaBleedRound(in, out, w, h, rounds > 0 ? 1 : 0, r + 1 >= rounds ? dSrc : nullptr, s);
                    ++launches;
                    in = out;
                }
                dSrc = in;
            });
        }
    }
    ensureFrameBuffers(w, h, passes);
    const int cw = w * scale, ch = h * scale;
    const Frame::Size out = outputSize(d);
    const int dstW = out.w, dstH = out.h;
    // a resized frame is stitched into the engine's canvas and resampled from there into dDst
    const bool resized = dstW != cw || dstH != ch;
    if (resized) ensureResize(cw, ch, dstW, dstH);
    const TileGrid& grid = fc.grid;
    const bool progressive = d.format != PixelFormat::Bgra8 && bands != nullptr && !cfg.tta && !fc.rowBands.empty();
    if (bands) bands->clear();
    auto stitchRows = [&](int yBegin, int yEnd) {
        StitchParams sp = stitchGrid(outTile, grid.nx, grid.ny, grid.outOvX, grid.outOvY, cw, ch, fc.rampX.get<float>(), fc.rampY.get<float>());
        sp.dst = resized ? resize.canvas.get<uint8_t>() : dDst;
        sp.pitch = resized ? (size_t)cw * 3 : d.dstStride;
        sp.tiles = cfg.tta ? fc.ttaMean.get() : fc.tileOut.get();
        sp.f32 = (cfg.tta || tf32()) ? 1 : 0;
        sp.tile_map = cfg.tta ? nullptr : fc.tileMap.get<int>();
        sp.y_begin = yBegin; sp.y_end = yEnd;
        sp.format = d.format;
        sp.alpha_off = passes == 2 ? grid.count : 0;   // TTA: index of the reduced alpha tile; else the alpha step of the tile's slot
        launchStitch(sp, s);
        ++launches;
    };
    // Canvas rows [y0, y1) have just been stitched: resample them horizontally, then every output row not yet written whose vertical
    // window ends at or above y1 (a prefix of the rows left, since the windows are monotone).  Returns the output rows written.
    int rowsOut = 0;
    auto resampleRows = [&](int y0, int y1) {
        launchResampleH(resize.canvas.get<uint8_t>(), (size_t)cw * 3, y0, y1, resize.tx, dstW, resize.tmp.get<float>(), s);
        ++launches;
        const int i0 = rowsOut;
        while (rowsOut < dstH && resize.rowEnd[rowsOut] <= y1) ++rowsOut;
        if (rowsOut > i0) {
            launchResampleV(resize.tmp.get<float>(), dstW, resize.ty, i0, rowsOut, dDst, d.dstStride, s);
            ++launches;
        }
        return std::make_pair(i0, rowsOut);
    };
    const size_t tileElems = (size_t)outTile * outTile * 4;
    const size_t inElems = (size_t)tile * tile * 4;
    // real (non-padding) slots: the reference computes the zero padding tiles of the last batch and discards them (:281,:298)
    const int realSteps = grid.count * (cfg.tta ? 8 : 1) * passes;
    // all tiles of the frame are unpacked by ONE launch into a frame-wide buffer; the batches then chain kernel -> kernel
    const bool frameWide = frameWideUnpack();
    if (frameWide)
        span(0, [&] {
            unpackTiles(dSrc, w, h, d.srcStride, fc.slots.get<TileSlot>(), realSteps, fc.unpacked.get(), s, d.format);
            ++launches;
        });
    for (int b = 0; b < fc.batchCount; ++b) {
        const auto t0 = std::chrono::steady_clock::now();
        const int nReal = std::min(batch, realSteps - b * batch);
        if (nReal <= 0) continue;
        if (!frameWide)
            span(0, [&] {
                unpackTiles(dSrc, w, h, d.srcStride, fc.slots.get<TileSlot>() + (size_t)b * batch, nReal, actIn.p, s, d.format);
                ++launches;
            });
        span(1, [&] { runModel(s, elemAt(fc.tileOut.get(), (size_t)b * batch * tileElems), nReal, frameWide ? elemAt(fc.unpacked.get(), (size_t)b * batch * inElems) : nullptr); });
        if (progressive) {
            // output rows that only depend on tile rows finished with this batch: stitch them now, hand the caller an event to copy after
            for (const RowBand& rb : fc.rowBands) {
                if (rb.batch != b) continue;
                std::pair<int, int> rows{rb.y0, rb.y1};
                span(2, [&] {
                    stitchRows(rb.y0, rb.y1);
                    if (resized) rows = resampleRows(rb.y0, rb.y1);
                });
                if (rows.second <= rows.first) continue;
                if (fc.bandEv.size() <= bands->size()) fc.bandEv.emplace_back(cudaEventDisableTiming);
                cudaEvent_t e = fc.bandEv[bands->size()].get();
                W2X_CUDA(cudaEventRecord(e, s));
                bands->push_back({rows.first, rows.second, e});
            }
        }
        if (progCb) {
            const double ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
            progCb(b + 1, fc.batchCount, 1000.0 / std::max(ms, 1e-6), progUser);  // render.cpp:336-338
        }
    }
    if (progressive) {
        W2X_CUDA(cudaGetLastError());
        return;
    }
    if (cfg.tta)
        span(4, [&] {
            ttaReduce(fc.tileOut.get(), grid.count * passes, fc.ttaMean.get<float>(), s);
            ++launches;
        });
    span(2, [&] {
        stitchRows(0, ch);
        if (resized) resampleRows(0, ch);
    });
    W2X_CUDA(cudaGetLastError());
}

void Engine::unpackTiles(const uint8_t* src, int w, int h, size_t pitch, const TileSlot* slots, int n, void* out, cudaStream_t s,
                         PixelFormat format) {
    if (tf32()) launchUnpack(src, w, h, pitch, slots, n, tile, static_cast<float*>(out), s, format);
    else launchUnpack(src, w, h, pitch, slots, n, tile, static_cast<__half*>(out), s, format);
}

void Engine::ttaReduce(const void* outs, int tiles, float* mean, cudaStream_t s) {
    if (tf32()) launchTtaReduce(static_cast<const float*>(outs), tiles, outTile, mean, s);
    else launchTtaReduce(static_cast<const __half*>(outs), tiles, outTile, mean, s);
}

int Engine::lastStageMs(float* out, int n) {
    if (!stream) return 0;
    cudaStreamSynchronize(stream);
    float acc[5] = {0, 0, 0, 0, 0};  // unpack, model, stitch, total, tta_reduce
    auto& pool = timing.pool;
    const auto& spans = timing.spans;
    for (const auto& sp : spans) {
        float ms = 0;
        if (cudaEventElapsedTime(&ms, pool[sp.e0].get(), pool[sp.e1].get()) == cudaSuccess) acc[sp.kind] += ms;
    }
    if (!spans.empty()) {
        float ms = 0;
        if (cudaEventElapsedTime(&ms, pool[spans.front().e0].get(), pool[spans.back().e1].get()) == cudaSuccess) acc[3] = ms;
    }
    const int k = std::min(n, 5);
    for (int i = 0; i < k; ++i) out[i] = acc[i];
    return k;
}

bool Engine::timerMark(int idx, int which) {
    if (idx < 0 || idx >= 16 || !stream) return false;
    if (cudaSetDevice(cfg.deviceId) != cudaSuccess) return false;
    cudaStream_t s = which == 1 ? h2dStream : which == 2 ? d2hStream : stream;
    try {
        return cudaEventRecord(timing.marks[idx].get(), s) == cudaSuccess;
    } catch (const Error&) {
        return false;
    }
}

float Engine::timerElapsedMs(int i0, int i1) {
    if (i0 < 0 || i1 < 0 || i0 >= 16 || i1 >= 16 || !timing.marks[i0].created() || !timing.marks[i1].created()) return -1.f;
    cudaEvent_t e0 = timing.marks[i0].get(), e1 = timing.marks[i1].get();
    if (cudaEventSynchronize(e0) != cudaSuccess || cudaEventSynchronize(e1) != cudaSuccess) return -1.f;
    float ms = -1.f;
    if (cudaEventElapsedTime(&ms, e0, e1) != cudaSuccess) return -1.f;
    return ms;
}

void Engine::checkFrame(const Frame& f, FramePath path) const {
    if (!isLoaded) throw Error("no engine loaded");
    if (!f.src || !f.dst) throw Error("null image pointer");
    if (f.w <= 0 || f.h <= 0) throw Error("invalid frame size");
    if (f.format == PixelFormat::Bgra8 && path != FramePath::Render) throw Error("BGRA frames are rendered synchronously only");
    if (f.out && f.format != PixelFormat::Bgr8) throw Error("resized output is u8 BGR only");
    if ((path == FramePath::Device || path == FramePath::Banded) && (f.format != PixelFormat::Bgr8 || f.out))
        throw Error("device and row-band frames are u8 BGR at the model's scale");
    const Frame::Size out = outputSize(f);
    if (out.w < 1 || out.w > f.w * scale || out.h < 1 || out.h > f.h * scale)
        throw Error("output size " + std::to_string(out.w) + "x" + std::to_string(out.h) + " is outside 1x1 .. " + std::to_string(f.w * scale) + "x" +
                    std::to_string(f.h * scale) + " (the resample only reduces the model's " + std::to_string(scale) + "x output)");
    const size_t bpp = bytesPerPixel(f.format);
    if (f.srcStride < (size_t)f.w * bpp || f.dstStride < (size_t)out.w * bpp)
        throw Error("row stride is smaller than " + std::to_string(bpp) + " bytes per pixel");
    if (f.format == PixelFormat::Bgr16) {
        if ((f.srcStride | f.dstStride) & 1) throw Error("row stride is odd (u16 rows must be 2-byte aligned)");
        if ((reinterpret_cast<uintptr_t>(f.src) | reinterpret_cast<uintptr_t>(f.dst)) & 1)
            throw Error("image pointer is odd (u16 samples must be 2-byte aligned)");
    }
}

namespace {
// f with its buffers replaced by packed ones of pitch srcPitch / dstPitch (the engine's copies on the device)
Frame packedOnDevice(Frame f, const void* src, size_t srcPitch, void* dst, size_t dstPitch) {
    f.src = src;
    f.srcStride = srcPitch;
    f.dst = dst;
    f.dstStride = dstPitch;
    return f;
}
}  // namespace

bool Engine::renderDevice(const Frame& f) {
    try {
        checkFrame(f, FramePath::Device);
        W2X_CUDA(cudaSetDevice(cfg.deviceId));
        renderOnStream(f, stream, true);
        return true;
    } catch (const std::exception& ex) {
        ELOG(W2X_ERROR, std::string("Render failed unexpectedly: ") + ex.what() + ".");
        return false;
    }
}

// host frame -> staging buffers -> renderOnStream -> host frame, synchronous
bool Engine::render(const Frame& f) {
    try {
        checkFrame(f, FramePath::Render);
        W2X_CUDA(cudaSetDevice(cfg.deviceId));
        const Frame::Size out = outputSize(f);
        const size_t ipitch = (size_t)f.w * bytesPerPixel(f.format), opitch = (size_t)out.w * bytesPerPixel(f.format);
        staging.in.ensure(ipitch * f.h);
        staging.out.ensure(opitch * out.h);
        uint8_t *dIn = staging.in.get<uint8_t>(), *dOut = staging.out.get<uint8_t>();
        uint8_t* dst = static_cast<uint8_t*>(f.dst);
        W2X_CUDA(cudaMemcpy2DAsync(dIn, ipitch, f.src, f.srcStride, ipitch, f.h, cudaMemcpyHostToDevice, stream));  // render.cpp:226
        // every kernel of the frame is queued first; the output then leaves band by band (rows that are final after a tile row), each copy
        // ordered behind its band's stitch only, so the download of a band overlaps the batches still computing (the reference downloads
        // the whole canvas after the last batch, render.cpp:344).  With --tta, and for BGRA frames, there is one band: the whole frame.
        std::vector<BandDone> bands;
        renderOnStream(packedOnDevice(f, dIn, ipitch, dOut, opitch), stream, true, &bands);
        if (bands.empty()) {
            W2X_CUDA(cudaMemcpy2DAsync(dst, f.dstStride, dOut, opitch, opitch, (size_t)out.h, cudaMemcpyDeviceToHost, stream));  // render.cpp:344
        } else {
            for (const BandDone& bd : bands) {
                W2X_CUDA(cudaStreamWaitEvent(d2hStream, bd.ev, 0));
                W2X_CUDA(cudaMemcpy2DAsync(dst + (size_t)bd.y0 * f.dstStride, f.dstStride, dOut + (size_t)bd.y0 * opitch, opitch, opitch,
                                           (size_t)(bd.y1 - bd.y0), cudaMemcpyDeviceToHost, d2hStream));
            }
            W2X_CUDA(cudaStreamSynchronize(d2hStream));
        }
        W2X_CUDA(cudaStreamSynchronize(stream));  // the sync the reference leaves commented out (render.cpp:345)
        return true;
    } catch (const std::exception& ex) {
        ELOG(W2X_ERROR, std::string("Render failed unexpectedly: ") + ex.what() + ".");
        return false;
    }
}

// Pipelined frames: H2D (copy stream) -> compute (engine stream) -> D2H (copy stream), kSlots frames in flight.
int Engine::submit(const Frame& f) {
    try {
        checkFrame(f, FramePath::Submit);
        W2X_CUDA(cudaSetDevice(cfg.deviceId));
        const int ticket = nextTicket;
        PipeSlot& ps = pipe[ticket % kSlots];
        if (ps.busy) { W2X_CUDA(cudaEventSynchronize(ps.evDone.get())); ps.busy = false; }
        const Frame::Size out = outputSize(f);
        const size_t ipitch = (size_t)f.w * bytesPerPixel(f.format), opitch = (size_t)out.w * bytesPerPixel(f.format);
        ps.in.ensure(ipitch * f.h);
        ps.out.ensure(opitch * out.h);
        uint8_t *dIn = ps.in.get<uint8_t>(), *dOut = ps.out.get<uint8_t>();
        ensureFrameBuffers(f.w, f.h);
        W2X_CUDA(cudaMemcpy2DAsync(dIn, ipitch, f.src, f.srcStride, ipitch, f.h, cudaMemcpyHostToDevice, h2dStream));
        W2X_CUDA(cudaEventRecord(ps.evH2D.get(), h2dStream));
        W2X_CUDA(cudaStreamWaitEvent(stream, ps.evH2D.get(), 0));
        renderOnStream(packedOnDevice(f, dIn, ipitch, dOut, opitch), stream, false);
        W2X_CUDA(cudaEventRecord(ps.evComp.get(), stream));
        W2X_CUDA(cudaStreamWaitEvent(d2hStream, ps.evComp.get(), 0));
        W2X_CUDA(cudaMemcpy2DAsync(f.dst, f.dstStride, dOut, opitch, opitch, (size_t)out.h, cudaMemcpyDeviceToHost, d2hStream));
        W2X_CUDA(cudaEventRecord(ps.evDone.get(), d2hStream));
        ps.busy = true;
        ++nextTicket;
        return ticket;
    } catch (const std::exception& ex) {
        ELOG(W2X_ERROR, std::string("Submit failed unexpectedly: ") + ex.what() + ".");
        return -1;
    }
}

// ------------------------------------------------------------------------------------------------
// Row-band mode (SURVEY 8e, "single large image"): the GLOBAL tile grid is computed once, exactly as for one GPU (bands are
// unions of the reference's tiles: SE pooling is per tile, so re-tiling would change results), and split into contiguous
// bands of tile rows, one per engine/GPU.  Each GPU receives only the input rows its tiles read (band rows + halo; replicate
// padding can then only trigger at the true image edges), renders its tiles (with --tta: eight augmentations + the mean), and
// stitches and downloads only its own output rows.  The one exchange is the blended seam: the bottom `oov` rows of the upper
// band's last tile row (cfg4: 9 x 64 x 960 x 8 B = 4.4 MB), copied peer-to-peer over NVLink into the lower neighbour's tile
// buffer.  No collective, no NCCL, no host synchronisation between the devices until the final wait; the result is
// byte-identical to the single-GPU render (same tiles, same fp32 add order).
// ------------------------------------------------------------------------------------------------
bool Engine::renderBanded(Engine* const* es, int count, const Frame& f) {
    if (!es || count < 1 || !es[0]) return false;
    Engine& e0 = *es[0];
    try {
        for (int r = 0; r < count; ++r) {
            if (!es[r] || !es[r]->isLoaded) throw Error("no engine loaded");
            if (es[r]->tile != e0.tile || es[r]->outTile != e0.outTile || es[r]->scale != e0.scale || es[r]->batch != e0.batch ||
                es[r]->cfg.overlapX != e0.cfg.overlapX || es[r]->cfg.overlapY != e0.cfg.overlapY || es[r]->cfg.tta != e0.cfg.tta ||
                es[r]->elemBytes != e0.elemBytes)
                throw Error("row-band render needs identically configured engines");
        }
        e0.checkFrame(f, FramePath::Banded);
        const uint8_t* src = static_cast<const uint8_t*>(f.src);
        uint8_t* dst = static_cast<uint8_t*>(f.dst);
        const int w = f.w, h = f.h;
        const size_t srcStride = f.srcStride, dstStride = f.dstStride;
        const int scale = e0.scale, outT = e0.outTile, tile = e0.tile, batch = e0.batch;
        const bool tta = e0.cfg.tta != 0;
        const int spt = tta ? 8 : 1;  // model runs per tile
        const TileGrid g = calculateTiles(w, h, w * scale, h * scale, tile, tile, outT, outT, scale, e0.cfg.overlapX, e0.cfg.overlapY);
        if (g.count <= 0) throw Error("frame is too small for the configured tile overlap");
        const int bands = std::min(count, g.ny);
        const size_t tileElems = (size_t)outT * outT * 4;
        const size_t elemBytes = tta ? sizeof(float) : e0.elemBytes;  // stitched tiles: the model outputs, or the f32 TTA means
        const int sty = outT - g.outOvY;
        const int cw = w * scale, ch = h * scale;
        struct Band { int j0, j1, own, steps, yBegin, yEnd, inY0, inY1; };
        std::vector<Band> bd(bands);
        for (int r = 0; r < bands; ++r) {
            const int base = g.ny / bands, extra = g.ny % bands;
            bd[r].j0 = r * base + std::min(r, extra);
            bd[r].j1 = bd[r].j0 + base + (r < extra ? 1 : 0);
            bd[r].own = (bd[r].j1 - bd[r].j0) * g.nx;
            bd[r].steps = (bd[r].own * spt + batch - 1) / batch * batch;       // own model runs padded to whole batches
            bd[r].yBegin = r == 0 ? 0 : bd[r].j0 * sty;
            bd[r].yEnd = r == bands - 1 ? ch : bd[r].j1 * sty;
            // input rows read by this band's tiles (tile rows are the inner index of the column-major grid: tile (0, j) is rect j)
            bd[r].inY0 = std::max(0, g.inRects[bd[r].j0].y);
            bd[r].inY1 = std::min(h, g.inRects[bd[r].j1 - 1].y + tile);
            if (bd[r].inY1 <= bd[r].inY0) { bd[r].inY0 = std::min(std::max(bd[r].inY0, 0), h - 1); bd[r].inY1 = bd[r].inY0 + 1; }
        }
        // ---- phase 1: every band uploads its rows, unpacks and runs the model on its tiles; nothing here waits for a device ----
        for (int r = 0; r < bands; ++r) {
            Engine& e = *es[r];
            const Band& b = bd[r];
            W2X_CUDA(cudaSetDevice(e.cfg.deviceId));
            e.ensureFrameBuffers(w, h);  // blend ramps for this frame size
            const int bandH = b.inY1 - b.inY0;
            e.staging.in.ensure((size_t)w * 3 * bandH);
            e.staging.out.ensure((size_t)cw * 3 * (size_t)(b.yEnd - b.yBegin));
            e.band.tiles.ensure(((size_t)b.steps * tileElems + (tta ? 0 : (size_t)g.nx * tileElems)) * e.elemBytes);
            if (tta) e.band.mean.ensure((size_t)(b.own + g.nx) * tileElems * sizeof(float));
            e.band.map.ensure((size_t)g.count * sizeof(int));
            e.band.slots.ensure((size_t)b.steps * sizeof(TileSlot));
            uint8_t* dIn = e.staging.in.get<uint8_t>();
            TileSlot* dSlots = e.band.slots.get<TileSlot>();
            // model runs in row-major band order (a tile row is contiguous for the seam copy), eight consecutive augmentations per
            // tile with --tta; map: global tile index -> slot of the stitched tile buffer.  The staging vectors live in the engine
            // so that the asynchronous copies below never outlive them.
            e.band.slotsHost.assign((size_t)b.steps, TileSlot{0, 0, 0, 0});
            e.band.mapHost.assign((size_t)g.count, -1);
            for (int j = b.j0; j < b.j1; ++j)
                for (int i = 0; i < g.nx; ++i) {
                    const int s = (j - b.j0) * g.nx + i, t = i * g.ny + j;
                    for (int a = 0; a < spt; ++a) e.band.slotsHost[(size_t)s * spt + a] = {g.inRects[t].x, g.inRects[t].y - b.inY0, a, 1};
                    e.band.mapHost[t] = s;
                }
            const int recvSlot = tta ? b.own : b.steps;  // where the seam row received from the band above lands
            if (r > 0)
                for (int i = 0; i < g.nx; ++i) e.band.mapHost[i * g.ny + b.j0 - 1] = recvSlot + i;
            W2X_CUDA(cudaMemcpyAsync(dSlots, e.band.slotsHost.data(), sizeof(TileSlot) * e.band.slotsHost.size(), cudaMemcpyHostToDevice, e.stream));
            W2X_CUDA(cudaMemcpyAsync(e.band.map.get(), e.band.mapHost.data(), sizeof(int) * e.band.mapHost.size(), cudaMemcpyHostToDevice, e.stream));
            W2X_CUDA(cudaMemcpy2DAsync(dIn, (size_t)w * 3, src + (size_t)b.inY0 * srcStride, srcStride, (size_t)w * 3, bandH, cudaMemcpyHostToDevice, e.stream));
            const int realSteps = b.own * spt;
            for (int bi = 0; bi < b.steps / batch; ++bi) {
                const int nReal = std::min(batch, realSteps - bi * batch);
                if (nReal <= 0) break;
                e.unpackTiles(dIn, w, bandH, (size_t)w * 3, dSlots + (size_t)bi * batch, nReal, e.actIn.p, e.stream, PixelFormat::Bgr8);
                ++e.launches;
                W2X_CUDA(cudaGetLastError());
                e.runModel(e.stream, e.elemAt(e.band.tiles.get(), (size_t)bi * batch * tileElems), nReal);
            }
            if (tta) {
                e.ttaReduce(e.band.tiles.get(), b.own, e.band.mean.get<float>(), e.stream);
                ++e.launches;
            }
            W2X_CUDA(cudaEventRecord(e.band.evModel.get(), e.stream));
        }
        // ---- phase 2: seam exchange (bottom overlap rows of band r-1's last tile row -> band r), stitch own rows, download ----
        for (int r = 0; r < bands; ++r) {
            Engine& e = *es[r];
            const Band& b = bd[r];
            W2X_CUDA(cudaSetDevice(e.cfg.deviceId));
            uint8_t* tilesBase = (tta ? e.band.mean : e.band.tiles).get<uint8_t>();
            if (r > 0 && g.outOvY > 0) {
                Engine& up = *es[r - 1];
                if (up.cfg.deviceId != e.cfg.deviceId) {
                    int can = 0;
                    if (cudaDeviceCanAccessPeer(&can, e.cfg.deviceId, up.cfg.deviceId) == cudaSuccess && can) {
                        const cudaError_t pe = cudaDeviceEnablePeerAccess(up.cfg.deviceId, 0);  // direct NVLink path for the seam copy
                        if (pe != cudaSuccess && pe != cudaErrorPeerAccessAlreadyEnabled) W2X_CUDA(pe);
                        (void)cudaGetLastError();
                    }
                }
                W2X_CUDA(cudaStreamWaitEvent(e.stream, up.band.evModel.get(), 0));
                const uint8_t* upBase = (tta ? up.band.mean : up.band.tiles).get<const uint8_t>();
                const size_t tileBytes = tileElems * elemBytes;
                const size_t rowOff = (size_t)(outT - g.outOvY) * outT * 4 * elemBytes;      // first blended row inside a tile
                const size_t stripBytes = (size_t)g.outOvY * outT * 4 * elemBytes;           // the overlap rows of one tile: contiguous
                const uint8_t* srcRow = upBase + (size_t)(bd[r - 1].j1 - 1 - bd[r - 1].j0) * g.nx * tileBytes + rowOff;
                uint8_t* dstRow = tilesBase + (size_t)(tta ? b.own : b.steps) * tileBytes + rowOff;
                W2X_CUDA(cudaMemcpy2DAsync(dstRow, tileBytes, srcRow, tileBytes, stripBytes, (size_t)g.nx, cudaMemcpyDefault, e.stream));
            }
            StitchParams sp = stitchGrid(outT, g.nx, g.ny, g.outOvX, g.outOvY, cw, ch, e.fc.rampX.get<float>(), e.fc.rampY.get<float>());
            sp.tiles = tilesBase; sp.f32 = elemBytes == 4 ? 1 : 0; sp.tile_map = e.band.map.get<int>();
            // the band's output rows land at the top of its (band-sized) output buffer
            sp.dst = e.staging.out.get<uint8_t>() - (size_t)b.yBegin * cw * 3; sp.pitch = (size_t)cw * 3;
            sp.y_begin = b.yBegin; sp.y_end = b.yEnd;
            launchStitch(sp, e.stream);
            ++e.launches;
            const size_t rows = (size_t)(b.yEnd - b.yBegin);
            if (rows)
                W2X_CUDA(cudaMemcpy2DAsync(dst + (size_t)b.yBegin * dstStride, dstStride, e.staging.out.get(), (size_t)cw * 3, (size_t)cw * 3, rows,
                                           cudaMemcpyDeviceToHost, e.stream));
        }
        for (int r = 0; r < bands; ++r) {
            W2X_CUDA(cudaSetDevice(es[r]->cfg.deviceId));
            W2X_CUDA(cudaStreamSynchronize(es[r]->stream));
        }
        return true;
    } catch (const std::exception& ex) {
        e0.log(W2X_ERROR, std::string("Row-band render failed unexpectedly: ") + ex.what() + ".", __FUNCTION__, __LINE__);
        return false;
    }
}

bool Engine::wait(int ticket) {
    try {
        if (ticket < 0 || ticket >= nextTicket) throw Error("invalid ticket");
        if (nextTicket - ticket > kSlots) return true;  // slot already recycled => that frame completed
        PipeSlot& ps = pipe[ticket % kSlots];
        if (ps.busy) { W2X_CUDA(cudaEventSynchronize(ps.evDone.get())); ps.busy = false; }
        return true;
    } catch (const std::exception& ex) {
        ELOG(W2X_ERROR, std::string("Wait failed: ") + ex.what() + ".");
        return false;
    }
}

bool Engine::sync() {
    try {
        if (h2dStream) W2X_CUDA(cudaStreamSynchronize(h2dStream));
        if (stream) W2X_CUDA(cudaStreamSynchronize(stream));
        if (d2hStream) W2X_CUDA(cudaStreamSynchronize(d2hStream));
        for (auto& s : pipe) s.busy = false;
        return true;
    } catch (const std::exception& ex) {
        ELOG(W2X_ERROR, std::string("Sync failed: ") + ex.what() + ".");
        return false;
    }
}

// Img2Img::infer-shaped entry (img2img_infer.cpp:41-93): NCHW f32 host -> NCHW f32 host.
bool Engine::infer(const float* inNchw, int n, float* outNchw) {
    try {
        if (!isLoaded) throw Error("no engine loaded");
        if (n < 1 || n > batch) {
            ELOG(W2X_ERROR, "Input has invalid batch size: expected " + std::to_string(batch) + ", got " + std::to_string(n) + ".");
            return false;
        }
        W2X_CUDA(cudaSetDevice(cfg.deviceId));
        const size_t inElems = (size_t)n * 3 * tile * tile, outElems = (size_t)n * 3 * outTile * outTile;
        DeviceBuffer in(inElems * 4), out(outElems * 4);
        DeviceBuffer outH((size_t)batch * outTile * outTile * 4 * elemBytes);  // model output, engine elements
        float *dIn = in.get<float>(), *dOut = out.get<float>();
        W2X_CUDA(cudaMemcpyAsync(dIn, inNchw, inElems * 4, cudaMemcpyHostToDevice, stream));
        W2X_CUDA(cudaMemsetAsync(actIn.p, 0, actIn.elems() * elemBytes, stream));
        if (tf32()) launchNchwToNhwc4(dIn, n, tile, reinterpret_cast<float*>(actIn.p), stream);
        else launchNchwToNhwc4(dIn, n, tile, actIn.p, stream);
        runModel(stream, outH.get(), n);
        if (tf32()) launchNhwc4ToNchw(outH.get<const float>(), n, outTile, dOut, stream);
        else launchNhwc4ToNchw(outH.get<const __half>(), n, outTile, dOut, stream);
        launches += 2;
        W2X_CUDA(cudaMemcpyAsync(outNchw, dOut, outElems * 4, cudaMemcpyDeviceToHost, stream));
        W2X_CUDA(cudaStreamSynchronize(stream));
        return true;
    } catch (const std::exception& ex) {
        ELOG(W2X_ERROR, std::string("Engine inference failed unexpectedly: ") + ex.what() + ".");
        return false;
    }
}

int Engine::profileLayers(int repeats, char (*names)[48], float* ms, double* flops, int cap) {
    try {
        if (!isLoaded) throw Error("no engine loaded");
        W2X_CUDA(cudaSetDevice(cfg.deviceId));
        CudaEvent ev0, ev1;
        cudaEvent_t e0 = ev0.get(), e1 = ev1.get();
        runModel(stream, nullptr);  // warm-up, and populates every activation
        W2X_CUDA(cudaStreamSynchronize(stream));
        int i = 0;
        for (auto& L : layers) {
            if (i >= cap) break;
            W2X_CUDA(cudaEventRecord(e0, stream));
            for (int r = 0; r < repeats; ++r) {
                if (L.seR) W2X_CUDA(cudaMemsetAsync(L.sePartial, 0, L.sePartialBytes, stream));
                launchLayer(L, stream, nullptr, batch);
                if (L.seR) launchSe(L, L.p.gn, stream);
            }
            W2X_CUDA(cudaEventRecord(e1, stream));
            W2X_CUDA(cudaEventSynchronize(e1));
            float t = 0;
            W2X_CUDA(cudaEventElapsedTime(&t, e0, e1));
            std::snprintf(names[i], 48, "%s", L.name.c_str());
            if (std::getenv("W2X_VERBOSE")) {
                char d[256] = "";
                layerKernel(i, d, sizeof(d));
                std::fprintf(stderr, "[w2x] %-28s %s\n", L.name.c_str(), d);
            }
            ms[i] = t / repeats;
            flops[i] = L.flops * batch;
            ++i;
        }
        return i;
    } catch (const std::exception& ex) {
        ELOG(W2X_ERROR, std::string("Profile failed: ") + ex.what() + ".");
        return -1;
    }
}

// ------------------------------------------------------------------------------------------------
// Single-layer test hooks (include/w2x_dev.h): one layer of the dense path on host data through the kernel the planner picks
// (`impl` 0), the dedicated head kernels (1) or the scalar CUDA-core reference kernel (2).
// ------------------------------------------------------------------------------------------------
static void convLayerGeometry(int kind, int n, int h, int w, int cin, int cout, int& npad, int& ktot, Act& out, Act& skip) {
    out = Act{};
    skip = Act{};
    if (kind == 0) { npad = (cout + 15) / 16 * 16; ktot = 9 * cin; out = {nullptr, n, h - 2, w - 2, cout}; }
    else if (kind == 1) { npad = (cout + 15) / 16 * 16; ktot = 4 * cin; out = {nullptr, n, h / 2, w / 2, cout}; }
    else if (kind == 2) { npad = 4 * cout; ktot = cin; out = {nullptr, n, 2 * h, 2 * w, cout}; skip = {nullptr, n, 2 * h + 8, 2 * w + 8, cout}; }
    else if (kind == 3) { npad = 16; ktot = 4 * cin; out = {nullptr, n, 2 * h - 4, 2 * w - 4, 4}; }
    else if (kind == 4) { npad = 16; ktot = 9 * cin; out = {nullptr, n, h - 2, w - 2, 4}; skip = {nullptr, n, h - 2 + 40, w - 2 + 40, 4}; }
    else throw Error("bad kind");
}

// The layer of `kind` on device copies of the host tensors, whose elements are `elemBytes` wide: fp16, or fp32 for the tf32 kernel (the
// ConvParams builders take the nominal fp16 pointer type of the engine's plan, see Act).  `bufs` owns the device memory; `out` is the
// zeroed output tensor.
static ConvParams uploadConvLayer(int kind, int n, int h, int w, int cin, int cout, size_t elemBytes, const void* in, const void* wPacked,
                                  const float* bias, const void* skipData, const void* outData, std::vector<DeviceBuffer>& bufs, Act& out) {
    int npad = 0, ktot = 0;
    Act skip{};
    convLayerGeometry(kind, n, h, w, cin, cout, npad, ktot, out, skip);
    if (!in || !wPacked || !bias || !outData || (skip.n && !skipData)) throw Error("null argument");
    auto dmal = [&](size_t bytes) { bufs.emplace_back(bytes + 256); return bufs.back().get(); };
    auto up = [&](const void* src, size_t bytes) { void* d = dmal(bytes); W2X_CUDA(cudaMemcpy(d, src, bytes, cudaMemcpyHostToDevice)); return d; };
    Act inA{nullptr, n, h, w, cin};
    inA.p = (__half*)up(in, inA.elems() * elemBytes);
    const __half* dWt = (const __half*)up(wPacked, (size_t)npad * ktot * elemBytes);
    const float* dB = (const float*)up(bias, (size_t)npad * 4);
    if (skip.n) skip.p = (__half*)up(skipData, skip.elems() * elemBytes);
    out.p = (__half*)dmal(out.elems() * elemBytes);
    W2X_CUDA(cudaMemset(out.p, 0, out.elems() * elemBytes));
    if (kind == 0) return makeConv3Params(inA, out, dWt, dB, npad, EPI_STORE, 0.1f, cout);
    if (kind == 1) return makeDown2Params(inA, out, dWt, dB, npad, 0.1f);
    if (kind == 2) return makeUp2Params(inA, out, dWt, dB, cout, 0.1f, &skip, 4);
    if (kind == 3) return makeUp4Params(inA, out, dWt, dB);
    ConvParams p = makeConv3Params(inA, out, dWt, dB, npad, EPI_FINAL, 1.f, 4);
    p.skip = skip.p; p.skip_h = skip.h; p.skip_w = skip.w; p.skip_c = 4; p.skip_off = 20;
    return p;
}

void runConvLayer(int device, int kind, int impl, int n, int h, int w, int cin, int cout, const uint16_t* in, const uint16_t* wPacked,
                  const float* bias, const uint16_t* skipData, uint16_t* outData) {
    W2X_CUDA(cudaSetDevice(device));
    std::vector<DeviceBuffer> bufs;
    Act out{};
    const ConvParams p = uploadConvLayer(kind, n, h, w, cin, cout, 2, in, wPacked, bias, skipData, outData, bufs, out);
    std::unique_ptr<IgemmPlan, void (*)(IgemmPlan*)> plan(nullptr, igemmDestroyPlan);
    std::unique_ptr<HeadPlan, void (*)(HeadPlan*)> hp(nullptr, convHeadDestroyPlan);
    if (impl == 2) {
        launchConvDirect(p, nullptr);
    } else if (impl == 1) {
        if (!convHeadSupported(p)) throw Error("no head kernel for this layer");
        hp.reset(convHeadCreatePlan(p));
        launchConvHead(hp.get(), nullptr);
    } else {
        plan.reset(igemmCreatePlan(p));
        // W2X_REPEAT (development build only): back-to-back launches, for steady-state clock / power readings of one layer
        const int reps = devEnv("W2X_REPEAT") ? std::max(1, std::atoi(devEnv("W2X_REPEAT"))) : 1;
        for (int r = 0; r < reps; ++r) igemmLaunch(plan.get(), nullptr, nullptr);
    }
    W2X_CUDA(cudaDeviceSynchronize());
    W2X_CUDA(cudaGetLastError());
    W2X_CUDA(cudaMemcpy(outData, out.p, out.elems() * 2, cudaMemcpyDeviceToHost));
}

void runConvLayerF32(int device, int kind, int n, int h, int w, int cin, int cout, const float* in, const float* wPacked, const float* bias,
                     const float* skipData, float* outData) {
    W2X_CUDA(cudaSetDevice(device));
    std::vector<DeviceBuffer> bufs;
    Act out{};
    const ConvParams p = uploadConvLayer(kind, n, h, w, cin, cout, 4, in, wPacked, bias, skipData, outData, bufs, out);
    std::unique_ptr<Tf32Plan, void (*)(Tf32Plan*)> plan(tf32CreatePlan(asF32(p)), tf32DestroyPlan);
    tf32Launch(plan.get(), nullptr);
    W2X_CUDA(cudaDeviceSynchronize());
    W2X_CUDA(cudaGetLastError());
    W2X_CUDA(cudaMemcpy(outData, out.p, out.elems() * 4, cudaMemcpyDeviceToHost));
}

// On-device self-check on random data: the tensor-core kernel vs the scalar CUDA-core reference kernel; returns max |diff|.
double selftestConv(int device, int kind, int n, int h, int w, int cin, int cout, unsigned seed) {
    const bool headKernel = kind == 5 || kind == 6;  // kinds 5 / 6: the layers of kinds 4 / 3 through the dedicated head kernels
    if (kind == 5) kind = 4;
    if (kind == 6) kind = 3;
    try {
        int npad = 0, ktot = 0;
        Act out{}, skip{};
        convLayerGeometry(kind, n, h, w, cin, cout, npad, ktot, out, skip);
        std::mt19937 rng(seed);
        std::uniform_real_distribution<float> U(-1.f, 1.f);
        auto randHalf = [&](size_t cnt, float scale_) {
            std::vector<uint16_t> v(cnt);
            for (auto& x : v) x = floatToHalfBits(U(rng) * scale_);
            return v;
        };
        const std::vector<uint16_t> inH = randHalf((size_t)n * h * w * cin, 1.f);
        std::vector<uint16_t> wh = randHalf((size_t)npad * ktot, 1.0f / std::sqrt((float)ktot));
        if (kind == 3 || kind == 4) {  // zero the padding columns like the packer does
            for (int nn = 0; nn < npad; ++nn) {
                const bool real = kind == 3 ? (nn % 4) < 3 : nn < 3;
                if (!real) for (int k = 0; k < ktot; ++k) wh[(size_t)nn * ktot + k] = 0;
            }
        }
        std::vector<float> bias(npad);
        for (int i = 0; i < npad; ++i) bias[i] = ((kind == 3 && (i % 4) == 3) || (kind == 4 && i >= 3)) ? 0.f : U(rng) * 0.1f;
        std::vector<uint16_t> skipH;
        if (skip.n) skipH = randHalf(skip.elems(), 0.5f);
        std::vector<uint16_t> ha(out.elems()), hb(out.elems());
        runConvLayer(device, kind, 2, n, h, w, cin, cout, inH.data(), wh.data(), bias.data(), skipH.empty() ? nullptr : skipH.data(), ha.data());
        runConvLayer(device, kind, headKernel ? 1 : 0, n, h, w, cin, cout, inH.data(), wh.data(), bias.data(), skipH.empty() ? nullptr : skipH.data(), hb.data());
        double md = 0, ma = 0;
        for (size_t i = 0; i < ha.size(); ++i) {
            const double a = halfBitsToFloat(ha[i]), b = halfBitsToFloat(hb[i]);
            md = std::max(md, std::fabs(a - b));
            ma = std::max(ma, std::fabs(a));
        }
        return (ma > 0) ? md : 1e9;  // an all-zero reference means the check itself is broken
    } catch (const std::exception& ex) {
        std::fprintf(stderr, "w2x selftest: %s\n", ex.what());
        return -1.0;
    }
}

}  // namespace w2x
