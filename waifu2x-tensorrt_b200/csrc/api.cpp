// extern "C" surface declared in include/w2x.h.  Nothing throws across this boundary.
#include <cuda_fp16.h>
#include <cuda_runtime.h>

#include <algorithm>
#include <cstring>
#include <filesystem>
#include <memory>

#include "engine.h"
#include "pool.h"
#include "../../include/w2x_dev.h"

using namespace w2x;

struct w2x_pool {
    EnginePool impl;
    w2x_pool(const int* d, int n) : impl(d, n) {}
};

namespace {
void setErr(char* err, int cap, const std::string& s) {
    if (err && cap > 0) {
        std::strncpy(err, s.c_str(), (size_t)cap - 1);
        err[cap - 1] = 0;
    }
}

// device memory for `count` elements of T, owned by `bufs`
template <class T> T* alloc(std::vector<DeviceBuffer>& bufs, size_t count) {
    bufs.emplace_back(count * sizeof(T) + 16);
    return bufs.back().get<T>();
}

// the stage hooks w2x_unpack_tiles(_u16) and w2x_stitch_tiles(_u16): a host frame of `format` <-> fp16 tiles on the device
int unpackTiles(const char* name, PixelFormat format, int device, const void* src, int width, int height, size_t src_stride, const w2x_rect* rects,
                const int* aug, int n, int tile, uint16_t* out) {
    try {
        W2X_CUDA(cudaSetDevice(device));
        std::vector<DeviceBuffer> b;
        const size_t row = (size_t)width * bytesPerPixel(format);
        uint8_t* dSrc = alloc<uint8_t>(b, row * height);
        W2X_CUDA(cudaMemcpy2D(dSrc, row, src, src_stride, row, height, cudaMemcpyHostToDevice));
        std::vector<TileSlot> slots(n);
        for (int i = 0; i < n; ++i) slots[i] = {rects[i].x, rects[i].y, aug ? aug[i] : 0, 1};
        TileSlot* dSlots = alloc<TileSlot>(b, n);
        W2X_CUDA(cudaMemcpy(dSlots, slots.data(), sizeof(TileSlot) * n, cudaMemcpyHostToDevice));
        const size_t elems = (size_t)n * tile * tile * 4;
        __half* dOut = alloc<__half>(b, elems);
        launchUnpack(dSrc, width, height, row, dSlots, n, tile, dOut, nullptr, format);
        W2X_CUDA(cudaGetLastError());
        W2X_CUDA(cudaMemcpy(out, dOut, elems * 2, cudaMemcpyDeviceToHost));
        return 1;
    } catch (const std::exception& ex) {
        std::fprintf(stderr, "%s: %s\n", name, ex.what());
        return 0;
    }
}

int stitchTiles(const char* name, PixelFormat format, int device, const uint16_t* tiles, int count, int out_tile, int nx, int ny, int overlap_x,
                int overlap_y, int canvas_w, int canvas_h, void* dst, size_t dst_stride) {
    try {
        W2X_CUDA(cudaSetDevice(device));
        std::vector<DeviceBuffer> b;
        const size_t elems = (size_t)count * out_tile * out_tile * 4;
        __half* dT = alloc<__half>(b, elems);
        W2X_CUDA(cudaMemcpy(dT, tiles, elems * 2, cudaMemcpyHostToDevice));
        std::vector<float> rx = blendRamp(overlap_x), ry = blendRamp(overlap_y);
        float* dRx = alloc<float>(b, rx.size() + 1);
        float* dRy = alloc<float>(b, ry.size() + 1);
        if (!rx.empty()) W2X_CUDA(cudaMemcpy(dRx, rx.data(), rx.size() * 4, cudaMemcpyHostToDevice));
        if (!ry.empty()) W2X_CUDA(cudaMemcpy(dRy, ry.data(), ry.size() * 4, cudaMemcpyHostToDevice));
        const size_t row = (size_t)canvas_w * bytesPerPixel(format);
        uint8_t* dDst = alloc<uint8_t>(b, row * canvas_h);
        StitchParams sp = stitchGrid(out_tile, nx, ny, overlap_x, overlap_y, canvas_w, canvas_h, dRx, dRy);
        sp.tiles = dT; sp.dst = dDst; sp.pitch = row; sp.format = format;
        launchStitch(sp, nullptr);
        W2X_CUDA(cudaGetLastError());
        W2X_CUDA(cudaMemcpy2D(dst, dst_stride, dDst, row, row, canvas_h, cudaMemcpyDeviceToHost));
        return 1;
    } catch (const std::exception& ex) {
        std::fprintf(stderr, "%s: %s\n", name, ex.what());
        return 0;
    }
}
}  // namespace

extern "C" {

void w2x_default_build_config(w2x_build_config* c) {
    if (!c) return;
    *c = w2x_build_config{0, W2X_PRECISION_FP16, 1, 1, 4, 3, 3, 3, 64, 256, 640, 64, 256, 640};  // config.h:12-31
}

void w2x_default_render_config(w2x_render_config* c) {
    if (!c) return;
    *c = w2x_render_config{0, W2X_PRECISION_FP16, 1, 3, 256, 256, 4, 0.0625, 0.0625, 0};  // config.h:33-43
}

w2x_engine* w2x_create(void) {
    try { return new w2x_engine(); } catch (...) { return nullptr; }
}

void w2x_destroy(w2x_engine* e) { delete e; }

void w2x_set_message_callback(w2x_engine* e, w2x_message_cb cb, void* user) { if (e) e->impl.setMessageCallback(cb, user); }
void w2x_set_progress_callback(w2x_engine* e, w2x_progress_cb cb, void* user) { if (e) e->impl.setProgressCallback(cb, user); }

int w2x_build(w2x_engine* e, const char* onnx_path, const w2x_build_config* cfg) {
    if (!e || !onnx_path || !cfg) return 0;
    return e->impl.build(onnx_path, *cfg) ? 1 : 0;
}

int w2x_load(w2x_engine* e, const char* onnx_path, const w2x_render_config* cfg) {
    if (!e || !onnx_path || !cfg) return 0;
    return e->impl.load(onnx_path, *cfg) ? 1 : 0;
}

int w2x_render(w2x_engine* e, const uint8_t* src, int width, int height, size_t src_stride, uint8_t* dst, size_t dst_stride) {
    if (!e) return 0;
    return e->impl.render(Frame{PixelFormat::Bgr8, src, width, height, src_stride, dst, dst_stride}) ? 1 : 0;
}

int w2x_render_bgra(w2x_engine* e, const uint8_t* src, int width, int height, size_t src_stride, uint8_t* dst, size_t dst_stride) {
    if (!e) return 0;
    return e->impl.render(Frame{PixelFormat::Bgra8, src, width, height, src_stride, dst, dst_stride}) ? 1 : 0;
}

int w2x_render_resized(w2x_engine* e, const uint8_t* src, int width, int height, size_t src_stride, uint8_t* dst, int dst_width, int dst_height,
                       size_t dst_stride) {
    if (!e) return 0;
    return e->impl.render(Frame{PixelFormat::Bgr8, src, width, height, src_stride, dst, dst_stride, Frame::Size{dst_width, dst_height}}) ? 1 : 0;
}

int w2x_submit_resized(w2x_engine* e, const uint8_t* src, int width, int height, size_t src_stride, uint8_t* dst, int dst_width, int dst_height,
                       size_t dst_stride) {
    if (!e) return -1;
    return e->impl.submit(Frame{PixelFormat::Bgr8, src, width, height, src_stride, dst, dst_stride, Frame::Size{dst_width, dst_height}});
}

int w2x_render_u16(w2x_engine* e, const uint16_t* src, int width, int height, size_t src_stride, uint16_t* dst, size_t dst_stride) {
    if (!e) return 0;
    return e->impl.render(Frame{PixelFormat::Bgr16, src, width, height, src_stride, dst, dst_stride}) ? 1 : 0;
}

int w2x_submit_u16(w2x_engine* e, const uint16_t* src, int width, int height, size_t src_stride, uint16_t* dst, size_t dst_stride) {
    if (!e) return -1;
    return e->impl.submit(Frame{PixelFormat::Bgr16, src, width, height, src_stride, dst, dst_stride});
}

int w2x_render_device(w2x_engine* e, const uint8_t* src, int width, int height, size_t src_stride, uint8_t* dst, size_t dst_stride) {
    if (!e) return 0;
    return e->impl.renderDevice(Frame{PixelFormat::Bgr8, src, width, height, src_stride, dst, dst_stride}) ? 1 : 0;
}

int w2x_submit(w2x_engine* e, const uint8_t* src, int width, int height, size_t src_stride, uint8_t* dst, size_t dst_stride) {
    if (!e) return -1;
    return e->impl.submit(Frame{PixelFormat::Bgr8, src, width, height, src_stride, dst, dst_stride});
}

int w2x_render_banded(w2x_engine* const* engines, int count, const uint8_t* src, int width, int height, size_t src_stride,
                      uint8_t* dst, size_t dst_stride) {
    if (!engines || count < 1 || count > 16) return 0;
    Engine* es[16];
    for (int i = 0; i < count; ++i) {
        if (!engines[i]) return 0;
        es[i] = &engines[i]->impl;
    }
    return Engine::renderBanded(es, count, Frame{PixelFormat::Bgr8, src, width, height, src_stride, dst, dst_stride}) ? 1 : 0;
}

w2x_pool* w2x_pool_create(const int* device_ids, int count) {
    try { return new w2x_pool(device_ids, count); } catch (...) { return nullptr; }
}
void w2x_pool_destroy(w2x_pool* p) { delete p; }
int w2x_pool_size(w2x_pool* p) { return p ? p->impl.size() : 0; }
w2x_engine* w2x_pool_engine(w2x_pool* p, int index) { return p ? p->impl.engine(index) : nullptr; }
void w2x_pool_set_message_callback(w2x_pool* p, w2x_message_cb cb, void* user) { if (p) p->impl.setMessageCallback(cb, user); }
int w2x_pool_build(w2x_pool* p, const char* onnx_path, const w2x_build_config* cfg) {
    try { return p && onnx_path && cfg && p->impl.build(onnx_path, *cfg) ? 1 : 0; } catch (...) { return 0; }
}
int w2x_pool_load(w2x_pool* p, const char* onnx_path, const w2x_render_config* cfg) {
    try { return p && onnx_path && cfg && p->impl.load(onnx_path, *cfg) ? 1 : 0; } catch (...) { return 0; }
}
int w2x_pool_submit(w2x_pool* p, const uint8_t* src, int width, int height, size_t src_stride, uint8_t* dst, size_t dst_stride) {
    if (!p) return -1;
    try { return p->impl.submit(Frame{PixelFormat::Bgr8, src, width, height, src_stride, dst, dst_stride}); } catch (...) { return -1; }
}
int w2x_pool_submit_resized(w2x_pool* p, const uint8_t* src, int width, int height, size_t src_stride, uint8_t* dst, int dst_width, int dst_height,
                            size_t dst_stride) {
    if (!p) return -1;
    if (dst_width < 1 || dst_height < 1) {   // the other refusals come from the engine that takes the frame, through w2x_pool_wait
        if (w2x_engine* e = p->impl.engine(0))
            e->impl.log(W2X_ERROR, "Submit failed: output size " + std::to_string(dst_width) + "x" + std::to_string(dst_height) + " is below 1x1.",
                        __FUNCTION__, __LINE__);
        return -1;
    }
    try {
        return p->impl.submit(Frame{PixelFormat::Bgr8, src, width, height, src_stride, dst, dst_stride, Frame::Size{dst_width, dst_height}});
    } catch (...) {
        return -1;
    }
}
int w2x_pool_submit_u16(w2x_pool* p, const uint16_t* src, int width, int height, size_t src_stride, uint16_t* dst, size_t dst_stride) {
    if (!p) return -1;   // the refusals come from the engine that takes the frame, through w2x_pool_wait
    try { return p->impl.submit(Frame{PixelFormat::Bgr16, src, width, height, src_stride, dst, dst_stride}); } catch (...) { return -1; }
}
int w2x_pool_wait(w2x_pool* p, int ticket) {
    try { return p && p->impl.wait(ticket) ? 1 : 0; } catch (...) { return 0; }
}
int w2x_pool_sync(w2x_pool* p) {
    try { return p && p->impl.sync() ? 1 : 0; } catch (...) { return 0; }
}

int w2x_wait(w2x_engine* e, int ticket) { return e && e->impl.wait(ticket) ? 1 : 0; }
int w2x_sync(w2x_engine* e) { return e && e->impl.sync() ? 1 : 0; }

void* w2x_host_alloc(size_t bytes) {
    void* p = nullptr;
    if (cudaHostAlloc(&p, bytes ? bytes : 1, cudaHostAllocPortable) != cudaSuccess) return nullptr;
    return p;
}
void w2x_host_free(void* p) { if (p) cudaFreeHost(p); }

void* w2x_device_alloc(w2x_engine* e, size_t bytes) {
    if (!e || cudaSetDevice(e->impl.device()) != cudaSuccess) return nullptr;
    void* p = nullptr;
    if (cudaMalloc(&p, bytes ? bytes : 1) != cudaSuccess) return nullptr;
    return p;
}
void w2x_device_free(w2x_engine* e, void* p) {
    if (e) cudaSetDevice(e->impl.device());
    if (p) cudaFree(p);
}
int w2x_memcpy_h2d(w2x_engine* e, void* dst, const void* src, size_t bytes) {
    if (!e || cudaSetDevice(e->impl.device()) != cudaSuccess) return 0;
    return cudaMemcpy(dst, src, bytes, cudaMemcpyHostToDevice) == cudaSuccess;
}
int w2x_memcpy_d2h(w2x_engine* e, void* dst, const void* src, size_t bytes) {
    if (!e || cudaSetDevice(e->impl.device()) != cudaSuccess) return 0;
    return cudaMemcpy(dst, src, bytes, cudaMemcpyDeviceToHost) == cudaSuccess;
}

const char* w2x_last_error(w2x_engine* e) { return e ? e->impl.lastError() : "null engine"; }
int w2x_output_tile_size(w2x_engine* e) { return e ? e->impl.outputTile() : 0; }
long long w2x_launch_count(w2x_engine* e) { return e ? e->impl.launchCount() : 0; }
double w2x_model_flops_per_tile(w2x_engine* e) { return e ? e->impl.flopsPerTile() : 0.0; }
int w2x_last_stage_ms(w2x_engine* e, float* out, int n) { return e && out ? e->impl.lastStageMs(out, n) : 0; }
int w2x_timer_mark(w2x_engine* e, int idx, int which) { return e && e->impl.timerMark(idx, which) ? 1 : 0; }
float w2x_timer_elapsed_ms(w2x_engine* e, int i0, int i1) { return e ? e->impl.timerElapsedMs(i0, i1) : -1.f; }
int w2x_profile_layers(w2x_engine* e, int repeats, char (*names)[48], float* ms, double* flops, int n) {
    return e ? e->impl.profileLayers(repeats < 1 ? 1 : repeats, names, ms, flops, n) : -1;
}
int w2x_layer_kernel(w2x_engine* e, int index, char* buf, int cap) { return e && buf && cap > 0 ? e->impl.layerKernel(index, buf, cap) : 0; }
long long w2x_layer_tensor(w2x_engine* e, int index, int which, void* dst, size_t cap, int* dims) {
    return e ? e->impl.layerTensor(index, which, dst, cap, dims) : -1;
}
int w2x_infer(w2x_engine* e, const float* in, int n, float* out) { return e && in && out && e->impl.infer(in, n, out) ? 1 : 0; }

// ---- stage entry points ---------------------------------------------------------------------------------
int w2x_calculate_tiles(int in_w, int in_h, int out_w, int out_h, int tile_w, int tile_h, int out_tile_w, int out_tile_h,
                        int scaling, double overlap_x, double overlap_y, w2x_rect* in_rects, w2x_rect* out_rects, int cap,
                        int* grid_out) {
    try {
        TileGrid g = calculateTiles(in_w, in_h, out_w, out_h, tile_w, tile_h, out_tile_w, out_tile_h, scaling, overlap_x, overlap_y);
        for (int i = 0; i < g.count && i < cap; ++i) {
            if (in_rects) in_rects[i] = g.inRects[i];
            if (out_rects) out_rects[i] = g.outRects[i];
        }
        if (grid_out) {
            const int v[8] = {g.nx, g.ny, g.scaledInW, g.scaledInH, g.inOvX, g.inOvY, g.outOvX, g.outOvY};
            std::memcpy(grid_out, v, sizeof(v));
        }
        return g.count;
    } catch (...) {
        return -1;
    }
}

int w2x_blend_ramp(int overlap, float* ramp) {
    if (overlap < 0) return -1;
    std::vector<float> r = blendRamp(overlap);
    if (ramp) std::memcpy(ramp, r.data(), r.size() * sizeof(float));
    return (int)r.size();
}

int w2x_unpack_tiles(int device, const uint8_t* src, int width, int height, size_t src_stride, const w2x_rect* rects,
                     const int* aug, int n, int tile, uint16_t* out) {
    if (!src || !rects || !out || n <= 0 || tile <= 0) return 0;
    return unpackTiles("w2x_unpack_tiles", PixelFormat::Bgr8, device, src, width, height, src_stride, rects, aug, n, tile, out);
}

int w2x_stitch_tiles(int device, const uint16_t* tiles, int count, int out_tile, int nx, int ny, int overlap_x, int overlap_y,
                     int canvas_w, int canvas_h, uint8_t* dst, size_t dst_stride) {
    if (!tiles || !dst || count != nx * ny) return 0;
    return stitchTiles("w2x_stitch_tiles", PixelFormat::Bgr8, device, tiles, count, out_tile, nx, ny, overlap_x, overlap_y, canvas_w, canvas_h, dst,
                       dst_stride);
}

int w2x_unpack_tiles_u16(int device, const uint16_t* src, int width, int height, size_t src_stride, const w2x_rect* rects, const int* aug, int n,
                         int tile, uint16_t* out) {
    if (!src || !rects || !out || n <= 0 || tile <= 0 || width <= 0 || height <= 0 || src_stride < (size_t)width * 6) return 0;
    return unpackTiles("w2x_unpack_tiles_u16", PixelFormat::Bgr16, device, src, width, height, src_stride, rects, aug, n, tile, out);
}

int w2x_stitch_tiles_u16(int device, const uint16_t* tiles, int count, int out_tile, int nx, int ny, int overlap_x, int overlap_y,
                         int canvas_w, int canvas_h, uint16_t* dst, size_t dst_stride) {
    if (!tiles || !dst || count != nx * ny || canvas_w <= 0 || canvas_h <= 0 || dst_stride < (size_t)canvas_w * 6) return 0;
    return stitchTiles("w2x_stitch_tiles_u16", PixelFormat::Bgr16, device, tiles, count, out_tile, nx, ny, overlap_x, overlap_y, canvas_w, canvas_h,
                       dst, dst_stride);
}

int w2x_alpha_bleed(int device, const uint8_t* src, int width, int height, size_t src_stride, int rounds, uint8_t* dst) {
    try {
        if (!src || !dst || width <= 0 || height <= 0 || src_stride < (size_t)width * 4 || rounds < 0) throw Error("invalid argument");
        W2X_CUDA(cudaSetDevice(device));
        std::vector<DeviceBuffer> b;
        const size_t row = (size_t)width * 4, bytes = row * height;
        uint8_t* dSrc = alloc<uint8_t>(b, bytes);
        uint8_t* dBuf[2] = {alloc<uint8_t>(b, bytes), alloc<uint8_t>(b, bytes)};
        W2X_CUDA(cudaMemcpy2D(dSrc, row, src, src_stride, row, height, cudaMemcpyHostToDevice));
        const uint8_t* in = dSrc;
        for (int r = 0; r < std::max(rounds, 1); ++r) {   // the engine's sequence (Engine::renderOnStream)
            launchAlphaBleedRound(in, dBuf[r & 1], width, height, rounds > 0 ? 1 : 0, r + 1 >= rounds ? dSrc : nullptr, nullptr);
            in = dBuf[r & 1];
        }
        W2X_CUDA(cudaGetLastError());
        W2X_CUDA(cudaMemcpy(dst, in, bytes, cudaMemcpyDeviceToHost));
        return 1;
    } catch (const std::exception& ex) {
        std::fprintf(stderr, "w2x_alpha_bleed: %s\n", ex.what());
        return 0;
    }
}

int w2x_resample(int device, const uint8_t* src, int width, int height, size_t src_stride, uint8_t* dst, int dst_width, int dst_height,
                 size_t dst_stride) {
    try {
        if (!src || !dst || width <= 0 || height <= 0 || src_stride < (size_t)width * 3 || dst_width < 1 || dst_width > width || dst_height < 1 ||
            dst_height > height || dst_stride < (size_t)dst_width * 3)
            throw Error("invalid argument");
        W2X_CUDA(cudaSetDevice(device));
        const ResampleAxis axes[2] = {resampleAxis(width, dst_width), resampleAxis(height, dst_height)};
        std::vector<DeviceBuffer> b;
        ResampleTable t[2];
        for (int a = 0; a < 2; ++a) {
            const ResampleAxis& ax = axes[a];
            int* first = alloc<int>(b, ax.nOut);
            int* count = alloc<int>(b, ax.nOut);
            float* w = alloc<float>(b, ax.w.size());
            W2X_CUDA(cudaMemcpy(first, ax.first.data(), ax.nOut * sizeof(int), cudaMemcpyHostToDevice));
            W2X_CUDA(cudaMemcpy(count, ax.count.data(), ax.nOut * sizeof(int), cudaMemcpyHostToDevice));
            W2X_CUDA(cudaMemcpy(w, ax.w.data(), ax.w.size() * sizeof(float), cudaMemcpyHostToDevice));
            t[a] = {first, count, w, ax.taps};
        }
        const size_t row = (size_t)width * 3, orow = (size_t)dst_width * 3;
        uint8_t* dSrc = alloc<uint8_t>(b, row * height);
        float* dTmp = alloc<float>(b, (size_t)height * orow);
        uint8_t* dDst = alloc<uint8_t>(b, orow * dst_height);
        W2X_CUDA(cudaMemcpy2D(dSrc, row, src, src_stride, row, height, cudaMemcpyHostToDevice));
        launchResampleH(dSrc, row, 0, height, t[0], dst_width, dTmp, nullptr);   // the engine's sequence (Engine::renderOnStream)
        launchResampleV(dTmp, dst_width, t[1], 0, dst_height, dDst, orow, nullptr);
        W2X_CUDA(cudaGetLastError());
        W2X_CUDA(cudaMemcpy2D(dst, dst_stride, dDst, orow, orow, dst_height, cudaMemcpyDeviceToHost));
        return 1;
    } catch (const std::exception& ex) {
        std::fprintf(stderr, "w2x_resample: %s\n", ex.what());
        return 0;
    }
}

int w2x_resample_table(int n_in, int n_out, int* first, int* count, float* weights, size_t cap) {
    try {
        const ResampleAxis ax = resampleAxis(n_in, n_out);
        if (weights) {
            if (!first || !count || cap < ax.w.size()) throw Error("weights capacity below n_out * taps");
            std::memcpy(first, ax.first.data(), ax.first.size() * sizeof(int));
            std::memcpy(count, ax.count.data(), ax.count.size() * sizeof(int));
            std::memcpy(weights, ax.w.data(), ax.w.size() * sizeof(float));
        }
        return ax.taps;
    } catch (const std::exception& ex) {
        std::fprintf(stderr, "w2x_resample_table: %s\n", ex.what());
        return 0;
    }
}

int w2x_tta_reduce(int device, const uint16_t* outs, int tiles, int out_tile, float* mean) {
    try {
        if (!outs || !mean || tiles <= 0) return 0;
        W2X_CUDA(cudaSetDevice(device));
        std::vector<DeviceBuffer> b;
        const size_t plane = (size_t)out_tile * out_tile * 4;
        __half* dIn = alloc<__half>(b, plane * 8 * tiles);
        float* dOut = alloc<float>(b, plane * tiles);
        W2X_CUDA(cudaMemcpy(dIn, outs, plane * 8 * tiles * 2, cudaMemcpyHostToDevice));
        launchTtaReduce(dIn, tiles, out_tile, dOut, nullptr);
        W2X_CUDA(cudaGetLastError());
        W2X_CUDA(cudaMemcpy(mean, dOut, plane * tiles * 4, cudaMemcpyDeviceToHost));
        return 1;
    } catch (const std::exception& ex) {
        std::fprintf(stderr, "w2x_tta_reduce: %s\n", ex.what());
        return 0;
    }
}

double w2x_selftest_conv(int device, int kind, int n, int h, int w, int cin, int cout, unsigned seed) {
    try {
        return selftestConv(device, kind, n, h, w, cin, cout, seed);
    } catch (...) {
        return -1.0;
    }
}

int w2x_run_conv_layer(int device, int kind, int head, int n, int h, int w, int cin, int cout, const uint16_t* in_nhwc, const uint16_t* weights,
                       const float* bias, const uint16_t* skip_nhwc, uint16_t* out_nhwc) {
    try {
        runConvLayer(device, kind, head ? 1 : 0, n, h, w, cin, cout, in_nhwc, weights, bias, skip_nhwc, out_nhwc);
        return 1;
    } catch (const std::exception& ex) {
        std::fprintf(stderr, "w2x_run_conv_layer: %s\n", ex.what());
        return 0;
    }
}

int w2x_run_conv_layer_f32(int device, int kind, int n, int h, int w, int cin, int cout, const float* in_nhwc, const float* weights, const float* bias,
                           const float* skip_nhwc, float* out_nhwc) {
    try {
        runConvLayerF32(device, kind, n, h, w, cin, cout, in_nhwc, weights, bias, skip_nhwc, out_nhwc);
        return 1;
    } catch (const std::exception& ex) {
        std::fprintf(stderr, "w2x_run_conv_layer_f32: %s\n", ex.what());
        return 0;
    }
}

int w2x_run_swin_mlp(int device, long long tokens, int c, int variant, uint16_t* x, const float* gamma, const float* beta, float eps, const uint16_t* w1,
                     const float* b1, const uint16_t* w2, const float* b2, int reps, float* ms_out) {
    try {
        if (tokens < 1 || !x || !gamma || !beta || !w1 || !b1 || !w2 || !b2 || !swinMlpSupported(c, 2 * c)) throw Error("invalid argument");
        W2X_CUDA(cudaSetDevice(device));
        const size_t C = (size_t)c;
        const size_t sizes[7] = {(size_t)tokens * C * 2, C * 4, C * 4, 2 * C * C * 2, 2 * C * 4, 2 * C * C * 2, C * 4};
        const void* host[7] = {x, gamma, beta, w1, b1, w2, b2};
        DeviceBuffer bufs[7];
        for (int i = 0; i < 7; ++i) {
            bufs[i].ensure(sizes[i]);
            W2X_CUDA(cudaMemcpy(bufs[i].get(), host[i], sizes[i], cudaMemcpyHostToDevice));
        }
        std::unique_ptr<SwinMlpPlan, void (*)(SwinMlpPlan*)> plan(
            swinMlpCreatePlan(bufs[0].get<__half>(), c, bufs[1].get<const float>(), bufs[2].get<const float>(), eps, bufs[3].get<const __half>(),
                              bufs[4].get<const float>(), bufs[5].get<const __half>(), bufs[6].get<const float>(), variant),
            swinMlpDestroyPlan);
        swinMlpLaunch(plan.get(), nullptr, tokens);
        W2X_CUDA(cudaDeviceSynchronize());
        W2X_CUDA(cudaMemcpy(x, bufs[0].get(), sizes[0], cudaMemcpyDeviceToHost));
        if (ms_out && reps > 0) {
            CudaEvent ev0, ev1;
            cudaEvent_t e0 = ev0.get(), e1 = ev1.get();
            W2X_CUDA(cudaEventRecord(e0, nullptr));
            for (int i = 0; i < reps; ++i) swinMlpLaunch(plan.get(), nullptr, tokens);
            W2X_CUDA(cudaEventRecord(e1, nullptr));
            W2X_CUDA(cudaEventSynchronize(e1));
            W2X_CUDA(cudaEventElapsedTime(ms_out, e0, e1));
            *ms_out /= (float)reps;
        }
        return 1;
    } catch (const std::exception& ex) {
        std::fprintf(stderr, "w2x_run_swin_mlp: %s\n", ex.what());
        return 0;
    }
}

// host-only hooks for the CPU test suite: the operand preparation of the fused Swin kernels
int w2x_swin_attn_prepare(const uint16_t* wqkv, const float* bqkv, const float* relpos, int c, int heads, uint16_t* w_out, float* b_out, float* rel_out) {
    try {
        if (!wqkv || !bqkv || !relpos || !w_out || !b_out || !rel_out) throw Error("invalid argument");
        std::vector<uint16_t> w;
        std::vector<float> b, r;
        swinAttnPrepare(wqkv, bqkv, relpos, c, heads, w, b, r);
        std::memcpy(w_out, w.data(), w.size() * 2);
        std::memcpy(b_out, b.data(), b.size() * 4);
        std::memcpy(rel_out, r.data(), r.size() * 4);
        return (int)(r.size() / ((size_t)heads * 36));   // floats per bias-table row
    } catch (const std::exception& ex) {
        std::fprintf(stderr, "w2x_swin_attn_prepare: %s\n", ex.what());
        return 0;
    }
}

int w2x_compose_up_to_image(const uint16_t* w_up, const float* b_up, const uint16_t* w_img, const float* b_img, int cmid, int k, uint16_t* w_out, float* b_out) {
    try {
        if (!w_up || !b_up || !w_img || !b_img || !w_out || !b_out || cmid < 1 || k < 1) throw Error("invalid argument");
        PackedLayer U, L;
        U.kind = L_UPLIN; U.cout = (uint32_t)cmid; U.npad = 4u * (uint32_t)cmid; U.ktot = (uint32_t)k;
        U.w.assign(w_up, w_up + (size_t)4 * cmid * k);
        U.bias.assign(b_up, b_up + (size_t)4 * cmid);
        L.kind = L_TOIMG; L.cout = 3; L.npad = 16; L.ktot = (uint32_t)cmid; L.upscale = 2;
        L.w.assign(w_img, w_img + (size_t)16 * cmid);
        L.bias.assign(b_img, b_img + 16);
        std::vector<uint16_t> w;
        std::vector<float> b;
        composeUpToImage(U, L, w, b);
        std::memcpy(w_out, w.data(), w.size() * 2);
        std::memcpy(b_out, b.data(), b.size() * 4);
        return 1;
    } catch (const std::exception& ex) {
        std::fprintf(stderr, "w2x_compose_up_to_image: %s\n", ex.what());
        return 0;
    }
}

int w2x_run_swin_attn(int device, int n, int h, int w, int c, int heads, int shift, uint16_t* x, const float* gamma, const float* beta, float eps, const uint16_t* wqkv,
                      const float* bqkv, const uint16_t* wproj, const float* bproj, const float* relpos, int reps, float* ms_out) {
    try {
        if (n < 1 || !x || !gamma || !beta || !wqkv || !bqkv || !relpos || !swinAttnSupported(c, heads, 6, h, w)) throw Error("invalid argument");
        const bool fuseProj = swinAttnFusesProj(c);
        if (fuseProj && (!wproj || !bproj)) throw Error("invalid argument");
        W2X_CUDA(cudaSetDevice(device));
        std::vector<uint16_t> wR;
        std::vector<float> bR, relR;
        swinAttnPrepare(wqkv, bqkv, relpos, c, heads, wR, bR, relR);
        const size_t C = (size_t)c;
        const size_t sizes[8] = {(size_t)n * h * w * C * 2, C * 4, C * 4, wR.size() * 2, bR.size() * 4, C * C * 2, C * 4, relR.size() * 4};
        const void* host[8] = {x, gamma, beta, wR.data(), bR.data(), wproj, bproj, relR.data()};
        DeviceBuffer bufs[9];
        for (int i = 0; i < 8; ++i) {
            if (!host[i]) continue;   // wproj / bproj of the variant that stops at the attention output
            bufs[i].ensure(sizes[i]);
            W2X_CUDA(cudaMemcpy(bufs[i].get(), host[i], sizes[i], cudaMemcpyHostToDevice));
        }
        if (!fuseProj) {
            bufs[8].ensure(sizes[0]);
            W2X_CUDA(cudaMemset(bufs[8].get(), 0, sizes[0]));
        }
        W2X_CUDA(cudaDeviceSynchronize());
        std::unique_ptr<SwinAttnPlan, void (*)(SwinAttnPlan*)> plan(
            swinAttnCreatePlan(bufs[0].get<__half>(), n, h, w, c, heads, 6, shift, bufs[1].get<const float>(), bufs[2].get<const float>(), eps,
                               bufs[3].get<const __half>(), bufs[4].get<const float>(), bufs[5].get<const __half>(), bufs[6].get<const float>(),
                               bufs[7].get<const float>(), bufs[8].get<__half>()),
            swinAttnDestroyPlan);
        swinAttnLaunch(plan.get(), nullptr, n);
        W2X_CUDA(cudaDeviceSynchronize());
        W2X_CUDA(cudaMemcpy(x, bufs[fuseProj ? 0 : 8].get(), sizes[0], cudaMemcpyDeviceToHost));
        if (ms_out && reps > 0) {
            CudaEvent ev0, ev1;
            cudaEvent_t e0 = ev0.get(), e1 = ev1.get();
            W2X_CUDA(cudaEventRecord(e0, nullptr));
            for (int i = 0; i < reps; ++i) swinAttnLaunch(plan.get(), nullptr, n);
            W2X_CUDA(cudaEventRecord(e1, nullptr));
            W2X_CUDA(cudaEventSynchronize(e1));
            W2X_CUDA(cudaEventElapsedTime(ms_out, e0, e1));
            *ms_out /= (float)reps;
        }
        return 1;
    } catch (const std::exception& ex) {
        std::fprintf(stderr, "w2x_run_swin_attn: %s\n", ex.what());
        return 0;
    }
}

#ifdef W2X_DEV
int w2x_probe_umma(int device, int mode, int pitch, float* err9) {
    try {
        if (!err9 || cudaSetDevice(device) != cudaSuccess) return -1;
        return probeUmma(mode, pitch, err9);
    } catch (...) {
        return -2;
    }
}

float w2x_probe_mma_rate(int device, int n, int iters, int sbo_a) {
    if (cudaSetDevice(device) != cudaSuccess) return -1.f;
    try { return probeMmaRate(n, iters, sbo_a); } catch (...) { return -3.f; }
}

float w2x_probe_hmma_rate(int device, int warps, int chains, int iters) {
    if (cudaSetDevice(device) != cudaSuccess) return -1.f;
    try { return probeHmmaRate(warps, chains, iters); } catch (...) { return -3.f; }
}

int w2x_probe_mma_rate_stream(int device, int n, int iters, int stream_bytes, float* res) {
    if (!res || cudaSetDevice(device) != cudaSuccess) return -1;
    try { return probeMmaRateStream(n, iters, stream_bytes, res); } catch (...) { return -3; }
}

float w2x_probe_mma_tiles(int device, int tiles, int mode) {
    if (cudaSetDevice(device) != cudaSuccess) return -1.f;
    try { return probeMmaTiles(tiles, mode); } catch (...) { return -3.f; }
}

float w2x_probe_l2_stream(int device, int bytes, int iters) {
    if (cudaSetDevice(device) != cudaSuccess) return -1.f;
    try { return probeL2Stream(bytes, iters); } catch (...) { return -3.f; }
}
#endif  // W2X_DEV

void w2x_config_hash(const char* device_name, const w2x_build_config* cfg, char out_hex[65]) {
    if (!out_hex) return;
    out_hex[0] = 0;
    if (!device_name || !cfg) return;
    const std::string h = configHash(device_name, *cfg);
    std::memcpy(out_hex, h.c_str(), 65);
}

int w2x_pack_onnx(const char* onnx_path, const char* out_path, int precision, char* err, int cap) {
    try {
        if (!onnx_path || !out_path) throw Error("null path");
        OnnxGraph g = parseOnnx(readFile(onnx_path));
        PackedModel pm = packFromOnnx(g, precision);
        const std::vector<uint8_t> blob = serializePack(pm);
        writeFile(out_path, blob.data(), blob.size());
        return 1;
    } catch (const std::exception& ex) {
        setErr(err, cap, ex.what());
        return 0;
    }
}

int w2x_select_engine(const char* model_path, const w2x_render_config* cfg, const char* device_name, char* out_path, size_t cap) {
    if (!model_path || !cfg || !device_name || !out_path || cap == 0) return 0;
    try {
        const std::string p = selectEngine(model_path, *cfg, device_name);
        std::snprintf(out_path, cap, "%s", p.c_str());
        return p.size() < cap ? 1 : 0;
    } catch (const std::exception& ex) {
        std::snprintf(out_path, cap, "%s", ex.what());
        return 0;
    }
}

int w2x_pack_info(const char* pack_path, int* arch, int* scale, int* offset, int* layers) {
    try {
        PackedModel pm = deserializePack(readFile(pack_path));
        if (arch) *arch = (int)pm.arch;
        if (scale) *scale = (int)pm.scale;
        if (offset) *offset = (int)pm.offset;
        if (layers) *layers = (int)pm.layers.size();
        return 1;
    } catch (...) {
        return 0;
    }
}

}  // extern "C"
