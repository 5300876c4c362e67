/*
 * w2x.h — C ABI of the B200-native waifu2x engine (drop-in for the reference's operator surface).
 *
 * The reference has no FFI layer: its operator surface is the C++ class trt::Img2Img
 * (/root/reference/src/tensorrt/img2img.h:14-50), its config PODs (src/tensorrt/config.h:7-43) and
 * two callback typedefs (src/tensorrt/logger.h:20-21).  Every entry point below names the reference
 * interface it replaces.  Plain pointers and sizes only; nothing throws across this boundary: like
 * the reference's function-try-blocks (img2img_build.cpp:54,170-173; img2img_load.cpp:117,288-291;
 * img2img_render.cpp:224,349-352) failures are logged through the message callback at `error`
 * severity and reported as a 0 ("false") return.  1 == true == success.
 *
 * A header-only C++ shim that re-creates trt::Img2Img on top of this ABI lives in
 * waifu2x-tensorrt_b200/host/img2img.hpp; the Python (ctypes) binding in waifu2x-tensorrt_b200/w2x/.
 */
#ifndef W2X_H
#define W2X_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define W2X_API __attribute__((visibility("default")))

/* trt::Precision, src/tensorrt/config.h:7-10 (same enumerator order). */
enum { W2X_PRECISION_TF32 = 0, W2X_PRECISION_FP16 = 1 };

/* trt::Severity, src/tensorrt/logger.h:11-18. */
enum { W2X_CRITICAL = 0, W2X_ERROR = 1, W2X_WARN = 2, W2X_INFO = 3, W2X_DEBUG = 4, W2X_TRACE = 5 };

/* trt::BuildConfig, src/tensorrt/config.h:12-31 (same fields, same defaults via w2x_default_build_config). */
typedef struct w2x_build_config {
    int deviceId;
    int precision;
    int minBatchSize, optBatchSize, maxBatchSize;
    int minChannels, optChannels, maxChannels;
    int minWidth, optWidth, maxWidth;
    int minHeight, optHeight, maxHeight;
} w2x_build_config;

/* trt::RenderConfig, src/tensorrt/config.h:33-43; cv::Point2d overlap becomes two doubles
 * (fractions of the INPUT tile size, img2img_render.cpp:21-29). */
typedef struct w2x_render_config {
    int deviceId;
    int precision;
    int batchSize;
    int channels;
    int height;
    int width;
    int scaling;
    double overlapX, overlapY;
    int tta;
} w2x_render_config;

/* cv::Rect2i */
typedef struct w2x_rect { int x, y, width, height; } w2x_rect;

typedef struct w2x_engine w2x_engine;

/* trt::MessageCallback / trt::ProgressCallback, src/tensorrt/logger.h:20-21, with a user pointer. */
typedef void (*w2x_message_cb)(int severity, const char* message, void* user);
typedef void (*w2x_progress_cb)(int current, int total, double speed, void* user);

W2X_API void w2x_default_build_config(w2x_build_config* cfg);   /* config.h:12-31 defaults */
W2X_API void w2x_default_render_config(w2x_render_config* cfg); /* config.h:33-43 defaults */

/* trt::Img2Img::Img2Img / ~Img2Img (img2img_base.cpp:3-10): the object owns all device memory. */
W2X_API w2x_engine* w2x_create(void);
W2X_API void w2x_destroy(w2x_engine* e);

/* Img2Img::setMessageCallback / setProgressCallback (img2img_base.cpp:12-17). */
W2X_API void w2x_set_message_callback(w2x_engine* e, w2x_message_cb cb, void* user);
W2X_API void w2x_set_progress_callback(w2x_engine* e, w2x_progress_cb cb, void* user);

/* Img2Img::build (img2img_build.cpp:54-173): ONNX -> `<stem>_<sha256(cfg)[:16]>.w2x` + `.json` sidecar next
 * to the ONNX file (same naming rule :151-154, same json keys :29-50; the plan is kernel-native packed
 * weights instead of a TensorRT plan).  Needs the CUDA device (device name is part of the hash, :8-27). */
W2X_API int w2x_build(w2x_engine* e, const char* onnx_path, const w2x_build_config* cfg);

/* Img2Img::load (img2img_load.cpp:117-291): takes the ONNX path, finds the engine file itself
 * (getEnginePath :79-114, isCompatible/isOptimized :9-27), allocates workspaces, streams, blend ramps. */
W2X_API int w2x_load(w2x_engine* e, const char* onnx_path, const w2x_render_config* cfg);

/* Img2Img::render (img2img_render.cpp:224-348): src CV_8UC3 BGR HWC (w x h, row pitch src_stride bytes) ->
 * dst CV_8UC3 BGR (w*scaling x h*scaling, row pitch dst_stride).  Caller owns both host buffers
 * (main.cpp:228-235).  Synchronous: dst is complete on return (the reference's missing sync, SURVEY q9, fixed). */
W2X_API int w2x_render(w2x_engine* e, const uint8_t* src_bgr, int width, int height, size_t src_stride,
                       uint8_t* dst_bgr, size_t dst_stride);

/* ---- extensions (not in the reference) ------------------------------------------------------------- */

/* Images with an alpha channel: src BGRA u8 HWC (w x h, row pitch src_stride >= 4 * width) -> dst BGRA (w*scaling x h*scaling, pitch
 * dst_stride >= 4 * width * scaling), synchronous, with any loaded engine (fp16 or tf32, with or without TTA).
 *  - Every alpha byte 255: B, G, R are byte-identical to w2x_render of the B, G, R planes, alpha is 255, and the model runs once.
 *  - Some alpha byte 0: before the model, the colour of the transparent pixels (alpha == 0) is replaced by a bleed of the visible
 *    colour: `offset / scale` rounds (the model's input border, w2x_pack_info), each of which gives every transparent pixel with a
 *    known 8-neighbour the rounded-half-up integer mean of its known neighbours; pixels still unknown become (0, 0, 0).  So the
 *    colour under alpha == 0 never reaches the output.  B, G, R out are w2x_render of the bled frame.
 *  - Some alpha byte < 255: the alpha plane goes through the same model, tiles, TTA and blending as a grey image (B = G = R = alpha),
 *    in the same batches as the colour tiles; output alpha = saturate(rint(255 * (r + g + b) / 3)) of its blended canvas.
 * Returns 0 and logs the reason on failure (no engine loaded, null pointers, strides below 4 bytes per pixel). */
W2X_API int w2x_render_bgra(w2x_engine* e, const uint8_t* src_bgra, int width, int height, size_t src_stride,
                            uint8_t* dst_bgra, size_t dst_stride);

/* Output at any size up to the model's: src BGR u8 HWC (w x h, pitch src_stride >= 3 * width) -> dst BGR u8 (dst_width x dst_height,
 * pitch dst_stride >= 3 * dst_width), synchronous, with any loaded engine, for 1 <= dst_width <= width * scaling and
 * 1 <= dst_height <= height * scaling.  Let C be the canvas w2x_render returns for src (width * scaling x height * scaling).  Then, per
 * channel, with the u8 values of C taken as reals:
 *     dst = clamp(rint(R_y(R_x(C))), 0, 255)
 * where R is the antialiased bicubic resample of torch.nn.functional.interpolate(mode="bicubic", antialias=True, align_corners=False),
 * i.e. PIL's BICUBIC reduction (a = -0.5).  On one axis n_in -> n_out, r = n_in / n_out, s = max(r, 1), output index i reads
 *     c = r * (i + 0.5),  taps j in [max(floor(c - 2s + 0.5), 0), min(floor(c + 2s + 0.5), n_in)),  weight cubic((j - c + 0.5) / s)
 * normalised to sum 1, cubic(x) = ((a + 2)|x| - (a + 3))x^2 + 1 for |x| < 1, a(|x|^3 - 5|x|^2 + 8|x| - 4) for 1 <= |x| < 2, else 0.
 * The device computes it in fp32 with no rounding between the two passes (within 1 of the float64 result).
 *  - dst_width x dst_height == the canvas: byte-identical to w2x_render, and no resample runs.
 *  - An axis with n_out == n_in has the single weight 1: it is left alone.
 *  - The resample never enlarges the model's output: larger sizes are refused.  BGR only.
 * Returns 0 and logs the reason on failure (no engine loaded, null pointers, an output size outside the range above, strides below 3
 * bytes per pixel). */
W2X_API int w2x_render_resized(w2x_engine* e, const uint8_t* src_bgr, int width, int height, size_t src_stride, uint8_t* dst_bgr,
                               int dst_width, int dst_height, size_t dst_stride);
/* w2x_render_resized through the pipeline of w2x_submit: returns a ticket >= 0 for w2x_wait, or -1 with the reason logged. */
W2X_API int w2x_submit_resized(w2x_engine* e, const uint8_t* src_bgr, int width, int height, size_t src_stride, uint8_t* dst_bgr,
                               int dst_width, int dst_height, size_t dst_stride);

/* 16 bits per channel: src BGR u16 HWC (w x h) -> dst BGR u16 (w*scaling x h*scaling), native-endian samples, synchronous like
 * w2x_render, with any loaded engine (fp16 or tf32, cunet/art or swin_unet, with or without TTA).
 *  - Strides are in BYTES: src_stride >= 6 * width, dst_stride >= 6 * width * scaling.  Both strides and both pointers must be even.
 *  - Input: each sample x becomes f32(x) * f32(1/65535) (one rounded multiply), rounded to the engine's element type.  Everything
 *    else is exactly what w2x_render does: replicate padding, D4 augmentation, BGR -> RGB, the tile grid, batching, the TTA mean, the
 *    blend weights and the fp32 accumulation order.
 *  - Output: each sample is saturate_u16(rint(f32(v) * 65535)) of the same fp32 canvas v that w2x_render packs to u8, then RGB -> BGR.
 *  - fp16 engines: fp16(f32(257 x) * f32(1/65535)) == fp16(f32(x) * f32(1/255)) for every u8 value x, so w2x_render_u16 of 257 * F runs
 *    the model on exactly the tiles w2x_render of F does, blends the same canvas, and every output sample satisfies
 *    |out16 - 257 * out8| <= 129.  tf32 engines see the two inputs one fp32 ulp apart and give no such guarantee.
 * Returns 0 and logs the reason on failure (no engine loaded, null pointers, strides below 6 bytes per pixel, odd strides or pointers).
 * Not available with an alpha channel, an output size other than the model's, or through w2x_render_banded / w2x_render_device. */
W2X_API int w2x_render_u16(w2x_engine* e, const uint16_t* src_bgr, int width, int height, size_t src_stride, uint16_t* dst_bgr,
                           size_t dst_stride);
/* w2x_render_u16 through the pipeline of w2x_submit: returns a ticket >= 0 for w2x_wait, or -1 with the reason logged. */
W2X_API int w2x_submit_u16(w2x_engine* e, const uint16_t* src_bgr, int width, int height, size_t src_stride, uint16_t* dst_bgr,
                           size_t dst_stride);

/* Same as w2x_render but src/dst are DEVICE pointers on cfg.deviceId; enqueued on the engine's stream,
 * returns without synchronising (w2x_sync to wait).  Used for the HBM-resident `value` measurement. */
W2X_API int w2x_render_device(w2x_engine* e, const uint8_t* d_src_bgr, int width, int height, size_t src_stride,
                              uint8_t* d_dst_bgr, size_t dst_stride);
/* Pipelined host-buffer render: H2D, compute and D2H of consecutive frames overlap on separate streams
 * (the reference serialises them, main.cpp:263-269).  Buffers should come from w2x_host_alloc (pinned).
 * Returns a ticket >= 0, or -1.  w2x_wait(ticket) blocks until that frame's dst is complete. */
W2X_API int w2x_submit(w2x_engine* e, const uint8_t* src_bgr, int width, int height, size_t src_stride,
                       uint8_t* dst_bgr, size_t dst_stride);
W2X_API int w2x_wait(w2x_engine* e, int ticket);
/* One image sharded over several engines (one per GPU, identically loaded) by contiguous bands of the GLOBAL tile grid's rows;
 * the seam tile row is exchanged peer-to-peer (cudaMemcpyPeerAsync over NVLink), no collective.  Byte-identical to w2x_render
 * on one GPU.  Host buffers as in w2x_render. */
W2X_API int w2x_render_banded(w2x_engine* const* engines, int count, const uint8_t* src_bgr, int width, int height,
                              size_t src_stride, uint8_t* dst_bgr, size_t dst_stride);
W2X_API int w2x_sync(w2x_engine* e);

/* Frame-parallel multi-GPU rendering in one process (the "device list" the reference's single `--device`, main.cpp:70-74, lacks):
 * one engine + weight replica + pinned-copy pipeline + host worker thread per listed device; frame f (the ticket, counted from 0 in
 * submission order) goes to device f mod count; no collective, no peer traffic.  w2x_pool_wait retires frames in whatever order
 * the caller asks (a writer asks in ticket order, which restores frame order).  A device id may be listed more than once.
 * build: cfg->deviceId is ignored, one artefact is built per distinct device NAME in the pool (the name is what the file name
 * hashes, img2img_build.cpp:8-27); load: cfg->deviceId is replaced by each engine's own device.  Buffers as for w2x_submit. */
typedef struct w2x_pool w2x_pool;
W2X_API w2x_pool* w2x_pool_create(const int* device_ids, int count);
W2X_API void w2x_pool_destroy(w2x_pool* p);
W2X_API int w2x_pool_size(w2x_pool* p);
W2X_API w2x_engine* w2x_pool_engine(w2x_pool* p, int index);   /* borrowed: introspection, w2x_render_banded */
W2X_API void w2x_pool_set_message_callback(w2x_pool* p, w2x_message_cb cb, void* user);
W2X_API int w2x_pool_build(w2x_pool* p, const char* onnx_path, const w2x_build_config* cfg);
W2X_API int w2x_pool_load(w2x_pool* p, const char* onnx_path, const w2x_render_config* cfg);
W2X_API int w2x_pool_submit(w2x_pool* p, const uint8_t* src_bgr, int width, int height, size_t src_stride, uint8_t* dst_bgr, size_t dst_stride);
/* w2x_pool_submit with the output of w2x_render_resized; a size the frame's engine refuses fails its w2x_pool_wait, with the reason
 * logged through the pool's message callback. */
W2X_API int w2x_pool_submit_resized(w2x_pool* p, const uint8_t* src_bgr, int width, int height, size_t src_stride, uint8_t* dst_bgr,
                                    int dst_width, int dst_height, size_t dst_stride);
/* w2x_pool_submit with the frames of w2x_render_u16; a frame the engine refuses fails its w2x_pool_wait, with the reason logged through
 * the pool's message callback. */
W2X_API int w2x_pool_submit_u16(w2x_pool* p, const uint16_t* src_bgr, int width, int height, size_t src_stride, uint16_t* dst_bgr,
                                size_t dst_stride);
W2X_API int w2x_pool_wait(w2x_pool* p, int ticket);
W2X_API int w2x_pool_sync(w2x_pool* p);
W2X_API void* w2x_host_alloc(size_t bytes);   /* cudaHostAlloc (pinned) */
W2X_API void w2x_host_free(void* p);
W2X_API void* w2x_device_alloc(w2x_engine* e, size_t bytes);
W2X_API void w2x_device_free(w2x_engine* e, void* p);
W2X_API int w2x_memcpy_h2d(w2x_engine* e, void* dst, const void* src, size_t bytes);
W2X_API int w2x_memcpy_d2h(w2x_engine* e, void* dst, const void* src, size_t bytes);

/* Introspection. */
W2X_API const char* w2x_last_error(w2x_engine* e);
W2X_API int w2x_output_tile_size(w2x_engine* e);          /* outputTensorShape.d[2], img2img_load.cpp:203 */
W2X_API long long w2x_launch_count(w2x_engine* e);        /* kernels launched by this engine so far */
W2X_API double w2x_model_flops_per_tile(w2x_engine* e);   /* algorithmic 2*MAC of the dense layers */
/* Per-stage device time of the LAST completed render, from CUDA events on the engine's stream:
 * out[0]=unpack ms, out[1]=model ms, out[2]=stitch/pack ms, out[3]=total ms, out[4]=tta_reduce ms (0 without --tta); returns count written (<= n). */
W2X_API int w2x_last_stage_ms(w2x_engine* e, float* out, int n);
/* CUDA-event timer on the engine's streams (which: 0 compute, 1 H2D copy, 2 D2H copy): mark idx in [0,16), then
 * w2x_timer_elapsed_ms synchronises both events and returns milliseconds between them (negative on error). */
W2X_API int w2x_timer_mark(w2x_engine* e, int idx, int which);
W2X_API float w2x_timer_elapsed_ms(w2x_engine* e, int idx0, int idx1);
/* Layer-level timing of the model (names + ms) for profiling; returns number of layers, fills up to n. */
W2X_API int w2x_profile_layers(w2x_engine* e, int repeats, char (*names)[48], float* ms, double* flops, int n);

/* Which kernel runs model layer `index` ("patch3x3 ...", "igemm ...", "first-layer mma.sync", "layernorm", "window-attention");
 * returns 0 when index is out of range. */
W2X_API int w2x_layer_kernel(w2x_engine* e, int index, char* buf, int cap);

/* ---- stage entry points (each replaces one reference helper; host buffers; used by the parity tests) ----- */

/* calculateTiles (img2img_render.cpp:7-66).  Writes up to `cap` rects in the reference's column-major order;
 * returns tileCount (or -1).  grid_out (optional, 8 ints): nx, ny, scaledIn w,h, inputOverlap x,y, outOverlap x,y. */
W2X_API int w2x_calculate_tiles(int in_w, int in_h, int out_w, int out_h, int tile_w, int tile_h,
                                int out_tile_w, int out_tile_h, int scaling, double overlap_x, double overlap_y,
                                w2x_rect* in_rects, w2x_rect* out_rects, int cap, int* grid_out);
/* createTileWeights (img2img_load.cpp:29-52): ramp[i] = (float)((double)(i+1)/(overlap+1)), i < overlap. */
W2X_API int w2x_blend_ramp(int overlap, float* ramp);
/* padRoi + applyAugmentation + blobFromImages (render.cpp:68-105,134-177; infer.cpp:5-21) as ONE kernel:
 * u8 BGR frame -> n tiles of fp16 RGB0 NHWC4 [n][tile][tile][4] (returned as raw uint16 bits).
 * aug[i] in 0..7 (render.cpp:123-132), rects may lie outside the frame (replicate). */
W2X_API int w2x_unpack_tiles(int device, const uint8_t* src_bgr, int width, int height, size_t src_stride,
                             const w2x_rect* rects, const int* aug, int n, int tile, uint16_t* out_f16_nhwc4);
/* applyWeights + canvas add + convertTo(8U,255) + RGB2BGR (render.cpp:107-121,325-330,342-343) as ONE kernel:
 * model-native tiles fp16 NHWC4 [count][out_tile][out_tile][4] -> u8 BGR canvas.  Tile i is placed at out_rects[i]. */
W2X_API int w2x_stitch_tiles(int device, const uint16_t* tiles_f16_nhwc4, int count, int out_tile,
                             int nx, int ny, int overlap_x, int overlap_y, int canvas_w, int canvas_h,
                             uint8_t* dst_bgr, size_t dst_stride);
/* reverseAugmentation + TTA accumulate + x(1/8) (render.cpp:179-222,305-318; mean per SURVEY q1):
 * [tiles][8][out_tile][out_tile][4] fp16 -> [tiles][out_tile][out_tile][4] f32. */
W2X_API int w2x_tta_reduce(int device, const uint16_t* outs_f16_nhwc4, int tiles, int out_tile, float* mean_f32_nhwc4);
/* Img2Img::infer (img2img_infer.cpp:41-93): [n,3,T,T] f32 NCHW in [0,1] -> [n,3,outT,outT] f32 NCHW, through the
 * loaded model (n <= batchSize).  Host buffers. */
W2X_API int w2x_infer(w2x_engine* e, const float* in_nchw, int n, float* out_nchw);
/* Host-only helpers (no GPU needed). */
/* getConfigHash (img2img_build.cpp:8-27) on an explicit device name: writes 64 hex chars + NUL. */
W2X_API void w2x_config_hash(const char* device_name, const w2x_build_config* cfg, char out_hex[65]);
/* ONNX -> packed kernel-native weights file, no device needed (the cold part of build). Returns 1/0;
 * err (optional, cap bytes) receives the reason. */
W2X_API int w2x_pack_onnx(const char* onnx_path, const char* out_path, int precision, char* err, int cap);
/* getEnginePath (img2img_load.cpp:79-114) without a GPU: which "<stem>_<16 hex>.w2x" next to model_path a render with *cfg on a
 * device called device_name would load (optimized = exact opt shape first, else the first compatible one in name order).
 * Returns 1 and the path in out_path, or 0 and the reason ("could not satisfy render configuration", ...). */
W2X_API int w2x_select_engine(const char* model_path, const w2x_render_config* cfg, const char* device_name, char* out_path, size_t cap);
/* Describe a packed file: arch id (1 CUNet 1x, 2 UpCUNet 2x), scale, border offset, layer count. */
W2X_API int w2x_pack_info(const char* pack_path, int* arch, int* scale, int* offset, int* layers);

#ifdef __cplusplus
}
#endif
#endif /* W2X_H */
