/*
 * w2x_dev.h -- development / test hooks of the B200-native waifu2x engine.  NOT part of the drop-in boundary (include/w2x.h).
 *
 * w2x_selftest_conv, w2x_run_conv_layer and w2x_run_conv_layer_f32 are exported by the shipped library (lib/libw2x.so): they run the product's own layer
 * kernels on caller-supplied or random data so that tests can compare single layers with an independent fp32 reference.  w2x_layer_tensor,
 * also shipped, reads the per-layer tensors of a loaded engine for the same purpose.
 * The w2x_probe_* micro-benchmarks and every switch that alters or skips kernel work (W2X_DBG, W2X_CONV_IMPL, W2X_NO_PATCH,
 * W2X_NO_FUSE_FIRST, W2X_NO_EPI_GROUPS, W2X_NO_HEAD_KERNEL, W2X_NO_PDL) exist only in the W2X_DEV build, lib/libw2x_dev.so.
 */
#ifndef W2X_DEV_H
#define W2X_DEV_H

#include "w2x.h"

#ifdef __cplusplus
extern "C" {
#endif

/* The colour bleed of w2x_render_bgra on host buffers: src BGRA (w x h, pitch src_stride >= 4 * width), `rounds` rounds ->
 * dst BGRA packed (pitch 4 * width), alpha bytes copied from src.  Returns 1 on success. */
W2X_API int w2x_alpha_bleed(int device, const uint8_t* src_bgra, int width, int height, size_t src_stride, int rounds, uint8_t* dst_bgra);

/* The u16 twins of w2x_unpack_tiles / w2x_stitch_tiles (the kernels of w2x_render_u16), on host buffers:
 *  - w2x_unpack_tiles_u16: u16 BGR frame (pitch src_stride >= 6 * width bytes) -> n fp16 RGB0 NHWC4 tiles, each sample x as
 *    fp16(f32(x) * f32(1/65535)); rects, aug and the replicate padding as w2x_unpack_tiles.
 *  - w2x_stitch_tiles_u16: fp16 NHWC4 tiles -> u16 BGR canvas (pitch dst_stride >= 6 * canvas_w bytes; the bytes between rows are left
 *    alone), each sample saturate(rint(65535 v)) of the fp32 blend that w2x_stitch_tiles packs to u8.
 * Return 1 on success. */
W2X_API int w2x_unpack_tiles_u16(int device, const uint16_t* src_bgr, int width, int height, size_t src_stride, const w2x_rect* rects,
                                 const int* aug, int n, int tile, uint16_t* out_f16_nhwc4);
W2X_API int w2x_stitch_tiles_u16(int device, const uint16_t* tiles_f16_nhwc4, int count, int out_tile, int nx, int ny, int overlap_x,
                                 int overlap_y, int canvas_w, int canvas_h, uint16_t* dst_bgr, size_t dst_stride);

/* The resample of w2x_render_resized alone, on host buffers: src BGR (w x h, pitch src_stride >= 3 * width) -> dst BGR (dst_width x
 * dst_height, pitch dst_stride >= 3 * dst_width; the bytes between rows are left alone), 1 <= dst_width <= width, 1 <= dst_height <= height.
 * Returns 1 on success. */
W2X_API int w2x_resample(int device, const uint8_t* src_bgr, int width, int height, size_t src_stride, uint8_t* dst_bgr, int dst_width, int dst_height,
                         size_t dst_stride);
/* Host only (no GPU): the resample's table of one axis n_in -> n_out (1 <= n_out <= n_in).  Returns taps, the row length of the weight
 * table (0 on error).  When weights != NULL and cap >= n_out * taps, also writes first[n_out] (first input index), count[n_out] (inputs
 * read: first .. first + count - 1, which covers every non-zero weight) and weights[n_out][taps] (fp32, zero past count). */
W2X_API int w2x_resample_table(int n_in, int n_out, int* first, int* count, float* weights, size_t cap);

/* Read-only view of a loaded CUNet/UpCUNet engine, for per-layer tests: after w2x_infer, w2x_render or w2x_submit + w2x_wait, copy one
 * tensor of plan layer `index` (the indexing of w2x_layer_kernel) as the last batch left it into dst (cap bytes); dims[4] receives its
 * shape, unused trailing entries 1.  which:
 *   0 the layer's output activation [batch][h][w][c], engine elements (fp16 bits, or fp32 in a tf32 engine)
 *   1 the model input tensor [batch][tile][tile][4] that w2x_infer fills (index ignored; render reads its tiles elsewhere)
 *   2 SE channel sums, int64 [batch][c], fixed point 2^-10 (SE layers only)
 *   3 SE gate, float [batch][c] (SE layers only)
 *   4 the per-image weights this layer reads, [batch][npad][ktot] engine elements (layers with an SE gate folded into their weights)
 * Slots at and after the image count of the last batch hold stale data.  The call synchronises the engine's streams, launches no kernel
 * and changes no engine state.  dst == NULL: only the size and dims.  Returns the bytes written (or needed); 0 when the layer has no
 * such tensor (the output of a layer computed inside the next one, or of the final layer, which goes to the caller); -1 on error
 * (e.g. a SwinUNet engine), with the message in w2x_last_error. */
W2X_API long long w2x_layer_tensor(w2x_engine* e, int index, int which, void* dst, size_t cap, int* dims);

/* One layer of the dense model path (SURVEY 8a row a17; replaces a slice of the engine enqueued at img2img_infer.cpp:80) on
 * caller-supplied host data, through the kernel the execution planner picks for that shape (head != 0: kinds 3 / 4 through the
 * dedicated head kernels).  Weights are the packed GEMM operand B[npad][ktot] (fp16 bits, K-major) and bias[npad] that `build`
 * writes, layouts in csrc/model_pack.h:
 *   kind 0 conv3x3 + bias + LeakyReLU(0.1)      npad = ceil16(cout), k = (ky*3+kx)*cin + ci                 out [n][h-2][w-2][cout]
 *   kind 1 conv2x2 stride 2 + bias + LeakyReLU  npad = ceil16(cout), k = (dy*2+dx)*cin + ci                 out [n][h/2][w/2][cout]
 *   kind 2 ConvTranspose 2x2 s2 + bias + LeakyReLU + skip[crop 4]   npad = 4*cout, row = (dy*2+dx)*cout + co, k = ci
 *                                               skip [n][2h+8][2w+8][cout]                                  out [n][2h][2w][cout]
 *   kind 3 ConvTranspose 4x4 s2 p3 -> 3 ch      npad = 16, row = (py*2+px)*4 + co, k = (wy*2+wx)*cin + ci, tap (2+py-2wy, 2+px-2wx)
 *                                                                                                           out [n][2h-4][2w-4][4]
 *   kind 4 conv3x3 -> 3 ch + z1[crop 20] + clamp[0,1]   npad = 16 (rows >= 3 zero), k as kind 0; skip [n][h+38][w+38][4]  out [n][h-2][w-2][4]
 * All tensors NHWC fp16 (raw bits).  Returns 1 on success. */
W2X_API int w2x_run_conv_layer(int device, int kind, int head, int n, int h, int w, int cin, int cout, const uint16_t* in_nhwc,
                               const uint16_t* weights, const float* bias, const uint16_t* skip_nhwc, uint16_t* out_nhwc);

/* The same layer kinds 0-4 through the tf32 kernel of `--precision tf32` engines (kernels/conv_tf32_sm100.cu: tcgen05 kind::tf32, fp32
 * accumulate): every tensor is NHWC fp32, the weights are the fp32 packed operand of a tf32 build (same layouts as above; the tensor core
 * uses their TF32 part).  Returns 1 on success. */
W2X_API int w2x_run_conv_layer_f32(int device, int kind, int n, int h, int w, int cin, int cout, const float* in_nhwc, const float* weights,
                                   const float* bias, const float* skip_nhwc, float* out_nhwc);

/* The fused MLP half of a SwinUNet block (kernels/swin_mlp_sm100.cu; replaces a slice of the engine enqueued at img2img_infer.cpp:80):
 * x[tokens][c] (NHWC fp16 bits, updated in place) += fc2(GELU(fc1(LayerNorm(x)))), c = 96 or 192, w1 = [2c][c], w2 = [c][2c] fp16 bits
 * (K-major), gamma / beta [c], b1 [2c], b2 [c].  variant 0 = the kernel the planner picks (weights resident for c = 96, streamed per
 * hidden chunk for c = 192), 1 = streamed weights.  ms_out (optional) receives the average device time of `reps` further launches on
 * the same buffer.  Returns 1 on success. */
W2X_API int w2x_run_swin_mlp(int device, long long tokens, int c, int variant, uint16_t* x, const float* gamma, const float* beta, float eps,
                             const uint16_t* w1, const float* b1, const uint16_t* w2, const float* b2, int reps, float* ms_out);

/* The fused attention half of a SwinUNet block (kernels/swin_attn_sm100.cu; replaces a slice of the engine enqueued at img2img_infer.cpp:80):
 * 6x6 windows, cyclic shift `shift` (0 or 3), relative-position bias relpos[heads][36][36] and torchvision's shift mask; heads = 6, h and w
 * multiples of 6.  c = 96: x[n][h][w][c] (NHWC fp16 bits, updated in place) += proj(window attention(LayerNorm(x))); c = 192: x receives
 * window attention(LayerNorm(x)), the kernel's output before the projection (wproj / bproj may be NULL).  wqkv = [3c][c] (rows q | k | v,
 * head-major), wproj = [c][c] fp16 bits (K-major), bqkv [3c], bproj [c], gamma / beta [c].  ms_out (optional) receives the average device
 * time of `reps` further launches on the same buffers.  Returns 1 on success. */
W2X_API int w2x_run_swin_attn(int device, int n, int h, int w, int c, int heads, int shift, uint16_t* x, const float* gamma, const float* beta, float eps,
                              const uint16_t* wqkv, const float* bqkv, const uint16_t* wproj, const float* bproj, const float* relpos, int reps, float* ms_out);

/* Host-only hooks (no GPU) behind the CPU tests of the fused Swin kernels' operand preparation:
 *  - w2x_swin_attn_prepare: wqkv [3c][c] fp16 bits (rows q | k | v, head-major), bqkv [3c], relpos [heads][36][36] -> the operands
 *    swin_attn_kernel reads: w_out [3c][c] regrouped per 32-channel chunk (q32 | k32 | v32) with the q rows multiplied by d^-1/2 log2(e),
 *    b_out [3c] alike, rel_out [heads][36][pitch] = relpos * log2(e) (rows padded).  Returns pitch (floats per table row), 0 on error.
 *  - w2x_compose_up_to_image: PatchUp (w_up [4*cmid][k] packed rows q0*cmid + c, b_up [4*cmid]) followed by ToImage with pixel shuffle 2
 *    (w_img [16][cmid] packed rows q1*4 + c3, b_img [16]) -> one linear map w_out [64][k], b_out [64] with a pixel shuffle of 4
 *    (row (oy*4 + ox)*4 + c3).  Returns 1 on success. */
W2X_API int w2x_swin_attn_prepare(const uint16_t* wqkv, const float* bqkv, const float* relpos, int c, int heads, uint16_t* w_out, float* b_out,
                                  float* rel_out);
W2X_API int w2x_compose_up_to_image(const uint16_t* w_up, const float* b_up, const uint16_t* w_img, const float* b_img, int cmid, int k, uint16_t* w_out,
                                    float* b_out);

/* One convolution layer of the implicit-GEMM family on random data, tcgen05 kernel vs the scalar CUDA reference
 * kernel, for on-device self-checks: returns max |diff| (negative on error).  kind: 0 conv3x3, 1 conv2x2s2,
 * 2 convT2x2s2(+skip), 3 convT4x4s2p3->4ch, 4 conv3x3->3ch final(+skip,clamp), 5 = kind 4 through the image-head kernel,
 * 6 = kind 3 through the convT-head kernel. */
W2X_API double w2x_selftest_conv(int device, int kind, int n, int h, int w, int cin, int cout, unsigned seed);

/* Development probe: which UMMA smem-descriptor base_offset convention lets a 3x3 tap read a SHIFTED view of one
 * TMA-loaded 128B-swizzled patch (mode 0: base_offset=(start>>7)&7, mode 1: 0; pitch = patch row pitch in pixels).
 * err9[tap] = max |device - host|.  Returns 0 on success. */
W2X_API int w2x_probe_umma(int device, int mode, int pitch, float* err9);

/* Development probe: milliseconds for `iters` x 4 back-to-back tcgen05.mma (M=128, N=n, K=16, fp16) issued on every SM
 * from the same smem operands (A descriptor SBO = sbo_a bytes); cycles per MMA = ms * clock / (4 * iters). */
W2X_API float w2x_probe_mma_rate(int device, int n, int iters, int sbo_a);
/* Same MMA loop while another warp streams `stream_bytes`-sized L2-resident copies into shared memory (0 = none): res[0] = SM
 * cycles per MMA, res[1] = bytes streamed per SM cycle.  Shows how operand reads and async shared-memory writes interfere. */
W2X_API int w2x_probe_mma_rate_stream(int device, int n, int iters, int stream_bytes, float* res);
/* Development probe: milliseconds for `iters` x `chains` (1..8 independent accumulators) mma.sync.m16n8k16 per warp with
 * `warps` warps per SM on every SM, operands in registers: issue rate of the legacy tensor path (first layer, image head, attention). */
W2X_API float w2x_probe_hmma_rate(int device, int warps, int chains, int iters);
/* Development probe: SM cycles per MMA of the 3x3 patch kernel's MMA schedule in isolation (36 N=64 UMMAs per tile from nine tap
 * views, alternating TMEM accumulators, one commit per tile; no loads, no epilogue).  mode bits: 1 = wait for tile t-2's commit
 * before issuing tile t, 2 = one B tile for all taps, 4 = unshifted A views, 8 = a single commit at the end. */
W2X_API float w2x_probe_mma_tiles(int device, int tiles, int mode);
/* Development probe: milliseconds for every SM to copy the same `bytes` (16-byte multiple, <= 48 KiB) L2-resident buffer into
 * shared memory `iters` times with cp.async.bulk, four copies in flight per SM: the L2 -> SM rate streamed weights would get. */
W2X_API float w2x_probe_l2_stream(int device, int bytes, int iters);

#ifdef __cplusplus
}
#endif
#endif /* W2X_DEV_H */
