// Memory-bound tiling kernels: the fused replacements for the reference's cv::cuda library launches in
// /root/reference/src/tensorrt/img2img_render.cpp and img2img_infer.cpp (SURVEY 2.1 table).
//
//   unpack     : padRoi (:68-105) + applyAugmentation (:134-177) + cvtColor BGR2RGB (:227) + split/convertTo(1/255)
//                (infer.cpp:5-21) -> fp16 (f32 for tf32 engines) RGB0 NHWC4 tile batch, one pass, no intermediate mats.
//   stitch     : applyWeights (:107-121) + canvas add (:329-330) + convertTo(8U, 255) (:342) + RGB2BGR (:343).
//                Gather formulation: each output pixel is owned by exactly one thread, which sums the <= 4 covering
//                tiles in the reference's tile order (column-major), so no zero-filled f32 canvas and no RMW passes.
//   tta_reduce : reverseAugmentation (:179-222) + accumulate + x(1/8) (:305-318).
#include <cuda_fp16.h>
#include <cuda_runtime.h>

#include <cstdint>
#include <cstdlib>

#include "conv_params.h"

namespace w2x {

// augmented[r][c] == original[rr][cc] for an n x n tile (D4 ops by OpenCV flip code / NPP CCW rotation; see
// oracle/tiling.py::augment_src_index which tests pin against np.rot90 / slicing).
__device__ __forceinline__ void augSrcIndex(int k, int r, int c, int n, int& rr, int& cc) {
    const int m = n - 1;
    switch (k) {
        default: rr = r; cc = c; break;
        case 1: rr = m - r; cc = c; break;
        case 2: rr = r; cc = m - c; break;
        case 3: rr = c; cc = m - r; break;
        case 4: rr = m - r; cc = m - c; break;
        case 5: rr = m - c; cc = r; break;
        case 6: rr = m - c; cc = m - r; break;
        case 7: rr = c; cc = r; break;
    }
}

// deaugmented[r][c] == model_out[rr][cc]
__device__ __forceinline__ void revSrcIndex(int k, int r, int c, int n, int& rr, int& cc) {
    const int m = n - 1;
    switch (k) {
        default: rr = r; cc = c; break;
        case 1: rr = m - r; cc = c; break;
        case 2: rr = r; cc = m - c; break;
        case 3: rr = m - c; cc = r; break;
        case 4: rr = m - r; cc = m - c; break;
        case 5: rr = c; cc = m - r; break;
        case 6: rr = m - c; cc = m - r; break;
        case 7: rr = c; cc = r; break;
    }
}

// one RGB0 pixel of an NHWC4 tensor: fp16 (fp16 engines) or f32 (tf32 engines)
__device__ __forceinline__ void storePx(__half* out, size_t i, float r, float g, float b) {
    Half4 o;
    o.a = __floats2half2_rn(r, g);
    o.b = __floats2half2_rn(b, 0.f);
    reinterpret_cast<Half4*>(out)[i] = o;
}
__device__ __forceinline__ void storePx(float* out, size_t i, float r, float g, float b) {
    reinterpret_cast<float4*>(out)[i] = make_float4(r, g, b, 0.f);
}
template <typename T> struct Px4;
template <> struct Px4<__half> {
    using type = Half4;
    __device__ __forceinline__ static float3 rgb(const Half4& v) {
        const float2 p0 = __half22float2(v.a), p1 = __half22float2(v.b);
        return make_float3(p0.x, p0.y, p1.x);
    }
};
template <> struct Px4<float> {
    using type = float4;
    __device__ __forceinline__ static float3 rgb(const float4& v) { return make_float3(v.x, v.y, v.z); }
};

// ---- unpack ---------------------------------------------------------------------------------------
// grid: (tile/32 x tile/32 blocks of 32 x 32 output pixels, nslots), 256 threads.  Under every D4 augmentation the source of a
// 32 x 32 output block is a 32 x 32 block of the (replicate-padded) frame, so the block first stages those 32 source rows (96
// bytes each, 128 for BGRA) in shared memory with coalesced loads -- 32-bit words from the 4-byte-aligned start of each row segment
// when the segment lies inside the frame, clamped byte loads on border blocks -- and then every thread converts four pixels, reading
// the staged bytes at the mirrored / transposed position, and writes them with 8-byte stores (256 contiguous bytes per warp).
// PS = source samples per pixel: 3 (BGR) or 4 (BGRA; a slot with valid == kSlotAlpha reads the alpha byte into R, G and B).
// S = source sample type: uint8_t (scaled by 1/255) or uint16_t (BGR only, scaled by 1/65535; 192 source bytes per staged row).
constexpr int kUB = 32;             // block edge
// staged bytes per source row: BGR 96 + up to 3 alignment bytes, rounded up to a word multiple; BGRA rows are word-aligned (128 bytes),
// padded by one word so that the column reads of the transposed augmentations do not all hit one bank; u16 BGR 192 + up to 2
// alignment bytes, rounded up to an odd number of words (49) for the same reason
template <int PS, typename S> constexpr int kURow = sizeof(S) == 2 ? 196 : PS == 3 ? 104 : 132;

template <typename T, int PS, typename S = uint8_t>
__global__ void __launch_bounds__(256) unpack_kernel(const uint8_t* __restrict__ frame, int w, int h, size_t pitch,
                                                     const TileSlot* __restrict__ slots, int tile, int wordOk,
                                                     T* __restrict__ out) {
    static_assert(sizeof(S) == 1 || PS == 3, "u16 frames are BGR");
    constexpr int kRow = kURow<PS, S>;
    __shared__ __align__(16) uint8_t sm[kUB * kRow];
    __shared__ int smOff[kUB];      // byte offset of local source column 0 inside each staged row (fast path: alignment slack)
    const int blocksPerSide = (tile + kUB - 1) / kUB;
    const int slot = blockIdx.y;
    const int br = blockIdx.x / blocksPerSide, bc = blockIdx.x - br * blocksPerSide;
    const int r0 = br * kUB, c0 = bc * kUB;
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
    const TileSlot ts = slots[slot];
    T* outp = out + (size_t)slot * tile * tile * 4;
    if (!ts.valid) {  // padding slot of the last batch (render.cpp:281): a zero tile
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const int r = r0 + ty + 8 * i, c = c0 + tx;
            if (r < tile && c < tile) storePx(outp, (size_t)r * tile + c, 0.f, 0.f, 0.f);
        }
        return;
    }
    // source block = image of the output block's corners (the maps are affine: the image of a square block is a square block)
    int ra, ca, rb, cb;
    const int r1 = min(r0 + kUB, tile) - 1, c1 = min(c0 + kUB, tile) - 1;
    augSrcIndex(ts.aug, r0, c0, tile, ra, ca);
    augSrcIndex(ts.aug, r1, c1, tile, rb, cb);
    const int rrMin = min(ra, rb), ccMin = min(ca, cb);
    const int rows = abs(ra - rb) + 1, cols = abs(ca - cb) + 1;
    const int x0 = ts.x + ccMin;                       // frame column of local source column 0 (may be outside the frame)
    const bool inside = x0 >= 0 && x0 + kUB <= w;      // no horizontal clamping in this block
    // ---- stage: warp `ty` loads rows ty, ty + 8, ...
    for (int lr = ty; lr < rows; lr += 8) {
        const int sy = min(max(ts.y + rrMin + lr, 0), h - 1);
        const uint8_t* rowp = frame + (size_t)sy * pitch;
        if constexpr (sizeof(S) == 2) {
            // u16 BGR: the 192-byte segment starts 2-byte aligned.  Fast path: the words from the 4-byte-aligned start that cover it
            // (48 or 49; the last one ends at most 2 bytes behind the segment, inside the row); else clamped sample loads.
            const size_t segStart = (size_t)sy * pitch + (size_t)x0 * 6;
            if (inside && wordOk && (size_t)(x0 + kUB) * 6 + 2 <= pitch) {
                const size_t a = segStart & ~(size_t)3;
                const int off = (int)(segStart - a), nw = (off + kUB * 6 + 3) >> 2;
                for (int q = tx; q < nw; q += 32)
                    *reinterpret_cast<uint32_t*>(sm + lr * kRow + 4 * q) = *reinterpret_cast<const uint32_t*>(frame + a + 4 * q);
                if (tx == 0) smOff[lr] = off;
            } else {
                const uint16_t* rows16 = reinterpret_cast<const uint16_t*>(rowp);
                uint16_t* d = reinterpret_cast<uint16_t*>(sm + lr * kRow);
                for (int e = tx; e < cols * 3; e += 32) {
                    const int cc = e / 3, ch = e - cc * 3;
                    const int sx = min(max(x0 + cc, 0), w - 1);   // BORDER_REPLICATE
                    d[e] = rows16[(size_t)sx * 3 + ch];
                }
                if (tx == 0) smOff[lr] = 0;
            }
            continue;
        }
        const size_t segStart = (size_t)sy * pitch + (size_t)x0 * PS;  // byte offset of the segment from `frame`
        // fast path: whole 32-pixel segment inside the row and (BGR) at least 4 bytes of the row (or the next row) behind it; a BGRA
        // segment is word-aligned (wordOk includes pitch % 4 == 0) and read exactly
        if (inside && wordOk && (PS == 4 || (size_t)(x0 + kUB) * 3 + 4 <= pitch)) {
            const size_t a = segStart & ~(size_t)3;
            if (tx < (PS == 3 ? kRow / 4 : kUB)) {
                const uint32_t v = *reinterpret_cast<const uint32_t*>(frame + a + 4 * tx);
                *reinterpret_cast<uint32_t*>(sm + lr * kRow + 4 * tx) = v;
            }
            if (tx == 0) smOff[lr] = (int)(segStart - a);
        } else {
            for (int b = tx; b < cols * PS; b += 32) {
                const int cc = b / PS, ch = b - cc * PS;
                const int sx = min(max(x0 + cc, 0), w - 1);   // BORDER_REPLICATE (padRoi, render.cpp:79-100)
                sm[lr * kRow + b] = rowp[(size_t)sx * PS + ch];
            }
            if (tx == 0) smOff[lr] = 0;
        }
    }
    __syncthreads();
    if constexpr (sizeof(S) == 2) {
        const float k = 1.0f / 65535.0f;  // f32(1/65535): a u16 sample 257x gives the fp16 of the u8 sample x
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const int r = r0 + ty + 8 * i, c = c0 + tx;
            if (r >= tile || c >= tile) continue;
            int rr, cc;
            augSrcIndex(ts.aug, r, c, tile, rr, cc);
            const int lr = rr - rrMin;
            const uint16_t* px = reinterpret_cast<const uint16_t*>(sm + lr * kRow + smOff[lr] + (cc - ccMin) * 6);
            const float b = __fmul_rn((float)px[0], k), g = __fmul_rn((float)px[1], k), rch = __fmul_rn((float)px[2], k);
            storePx(outp, (size_t)r * tile + c, rch, g, b);
        }
        return;
    }
    const float k = 1.0f / 255.0f;  // float(1.0/255.0), infer.cpp:19
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int r = r0 + ty + 8 * i, c = c0 + tx;
        if (r >= tile || c >= tile) continue;
        int rr, cc;
        augSrcIndex(ts.aug, r, c, tile, rr, cc);
        const int lr = rr - rrMin;
        const uint8_t* px = sm + lr * kRow + smOff[lr] + (cc - ccMin) * PS;
        if (PS == 4 && ts.valid == kSlotAlpha) {
            const float a = __fmul_rn((float)px[3], k);
            storePx(outp, (size_t)r * tile + c, a, a, a);
            continue;
        }
        const float b = __fmul_rn((float)px[0], k), g = __fmul_rn((float)px[1], k), rch = __fmul_rn((float)px[2], k);
        storePx(outp, (size_t)r * tile + c, rch, g, b);
    }
}

template <typename T>
void launchUnpackT(const uint8_t* frame, int w, int h, size_t pitch, const TileSlot* slots, int nslots, int tile, T* out, cudaStream_t s,
                   PixelFormat format) {
    if (nslots <= 0) return;
    const int side = (tile + kUB - 1) / kUB;
    dim3 grid(side * side, nslots);
    const bool aligned = (reinterpret_cast<uintptr_t>(frame) & 3) == 0;
    switch (format) {
    case PixelFormat::Bgr16: unpack_kernel<T, 3, uint16_t><<<grid, 256, 0, s>>>(frame, w, h, pitch, slots, tile, aligned ? 1 : 0, out); break;
    case PixelFormat::Bgra8:
        unpack_kernel<T, 4><<<grid, 256, 0, s>>>(frame, w, h, pitch, slots, tile, aligned && (pitch & 3) == 0 ? 1 : 0, out);
        break;
    case PixelFormat::Bgr8: unpack_kernel<T, 3><<<grid, 256, 0, s>>>(frame, w, h, pitch, slots, tile, aligned ? 1 : 0, out); break;
    }
}
void launchUnpack(const uint8_t* frame, int w, int h, size_t pitch, const TileSlot* slots, int nslots, int tile, __half* out, cudaStream_t s,
                  PixelFormat format) {
    launchUnpackT(frame, w, h, pitch, slots, nslots, tile, out, s, format);
}
void launchUnpack(const uint8_t* frame, int w, int h, size_t pitch, const TileSlot* slots, int nslots, int tile, float* out, cudaStream_t s,
                  PixelFormat format) {
    launchUnpackT(frame, w, h, pitch, slots, nslots, tile, out, s, format);
}

// ---- stitch + pack ----------------------------------------------------------------------------------
template <bool F32>
__device__ __forceinline__ void loadTilePx(const void* tiles, size_t idx, float& r, float& g, float& b) {
    if (F32) {
        const float4 v = reinterpret_cast<const float4*>(tiles)[idx];
        r = v.x; g = v.y; b = v.z;
    } else {
        const Half4 v = reinterpret_cast<const Half4*>(tiles)[idx];
        const float2 p0 = __half22float2(v.a), p1 = __half22float2(v.b);
        r = p0.x; g = p0.y; b = p1.x;
    }
}

// Block = 256 consecutive output pixels x kSR rows; thread t owns column ox0 + t in every row of the block, so the horizontal cover
// (tiles, ramp weights: two integer divisions) is computed once per thread and reused for kSR pixels, the vertical cover of each row
// is computed once per block (threads 0..kSR-1) and broadcast through shared memory, and the tile reads of a warp are 256
// contiguous bytes.  Along each axis a pixel is covered by at most two tiles (stride = outT - ov > outT / 2).  The packed BGR bytes
// of a row (768 per block) are staged in shared memory and leave as 16-byte vector stores (scalar on unaligned canvases / tails).
// PB = output samples per pixel: 3 (BGR) or 4 (BGRA); O = output sample type: uint8_t, or uint16_t (BGR only: 1536 bytes per block
// row, saturate(rint(65535 v)) of the same fp32 canvas).  A BGRA pixel blends the alpha pass's tile of the same reference tile (slot +
// alpha_off) with the same weights in the same order, and packs the mean of its three channels as alpha; without an alpha pass
// (alpha_off == 0) alpha is 255.
constexpr int kSW = 256, kSR = 16;

__device__ __forceinline__ uint8_t packU8(float v) { return (uint8_t)min(max(__float2int_rn(__fmul_rn(v, 255.f)), 0), 255); }
__device__ __forceinline__ uint16_t packU16(float v) { return (uint16_t)min(max(__float2int_rn(__fmul_rn(v, 65535.f)), 0), 65535); }

struct StitchRow {
    int n;            // covering tile rows (0 past the band end)
    int j[2], ly[2];
    float wt[2], wb[2];
};

template <bool F32, int PB, typename O = uint8_t>
__global__ void __launch_bounds__(kSW) stitch_kernel(StitchParams p, int vecOk) {
    static_assert(sizeof(O) == 1 || PB == 3, "u16 canvases are BGR");
    constexpr int kOB = PB * (int)sizeof(O);   // output bytes per pixel
    __shared__ __align__(16) uint8_t sm[kSR][kSW * kOB];
    __shared__ StitchRow rowInfo[kSR];
    const int ox0 = blockIdx.x * kSW, ox = ox0 + threadIdx.x;
    const int oyBase = p.y_begin + blockIdx.y * kSR;
    const int stx = p.outT - p.ovx, sty = p.outT - p.ovy;
    if (threadIdx.x < kSR) {
        StitchRow ri;
        ri.n = 0;
        const int oy = oyBase + threadIdx.x;
        if (oy < p.y_end) {
            const int j1 = min(oy / sty, p.ny - 1);
            int cand[2], nc = 0;
            if (j1 > 0 && oy - (j1 - 1) * sty < p.outT) cand[nc++] = j1 - 1;
            if (oy - j1 * sty < p.outT) cand[nc++] = j1;
            for (int a = 0; a < nc; ++a) {
                const int j = cand[a];
                const int ty0 = j * sty;
                const int ly = oy - ty0;
                const int th = ty0 + p.outT > p.ch ? p.ch - ty0 : p.outT;  // clipped rect height (render.cpp:60)
                float wt = 1.f, wb = 1.f;
                if (ty0 > 0 && ly < p.ovy) wt = p.rampy[ly];
                if (ty0 + th < p.ch && p.outT - 1 - ly < p.ovy) wb = p.rampy[p.outT - 1 - ly];
                ri.j[a] = j; ri.ly[a] = ly; ri.wt[a] = wt; ri.wb[a] = wb;
            }
            ri.n = nc;
        }
        rowInfo[threadIdx.x] = ri;
    }
    const bool live = ox < p.cw;
    int ti[2] = {0, 0}, lxs[2] = {0, 0}, ni = 0;
    float wls[2] = {1.f, 1.f}, wrs[2] = {1.f, 1.f};
    if (live) {
        const int i1 = min(ox / stx, p.nx - 1);
        int cand[2] = {0, 0}, nc = 0;
        const bool prev = i1 > 0 && ox - (i1 - 1) * stx < p.outT, cur = ox - i1 * stx < p.outT;
        if (prev) { cand[0] = i1 - 1; cand[1] = i1; nc = cur ? 2 : 1; }
        else if (cur) { cand[0] = i1; nc = 1; }
#pragma unroll
        for (int a = 0; a < 2; ++a) {
            if (a >= nc) break;
            const int i = cand[a];
            const int tx0 = i * stx;
            const int lx = ox - tx0;
            const int tw = tx0 + p.outT > p.cw ? p.cw - tx0 : p.outT;  // clipped rect width (render.cpp:59)
            // applyWeights predicates on the clipped rect (render.cpp:110-120); ramps per img2img_load.cpp:29-52
            float wl = 1.f, wr = 1.f;
            if (tx0 > 0 && lx < p.ovx) wl = p.rampx[lx];
            if (tx0 + tw < p.cw && p.outT - 1 - lx < p.ovx) wr = p.rampx[p.outT - 1 - lx];
            ti[a] = i; lxs[a] = lx; wls[a] = wl; wrs[a] = wr;
        }
        ni = nc;
    }
    __syncthreads();
    // a pixel covered by one tile with unit weights (85 % of the canvas at blend 1/16): x 1.0 and 0 + x are exact, so the
    // multiplies and the accumulate can be skipped without changing a bit
    const bool plainX = ni == 1 && wls[0] == 1.f && wrs[0] == 1.f;
#pragma unroll 2
    for (int row = 0; row < kSR; ++row) {
        const StitchRow& ri = rowInfo[row];   // shared-memory broadcast reads
        const int rn = ri.n;
        if (!live || rn == 0) continue;
        float accr = 0.f, accg = 0.f, accb = 0.f;
        float alr = 0.f, alg = 0.f, alb = 0.f;   // BGRA: the alpha pass's canvas
        const bool alpha = PB == 4 && p.alpha_off > 0;
        if (plainX && rn == 1 && ri.wt[0] == 1.f && ri.wb[0] == 1.f) {
            const int slot = p.tile_map ? __ldg(p.tile_map + ti[0] * p.ny + ri.j[0]) : ti[0] * p.ny + ri.j[0];
            loadTilePx<F32>(p.tiles, ((size_t)slot * p.outT + ri.ly[0]) * p.outT + lxs[0], accr, accg, accb);
            if (alpha) loadTilePx<F32>(p.tiles, ((size_t)(slot + p.alpha_off) * p.outT + ri.ly[0]) * p.outT + lxs[0], alr, alg, alb);
        } else {
#pragma unroll
            for (int a = 0; a < 2; ++a) {       // tile order of the reference: x outer, y inner (render.cpp:43-44)
                if (a >= ni) break;
                const float wl = wls[a], wr = wrs[a];
#pragma unroll
                for (int bsel = 0; bsel < 2; ++bsel) {
                    if (bsel >= rn) break;
                    const float wt = ri.wt[bsel], wb = ri.wb[bsel];
                    float r, g, b;
                    const int slot = p.tile_map ? __ldg(p.tile_map + ti[a] * p.ny + ri.j[bsel]) : ti[a] * p.ny + ri.j[bsel];
                    loadTilePx<F32>(p.tiles, ((size_t)slot * p.outT + ri.ly[bsel]) * p.outT + lxs[a], r, g, b);
                    // sequential in-place multiplies in the reference order: left, top, right, bottom (x1.0 is exact)
                    r = __fmul_rn(__fmul_rn(__fmul_rn(__fmul_rn(r, wl), wt), wr), wb);
                    g = __fmul_rn(__fmul_rn(__fmul_rn(__fmul_rn(g, wl), wt), wr), wb);
                    b = __fmul_rn(__fmul_rn(__fmul_rn(__fmul_rn(b, wl), wt), wr), wb);
                    accr = __fadd_rn(accr, r);
                    accg = __fadd_rn(accg, g);
                    accb = __fadd_rn(accb, b);
                    if (alpha) {
                        loadTilePx<F32>(p.tiles, ((size_t)(slot + p.alpha_off) * p.outT + ri.ly[bsel]) * p.outT + lxs[a], r, g, b);
                        r = __fmul_rn(__fmul_rn(__fmul_rn(__fmul_rn(r, wl), wt), wr), wb);
                        g = __fmul_rn(__fmul_rn(__fmul_rn(__fmul_rn(g, wl), wt), wr), wb);
                        b = __fmul_rn(__fmul_rn(__fmul_rn(__fmul_rn(b, wl), wt), wr), wb);
                        alr = __fadd_rn(alr, r);
                        alg = __fadd_rn(alg, g);
                        alb = __fadd_rn(alb, b);
                    }
                }
            }
        }
        if constexpr (sizeof(O) == 2) {
            uint16_t* d = reinterpret_cast<uint16_t*>(sm[row]) + threadIdx.x * 3;
            d[0] = packU16(accb);
            d[1] = packU16(accg);
            d[2] = packU16(accr);
            continue;
        }
        // convertTo(CV_8UC3, 255): saturate_cast<uchar>(rint(v * 255)) (render.cpp:342), then RGB -> BGR (:343)
        uint8_t* d = sm[row] + threadIdx.x * PB;
        d[0] = packU8(accb);
        d[1] = packU8(accg);
        d[2] = packU8(accr);
        if (PB == 4) d[3] = alpha ? packU8(__fdiv_rn(__fadd_rn(__fadd_rn(alr, alg), alb), 3.f)) : (uint8_t)255;
    }
    __syncthreads();
    const int nbytes = min(kSW, p.cw - ox0) * kOB;
    if (nbytes <= 0) return;
    const int rowsHere = min(kSR, p.y_end - oyBase);
    if (vecOk) {
        const int nvec = nbytes >> 4;                       // 48 (BGRA: 64, u16 BGR: 96) vectors per full row
        for (int v = threadIdx.x; v < nvec * rowsHere; v += kSW) {
            const int row = v / nvec, c = v - row * nvec;
            reinterpret_cast<uint4*>(p.dst + (size_t)(oyBase + row) * p.pitch + (size_t)ox0 * kOB)[c] = reinterpret_cast<const uint4*>(sm[row])[c];
        }
        const int tail = nbytes - (nvec << 4);
        for (int b = threadIdx.x; b < tail * rowsHere; b += kSW) {
            const int row = b / tail, c = (nvec << 4) + b - row * tail;
            p.dst[(size_t)(oyBase + row) * p.pitch + (size_t)ox0 * kOB + c] = sm[row][c];
        }
    } else {
        for (int row = 0; row < rowsHere; ++row)
            for (int b = threadIdx.x; b < nbytes; b += kSW) p.dst[(size_t)(oyBase + row) * p.pitch + (size_t)ox0 * kOB + b] = sm[row][b];
    }
}

void launchStitch(const StitchParams& pin, cudaStream_t s) {
    StitchParams p = pin;
    if (p.y_end <= 0) { p.y_begin = 0; p.y_end = p.ch; }  // whole canvas
    if (p.y_end <= p.y_begin) return;
    dim3 grid((p.cw + kSW - 1) / kSW, (p.y_end - p.y_begin + kSR - 1) / kSR);
    // 16-byte stores need 16-byte aligned row segments: block columns start at multiples of 768 (BGRA: 1024, u16 BGR: 1536) bytes
    const int vecOk = ((reinterpret_cast<uintptr_t>(p.dst) & 15) == 0 && (p.pitch & 15) == 0) ? 1 : 0;
    switch (p.format) {
    case PixelFormat::Bgr16:
        if (p.f32) stitch_kernel<true, 3, uint16_t><<<grid, kSW, 0, s>>>(p, vecOk);
        else stitch_kernel<false, 3, uint16_t><<<grid, kSW, 0, s>>>(p, vecOk);
        break;
    case PixelFormat::Bgra8:
        if (p.f32) stitch_kernel<true, 4><<<grid, kSW, 0, s>>>(p, vecOk);
        else stitch_kernel<false, 4><<<grid, kSW, 0, s>>>(p, vecOk);
        break;
    case PixelFormat::Bgr8:
        if (p.f32) stitch_kernel<true, 3><<<grid, kSW, 0, s>>>(p, vecOk);
        else stitch_kernel<false, 3><<<grid, kSW, 0, s>>>(p, vecOk);
        break;
    }
}

// ---- TTA reduce -------------------------------------------------------------------------------------
// acc = 0 + out_0; acc += rev_k(out_k), k = 1..7 (index order); acc *= 1/8   (render.cpp:305-318, mean per SURVEY q1).
// Block = 32 x 32 output pixels of one tile.  For each augmentation the 32 x 32 source block of that model output (again a square
// block, see unpack) is staged in shared memory with coalesced 8-byte loads (256 contiguous bytes per row), so the transposed
// augmentations gather from shared memory instead of striding through HBM; every thread then adds its four pixels in index order.
template <typename T>
__global__ void __launch_bounds__(256) tta_reduce_kernel(const T* __restrict__ outs, int outT, float* __restrict__ mean) {
    using P = typename Px4<T>::type;
    __shared__ P sm[kUB][kUB + 1];
    const int tile = blockIdx.y;
    const int side = (outT + kUB - 1) / kUB;
    const int br = blockIdx.x / side, bc = blockIdx.x - br * side;
    const int r0 = br * kUB, c0 = bc * kUB;
    const int r1 = min(r0 + kUB, outT) - 1, c1 = min(c0 + kUB, outT) - 1;
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
    const size_t plane = (size_t)outT * outT;
    float ar[4] = {0.f, 0.f, 0.f, 0.f}, ag[4] = {0.f, 0.f, 0.f, 0.f}, ab[4] = {0.f, 0.f, 0.f, 0.f};
    for (int k = 0; k < 8; ++k) {
        int ra, ca, rb, cb;
        revSrcIndex(k, r0, c0, outT, ra, ca);
        revSrcIndex(k, r1, c1, outT, rb, cb);
        const int rrMin = min(ra, rb), ccMin = min(ca, cb);
        const int rows = abs(ra - rb) + 1, cols = abs(ca - cb) + 1;
        const P* src = reinterpret_cast<const P*>(outs) + ((size_t)tile * 8 + k) * plane;
        __syncthreads();  // the previous augmentation's reads of sm are done
        for (int lr = ty; lr < rows; lr += 8)
            if (tx < cols) sm[lr][tx] = src[(size_t)(rrMin + lr) * outT + ccMin + tx];
        __syncthreads();
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const int r = r0 + ty + 8 * i, c = c0 + tx;
            if (r >= outT || c >= outT) continue;
            int rr, cc;
            revSrcIndex(k, r, c, outT, rr, cc);
            const float3 v = Px4<T>::rgb(sm[rr - rrMin][cc - ccMin]);
            ar[i] = __fadd_rn(ar[i], v.x);
            ag[i] = __fadd_rn(ag[i], v.y);
            ab[i] = __fadd_rn(ab[i], v.z);
        }
    }
    const float k8 = 0.125f;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int r = r0 + ty + 8 * i, c = c0 + tx;
        if (r >= outT || c >= outT) continue;
        reinterpret_cast<float4*>(mean)[(size_t)tile * plane + (size_t)r * outT + c] =
            make_float4(__fmul_rn(ar[i], k8), __fmul_rn(ag[i], k8), __fmul_rn(ab[i], k8), 0.f);
    }
}

template <typename T>
void launchTtaReduceT(const T* outs, int tiles, int outT, float* mean, cudaStream_t s) {
    if (tiles <= 0) return;
    const int side = (outT + kUB - 1) / kUB;
    dim3 grid(side * side, tiles);
    tta_reduce_kernel<T><<<grid, 256, 0, s>>>(outs, outT, mean);
}
void launchTtaReduce(const __half* outs, int tiles, int outT, float* mean, cudaStream_t s) { launchTtaReduceT(outs, tiles, outT, mean, s); }
void launchTtaReduce(const float* outs, int tiles, int outT, float* mean, cudaStream_t s) { launchTtaReduceT(outs, tiles, outT, mean, s); }

// ---- layout helpers for the Img2Img::infer-shaped entry point ---------------------------------------------
template <typename T>
__global__ void nchw_to_nhwc4_kernel(const float* __restrict__ in, int t, T* __restrict__ out) {
    const int n = blockIdx.y;
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= t * t) return;
    const size_t plane = (size_t)t * t;
    const float* b = in + (size_t)n * 3 * plane;
    storePx(out, (size_t)n * plane + idx, b[idx], b[plane + idx], b[2 * plane + idx]);
}

template <typename T>
__global__ void nhwc4_to_nchw_kernel(const T* __restrict__ in, int t, float* __restrict__ out) {
    const int n = blockIdx.y;
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= t * t) return;
    const size_t plane = (size_t)t * t;
    const float3 v = Px4<T>::rgb(reinterpret_cast<const typename Px4<T>::type*>(in)[(size_t)n * plane + idx]);
    float* b = out + (size_t)n * 3 * plane;
    b[idx] = v.x;
    b[plane + idx] = v.y;
    b[2 * plane + idx] = v.z;
}

void launchNchwToNhwc4(const float* in, int n, int t, __half* out, cudaStream_t s) {
    nchw_to_nhwc4_kernel<<<dim3((t * t + 255) / 256, n), 256, 0, s>>>(in, t, out);
}
void launchNchwToNhwc4(const float* in, int n, int t, float* out, cudaStream_t s) {
    nchw_to_nhwc4_kernel<<<dim3((t * t + 255) / 256, n), 256, 0, s>>>(in, t, out);
}
void launchNhwc4ToNchw(const __half* in, int n, int t, float* out, cudaStream_t s) {
    nhwc4_to_nchw_kernel<<<dim3((t * t + 255) / 256, n), 256, 0, s>>>(in, t, out);
}
void launchNhwc4ToNchw(const float* in, int n, int t, float* out, cudaStream_t s) {
    nhwc4_to_nchw_kernel<<<dim3((t * t + 255) / 256, n), 256, 0, s>>>(in, t, out);
}

}  // namespace w2x
