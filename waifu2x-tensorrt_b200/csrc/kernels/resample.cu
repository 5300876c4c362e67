// Antialiased bicubic reduction of a u8 BGR canvas (frames with an output size): a horizontal pass from the canvas into an fp32 image of
// dst_w columns, then a vertical pass from that image into the u8 destination.  Both passes read host-built per-axis tables
// (hostutil.h, resampleAxis); nothing is rounded between them.  The horizontal pass works on any band of canvas rows and the vertical
// pass on any band of output rows, so the engine can resample a frame band by band while the model still computes the rest.
#include <cuda_runtime.h>

#include <cstdint>

#include "conv_params.h"

namespace w2x {

// One thread per (output column, canvas row), three channels each.  The taps of neighbouring threads overlap: the reads hit L1.
__global__ void __launch_bounds__(256) resample_h_kernel(const uint8_t* __restrict__ canvas, size_t pitch, int y0, int y1, ResampleTable t, int dstW,
                                                         float* __restrict__ tmp) {
    const int x = blockIdx.x * blockDim.x + threadIdx.x, y = y0 + blockIdx.y * blockDim.y + threadIdx.y;
    if (x >= dstW || y >= y1) return;
    const int first = __ldg(t.first + x), n = __ldg(t.count + x);
    const uint8_t* p = canvas + (size_t)y * pitch + (size_t)first * 3;
    const float* w = t.w + (size_t)x * t.taps;
    float b = 0.f, g = 0.f, r = 0.f;
    for (int k = 0; k < n; ++k) {
        const float wk = __ldg(w + k);
        b = fmaf(wk, (float)__ldg(p + 3 * k), b);
        g = fmaf(wk, (float)__ldg(p + 3 * k + 1), g);
        r = fmaf(wk, (float)__ldg(p + 3 * k + 2), r);
    }
    float* o = tmp + ((size_t)y * dstW + x) * 3;
    o[0] = b;
    o[1] = g;
    o[2] = r;
}

// One thread per (output byte of a row, output row): consecutive threads read consecutive floats of each tap row.
__global__ void __launch_bounds__(256) resample_v_kernel(const float* __restrict__ tmp, int rowElems, ResampleTable t, int i0, int i1,
                                                         uint8_t* __restrict__ dst, size_t pitch) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x, i = i0 + blockIdx.y * blockDim.y + threadIdx.y;
    if (j >= rowElems || i >= i1) return;
    const int first = __ldg(t.first + i), n = __ldg(t.count + i);
    const float* p = tmp + (size_t)first * rowElems + j;
    const float* w = t.w + (size_t)i * t.taps;
    float acc = 0.f;
    for (int k = 0; k < n; ++k) acc = fmaf(__ldg(w + k), __ldg(p + (size_t)k * rowElems), acc);
    dst[(size_t)i * pitch + j] = (uint8_t)min(max(__float2int_rn(acc), 0), 255);
}

void launchResampleH(const uint8_t* canvas, size_t pitch, int y0, int y1, const ResampleTable& tx, int dstW, float* tmp, cudaStream_t s) {
    if (y1 <= y0 || dstW <= 0) return;
    const dim3 block(64, 4);
    resample_h_kernel<<<dim3((dstW + 63) / 64, (y1 - y0 + 3) / 4), block, 0, s>>>(canvas, pitch, y0, y1, tx, dstW, tmp);
}

void launchResampleV(const float* tmp, int dstW, const ResampleTable& ty, int i0, int i1, uint8_t* dst, size_t pitch, cudaStream_t s) {
    if (i1 <= i0 || dstW <= 0) return;
    const int rowElems = dstW * 3;
    const dim3 block(128, 2);
    resample_v_kernel<<<dim3((rowElems + 127) / 128, (i1 - i0 + 1) / 2), block, 0, s>>>(tmp, rowElems, ty, i0, i1, dst, pitch);
}

}  // namespace w2x
