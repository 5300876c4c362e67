// Memory-bound kernels of the BGRA path (Bgra8 frames): the alpha scan that decides whether a frame needs the colour bleed and
// the alpha model pass, and one round of the colour bleed.  Frames are packed w x h BGRA on the device (one 32-bit word per pixel,
// alpha in the top byte).
#include <cuda_runtime.h>

#include <algorithm>
#include <cstdint>

#include "conv_params.h"

namespace w2x {

// Grid-stride over 16-byte vectors (four pixels), the last n % 4 pixels by the first threads.  One store per warp that saw a hit:
// the flags only ever go from 0 to 1, so racing stores are harmless.
__global__ void __launch_bounds__(256) alpha_scan_kernel(const uint32_t* __restrict__ px, size_t n, int* __restrict__ flags) {
    bool below = false, zero = false;
    const size_t n4 = n / 4, stride = (size_t)gridDim.x * blockDim.x;
    const size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const uint4* v = reinterpret_cast<const uint4*>(px);
    for (size_t i = t; i < n4; i += stride) {
        const uint4 q = __ldg(v + i);
        below |= ((q.x & q.y & q.z & q.w) >> 24) != 255u;
        zero |= (q.x >> 24) == 0u || (q.y >> 24) == 0u || (q.z >> 24) == 0u || (q.w >> 24) == 0u;
    }
    if (t < n - n4 * 4) {
        const uint32_t a = __ldg(px + n4 * 4 + t) >> 24;
        below |= a != 255u;
        zero |= a == 0u;
    }
    below = __any_sync(0xffffffffu, below);
    zero = __any_sync(0xffffffffu, zero);
    if ((threadIdx.x & 31) == 0) {
        if (below) flags[0] = 1;
        if (zero) flags[1] = 1;
    }
}

void launchAlphaScan(const uint8_t* bgra, size_t pixels, int* flags, cudaStream_t s) {
    if (pixels == 0) return;
    const size_t vecs = pixels / 4 + 1;
    const int blocks = (int)std::min<size_t>((vecs + 255) / 256, 148 * 8);
    alpha_scan_kernel<<<blocks, 256, 0, s>>>(reinterpret_cast<const uint32_t*>(bgra), pixels, flags);
}

// One thread per pixel, 32 x 8 blocks; the 3 x 3 neighbourhood reads hit L1.  Integer arithmetic only: the result is exact.
__global__ void __launch_bounds__(256) alpha_bleed_kernel(const uint32_t* __restrict__ in, uint32_t* __restrict__ out, int w, int h, int grow,
                                                          const uint32_t* __restrict__ alphaOf) {
    const int x = blockIdx.x * 32 + threadIdx.x, y = blockIdx.y * 8 + threadIdx.y;
    if (x >= w || y >= h) return;
    const size_t i = (size_t)y * w + x;
    const uint32_t c = __ldg(in + i);
    uint32_t res = 0;
    if (c >> 24) {
        res = c | 0xff000000u;
    } else if (grow) {
        int n = 0, sb = 0, sg = 0, sr = 0;
#pragma unroll
        for (int dy = -1; dy <= 1; ++dy) {
            const int yy = y + dy;
            if (yy < 0 || yy >= h) continue;
#pragma unroll
            for (int dx = -1; dx <= 1; ++dx) {
                const int xx = x + dx;
                if (xx < 0 || xx >= w) continue;
                const uint32_t v = __ldg(in + (size_t)yy * w + xx);   // the centre is unknown: it never counts
                if (v >> 24) {
                    ++n;
                    sb += v & 255u;
                    sg += (v >> 8) & 255u;
                    sr += (v >> 16) & 255u;
                }
            }
        }
        if (n) {
            const int d = 2 * n;   // mean rounded half up
            res = 0xff000000u | (uint32_t)((2 * sr + n) / d) << 16 | (uint32_t)((2 * sg + n) / d) << 8 | (uint32_t)((2 * sb + n) / d);
        }
    }
    if (alphaOf) res = (res & 0x00ffffffu) | (__ldg(alphaOf + i) & 0xff000000u);
    out[i] = res;
}

void launchAlphaBleedRound(const uint8_t* in, uint8_t* out, int w, int h, int grow, const uint8_t* alphaOf, cudaStream_t s) {
    if (w <= 0 || h <= 0) return;
    alpha_bleed_kernel<<<dim3((w + 31) / 32, (h + 7) / 8), dim3(32, 8), 0, s>>>(reinterpret_cast<const uint32_t*>(in), reinterpret_cast<uint32_t*>(out),
                                                                               w, h, grow, reinterpret_cast<const uint32_t*>(alphaOf));
}

}  // namespace w2x
