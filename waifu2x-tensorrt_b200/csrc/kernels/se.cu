// Squeeze/excite (SEBlock of the CUNet family, SURVEY 2.2): per-tile global mean -> FC -> ReLU -> FC -> sigmoid ->
// per-(tile, channel) scale.  Deterministic two-stage reduction (no float atomics): the result must not depend on
// scheduling, because tile outputs are compared bit-for-bit between 1-GPU and N-GPU runs.
#include <cuda_fp16.h>
#include <cuda_runtime.h>

#include "../model_pack.h"
#include "conv_params.h"
#include "launch.h"

namespace w2x {

// Stand-alone squeeze (only used when the producing conv cannot fuse it, e.g. W2X_CONV_IMPL=direct): same exact
// fixed-point integer accumulation as the fused epilogue.  grid (nblk, n), 256 threads; thread t owns channel t % c.
__global__ void __launch_bounds__(256) se_squeeze_kernel(const __half* __restrict__ x, int hw, int c, long long* __restrict__ sums, int nblk) {
    const int img = blockIdx.y, blk = blockIdx.x;
    const int lane_c = threadIdx.x % c, lane_p = threadIdx.x / c, pstride = 256 / c;
    const int per = (hw + nblk - 1) / nblk;
    const int p0 = blk * per, p1 = min(hw, p0 + per);
    const __half* base = x + (size_t)img * hw * c;
    long long s = 0;
    if (lane_p < pstride)
        for (int p = p0 + lane_p; p < p1; p += pstride) s += (long long)__float2int_rn(__half2float(base[(size_t)p * c + lane_c]) * kSeFixedScale);
    if (s != 0) atomicAdd(reinterpret_cast<unsigned long long*>(sums + (size_t)img * c + lane_c), (unsigned long long)s);
}

void launchSeSqueeze(const __half* x, int n, int h, int w, int c, long long* sums, cudaStream_t s) {
    dim3 grid(64, n);
    se_squeeze_kernel<<<grid, 256, 0, s>>>(x, h * w, c, sums, 64);
}

// grid n, block 256.  mean -> relu(W1 mean + b1) -> sigmoid(W2 h + b2)
__global__ void __launch_bounds__(256) se_excite_kernel(const long long* __restrict__ sums, int c, int r, float inv_hw,
                                                        const float* __restrict__ w1, const float* __restrict__ b1,
                                                        const float* __restrict__ w2, const float* __restrict__ b2,
                                                        float* __restrict__ scale) {
    __shared__ float mean[256];
    __shared__ float hid[64];
    __shared__ float sw1[2048], sw2[2048];  // FC weights (r * c <= 2048 for c <= 128, r = c / 8); larger blocks read global
    const int img = blockIdx.x;
    const int fcElems = r * c;
    const bool fcInSmem = fcElems <= 2048;
    pdlLaunchDependents();
    if (fcInSmem)
        for (int i = threadIdx.x; i < fcElems; i += blockDim.x) { sw1[i] = w1[i]; sw2[i] = w2[i]; }
    pdlWait();  // the FC weights above are constants; the channel sums come from the preceding conv
    for (int ch = threadIdx.x; ch < c; ch += blockDim.x)
        mean[ch] = (float)((double)sums[(size_t)img * c + ch] * (1.0 / (double)kSeFixedScale)) * inv_hw;
    __syncthreads();
    const float* W1 = fcInSmem ? sw1 : w1;
    const float* W2 = fcInSmem ? sw2 : w2;
    {
        // hid[j] = relu(b1[j] + <W1[j], mean>): one warp per j, lanes stride the channels
        const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
        for (int j = warp; j < r; j += (blockDim.x >> 5)) {
            float s = 0.f;
            for (int ch = lane; ch < c; ch += 32) s = fmaf(W1[j * c + ch], mean[ch], s);
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
            if (lane == 0) hid[j] = fmaxf(s + b1[j], 0.f);
        }
    }
    __syncthreads();
    for (int ch = threadIdx.x; ch < c; ch += blockDim.x) {
        float s = b2[ch];
        for (int j = 0; j < r; ++j) s = fmaf(W2[ch * r + j], hid[j], s);
        scale[(size_t)img * c + ch] = 1.f / (1.f + expf(-s));
    }
}

void launchSeExcite(const long long* sums, int n, int c, int r, int hw, const float* w1, const float* b1,
                    const float* w2, const float* b2, float* scale, cudaStream_t s) {
    launchPdl(se_excite_kernel, dim3(n), dim3(256), 0, s, sums, c, r, 1.0f / (float)hw, w1, b1, w2, b2, scale);
}

// in-place x *= scale[img][ch], 8 channels (16 B) per thread
__global__ void __launch_bounds__(256) se_scale_kernel(__half* __restrict__ x, long long vec_per_img, int c,
                                                       const float* __restrict__ scale) {
    const int img = blockIdx.y;
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= vec_per_img) return;
    const int c0 = (int)((i * 8) % c);
    const float* sc = scale + (size_t)img * c + c0;
    Half8* px = reinterpret_cast<Half8*>(x) + (size_t)img * vec_per_img + i;
    Half8 v = *px;
    float2 t;
    t = __half22float2(v.a); v.a = __floats2half2_rn(t.x * sc[0], t.y * sc[1]);
    t = __half22float2(v.b); v.b = __floats2half2_rn(t.x * sc[2], t.y * sc[3]);
    t = __half22float2(v.c); v.c = __floats2half2_rn(t.x * sc[4], t.y * sc[5]);
    t = __half22float2(v.d); v.d = __floats2half2_rn(t.x * sc[6], t.y * sc[7]);
    *px = v;
}

__global__ void __launch_bounds__(256) scale_weights_kernel(const __half* __restrict__ w, __half* __restrict__ wOut, const float* __restrict__ scale,
                                                            int total, int ktot, int cin) {
    pdlLaunchDependents();
    pdlWait();
    const int img = blockIdx.y;
    const int i = blockIdx.x * blockDim.x + threadIdx.x;  // pair index
    if (2 * i >= total) return;
    const int k = (2 * i) % ktot;
    const float2 v = __half22float2(reinterpret_cast<const __half2*>(w)[i]);
    const float* sc = scale + (size_t)img * cin + (k % cin);
    reinterpret_cast<__half2*>(wOut + (size_t)img * total)[i] = __floats2half2_rn(v.x * sc[0], v.y * sc[1]);
}

void launchScaleWeights(const __half* w, __half* wOut, const float* scale, int nimg, int npad, int ktot, int cin, cudaStream_t s) {
    const int total = npad * ktot;  // even; k and k+1 share a tap because cin is even
    dim3 grid((total / 2 + 255) / 256, nimg);
    launchPdl(scale_weights_kernel, grid, dim3(256), 0, s, w, wOut, scale, total, ktot, cin);
}

// fp32 twin for tf32 engines: the scaled weights are rounded to nearest TF32 like the packed ones (model_pack.h: roundToTf32)
__global__ void __launch_bounds__(256) scale_weights_f32_kernel(const float* __restrict__ w, float* __restrict__ wOut, const float* __restrict__ scale,
                                                                int total, int ktot, int cin) {
    pdlLaunchDependents();
    pdlWait();
    const int img = blockIdx.y;
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= total) return;
    wOut[(size_t)img * total + i] = roundToTf32(w[i] * scale[(size_t)img * cin + (i % ktot) % cin]);
}

void launchScaleWeightsF32(const float* w, float* wOut, const float* scale, int nimg, int npad, int ktot, int cin, cudaStream_t s) {
    const int total = npad * ktot;
    dim3 grid((total + 255) / 256, nimg);
    launchPdl(scale_weights_f32_kernel, grid, dim3(256), 0, s, w, wOut, scale, total, ktot, cin);
}

void launchSeScale(__half* x, int n, int h, int w, int c, const float* scale, cudaStream_t s) {
    const long long vec = (long long)h * w * c / 8;
    dim3 grid((unsigned)((vec + 255) / 256), n);
    se_scale_kernel<<<grid, 256, 0, s>>>(x, vec, c, scale);
}

}  // namespace w2x
