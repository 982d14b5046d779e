// pool.cu — data-movement kernels over bf16 NHWC slices: MaxPool (YOLOv3-tiny), the Resize/Concat fallback
// copy, and the layout converters behind the parity hooks.  They replace the MaxPool / Resize / Concat nodes
// ONNX Runtime executes at reference server/detector.py:135.  HBM-bound: one 16-byte vector (8 channels)
// per thread, consecutive threads on consecutive channel groups of consecutive pixels.
#include <math.h>
#include <string.h>

#include "kernels.h"

namespace fd {

__device__ __forceinline__ uint4 max_bf16x8(uint4 a, uint4 b) {
    uint4 r;
    const __nv_bfloat162* pa = reinterpret_cast<const __nv_bfloat162*>(&a);
    const __nv_bfloat162* pb = reinterpret_cast<const __nv_bfloat162*>(&b);
    __nv_bfloat162* pr = reinterpret_cast<__nv_bfloat162*>(&r);
#pragma unroll
    for (int i = 0; i < 4; ++i) pr[i] = __hmax2(pa[i], pb[i]);
    return r;
}

__global__ void __launch_bounds__(256)
maxpool_kernel(const __nv_bfloat16* __restrict__ in, int in_pitch, __nv_bfloat16* __restrict__ out, int out_pitch,
               int n, int hi, int wi, int groups, int k, int stride, int pad_lo, int ho, int wo, float pad_value) {
    const long long total = 1LL * n * ho * wo * groups;
    const __nv_bfloat16 pv = __float2bfloat16(pad_value);
    const __nv_bfloat162 pv2 = __halves2bfloat162(pv, pv);
    uint4 padv;
    padv.x = padv.y = padv.z = padv.w = *reinterpret_cast<const uint32_t*>(&pv2);
    const __nv_bfloat16 ninf = __float2bfloat16(-INFINITY);
    const __nv_bfloat162 ninf2 = __halves2bfloat162(ninf, ninf);
    uint4 lowest;
    lowest.x = lowest.y = lowest.z = lowest.w = *reinterpret_cast<const uint32_t*>(&ninf2);
    for (long long i = blockIdx.x * 256LL + threadIdx.x; i < total; i += 256LL * gridDim.x) {
        const int g = static_cast<int>(i % groups);
        long long pix = i / groups;
        const int ox = static_cast<int>(pix % wo);
        pix /= wo;
        const int oy = static_cast<int>(pix % ho);
        const int f = static_cast<int>(pix / ho);
        uint4 acc = lowest;
        for (int r = 0; r < k; ++r)
            for (int s = 0; s < k; ++s) {
                const int iy = oy * stride - pad_lo + r, ix = ox * stride - pad_lo + s;
                uint4 v = padv;
                if (iy >= 0 && iy < hi && ix >= 0 && ix < wi)
                    v = __ldg(reinterpret_cast<const uint4*>(in + ((1LL * f * hi + iy) * wi + ix) * in_pitch + g * 8));
                acc = max_bf16x8(acc, v);
            }
        *reinterpret_cast<uint4*>(out + ((1LL * f * ho + oy) * wo + ox) * out_pitch + g * 8) = acc;
    }
}

int launch_maxpool(const __nv_bfloat16* in, int in_pitch, __nv_bfloat16* out, int out_pitch, int n, int hi, int wi,
                   int c, int k, int stride, int pad_lo, int ho, int wo, float pad_value, cudaStream_t s) {
    if (c % 8) return -1;
    const long long total = 1LL * n * ho * wo * (c / 8);
    const int blocks = static_cast<int>(total / 256 + 1 < 148 * 16 ? total / 256 + 1 : 148 * 16);
    maxpool_kernel<<<blocks, 256, 0, s>>>(in, in_pitch, out, out_pitch, n, hi, wi, c / 8, k, stride, pad_lo, ho, wo,
                                          pad_value);
    return cudaPeekAtLastError() == cudaSuccess ? 0 : -1;  // (peek: the caller reports the reason)
}

// SPP (see kernels.h).  A window clipped to the map is the same set of values as the -inf padded one, so every pool is a
// row maximum over k (slab -> rows buffer) then a column maximum over k (rows buffer -> global): each input element is read
// from global memory once, each output written once with a 16-byte store.  The result is bit-exact (max is exact).
struct SppArgs {
    int k[SPP_MAX_POOLS];
    __nv_bfloat16* out[SPP_MAX_POOLS];
    int npools;
};

__global__ void __launch_bounds__(256)
spp_kernel(const __nv_bfloat16* __restrict__ in, int in_pitch, int out_pitch, int h, int w, int c, const SppArgs a) {
    extern __shared__ uint4 spp_smem[];
    const int hw = h * w;
    uint4* slab = spp_smem;         // [pixel][8 x 16 bytes]
    uint4* rows = spp_smem + hw * 8;
    const int cgroups = (c + 63) / 64;
    const int f = blockIdx.x / cgroups, c0 = (blockIdx.x - f * cgroups) * 64;
    const int nq = (c - c0) / 8 < 8 ? (c - c0) / 8 : 8;  // 16-byte channel groups of this CTA
    const long long pix0 = 1LL * f * hw;
    for (int i = threadIdx.x; i < hw * 8; i += 256) {
        const int pix = i >> 3, q = i & 7;
        if (q < nq) slab[i] = __ldg(reinterpret_cast<const uint4*>(in + (pix0 + pix) * in_pitch + c0 + 8 * q));
    }
    __syncthreads();
#pragma unroll
    for (int j = 0; j < SPP_MAX_POOLS; ++j) {  // (unrolled: a run-time index into the parameters would copy them to the stack)
        if (j >= a.npools) break;
        const int r = a.k[j] >> 1;
        for (int i = threadIdx.x; i < hw * 8; i += 256) {
            const int pix = i >> 3, q = i & 7, y = pix / w, x = pix - y * w;
            if (q >= nq) continue;
            const int x0 = x - r < 0 ? 0 : x - r, x1 = x + r < w ? x + r : w - 1;
            uint4 m = slab[(y * w + x0) * 8 + q];
            for (int xx = x0 + 1; xx <= x1; ++xx) m = max_bf16x8(m, slab[(y * w + xx) * 8 + q]);
            rows[i] = m;
        }
        __syncthreads();
        __nv_bfloat16* out = a.out[j];
        for (int i = threadIdx.x; i < hw * 8; i += 256) {
            const int pix = i >> 3, q = i & 7, y = pix / w, x = pix - y * w;
            if (q >= nq) continue;
            const int y0 = y - r < 0 ? 0 : y - r, y1 = y + r < h ? y + r : h - 1;
            uint4 m = rows[(y0 * w + x) * 8 + q];
            for (int yy = y0 + 1; yy <= y1; ++yy) m = max_bf16x8(m, rows[(yy * w + x) * 8 + q]);
            *reinterpret_cast<uint4*>(out + (pix0 + pix) * out_pitch + c0 + 8 * q) = m;
        }
        __syncthreads();  // the next pool rewrites the rows buffer
    }
}

int spp_init() { return cudaFuncSetAttribute(spp_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024) == cudaSuccess ? 0 : -1; }

int launch_spp(const __nv_bfloat16* in, int in_pitch, int n, int h, int w, int c, int npools, const int* ks,
               __nv_bfloat16* const* outs, int out_pitch, cudaStream_t s) {
    if (c % 8 || in_pitch % 8 || out_pitch % 8 || npools < 1 || npools > SPP_MAX_POOLS || !spp_fits(h, w)) return -1;
    SppArgs a;
    memset(&a, 0, sizeof(a));
    a.npools = npools;
    for (int j = 0; j < npools; ++j) {
        if (ks[j] < 1 || !(ks[j] & 1)) return -1;
        a.k[j] = ks[j];
        a.out[j] = outs[j];
    }
    const size_t smem = 2ULL * h * w * 64 * 2;
    spp_kernel<<<n * ((c + 63) / 64), 256, smem, s>>>(in, in_pitch, out_pitch, h, w, c, a);
    return cudaPeekAtLastError() == cudaSuccess ? 0 : -1;  // (peek: the caller reports the reason)
}

__global__ void __launch_bounds__(256)
copy_slice_kernel(const __nv_bfloat16* __restrict__ in, int in_pitch, __nv_bfloat16* __restrict__ out, int out_pitch,
                  int n, int hi, int wi, int groups, int up) {
    const int ho = up ? 2 * hi : hi, wo = up ? 2 * wi : wi;
    const long long total = 1LL * n * ho * wo * groups;
    for (long long i = blockIdx.x * 256LL + threadIdx.x; i < total; i += 256LL * gridDim.x) {
        const int g = static_cast<int>(i % groups);
        long long pix = i / groups;
        const int ox = static_cast<int>(pix % wo);
        pix /= wo;
        const int oy = static_cast<int>(pix % ho);
        const int f = static_cast<int>(pix / ho);
        const int iy = up ? oy >> 1 : oy, ix = up ? ox >> 1 : ox;
        const uint4 v = __ldg(reinterpret_cast<const uint4*>(in + ((1LL * f * hi + iy) * wi + ix) * in_pitch + g * 8));
        *reinterpret_cast<uint4*>(out + ((1LL * f * ho + oy) * wo + ox) * out_pitch + g * 8) = v;
    }
}

int launch_copy_slice(const __nv_bfloat16* in, int in_pitch, __nv_bfloat16* out, int out_pitch, int n, int hi,
                      int wi, int c, int upsample2x, cudaStream_t s) {
    if (c % 8) return -1;
    const long long total = 1LL * n * hi * wi * (upsample2x ? 4 : 1) * (c / 8);
    const int blocks = static_cast<int>(total / 256 + 1 < 148 * 16 ? total / 256 + 1 : 148 * 16);
    copy_slice_kernel<<<blocks, 256, 0, s>>>(in, in_pitch, out, out_pitch, n, hi, wi, c / 8, upsample2x);
    return cudaPeekAtLastError() == cudaSuccess ? 0 : -1;  // (peek: the caller reports the reason)
}

__global__ void __launch_bounds__(256)
nhwc_to_nchw_f32_kernel(const void* __restrict__ in, int in_pitch, int in_fp32, float* __restrict__ out, int n,
                        int hw, int c) {
    const long long total = 1LL * n * c * hw;
    for (long long i = blockIdx.x * 256LL + threadIdx.x; i < total; i += 256LL * gridDim.x) {
        const int p = static_cast<int>(i % hw);
        const long long t = i / hw;
        const int ch = static_cast<int>(t % c);
        const long long f = t / c;
        const long long src = (f * hw + p) * in_pitch + ch;
        out[i] = in_fp32 ? reinterpret_cast<const float*>(in)[src]
                         : __bfloat162float(reinterpret_cast<const __nv_bfloat16*>(in)[src]);
    }
}

int launch_nhwc_to_nchw_f32(const void* in, int in_pitch, int in_fp32, float* out, int n, int h, int w, int c,
                            cudaStream_t s) {
    const long long total = 1LL * n * c * h * w;
    const int blocks = static_cast<int>(total / 256 + 1 < 148 * 16 ? total / 256 + 1 : 148 * 16);
    nhwc_to_nchw_f32_kernel<<<blocks, 256, 0, s>>>(in, in_pitch, in_fp32, out, n, h * w, c);
    return cudaPeekAtLastError() == cudaSuccess ? 0 : -1;  // (peek: the caller reports the reason)
}

__global__ void __launch_bounds__(256)
nchw_to_rows_f32_kernel(const float* __restrict__ in, float* __restrict__ out, int out_pitch, int n, int hw, int c) {
    const long long total = 1LL * n * hw * c;
    for (long long i = blockIdx.x * 256LL + threadIdx.x; i < total; i += 256LL * gridDim.x) {
        const int ch = static_cast<int>(i % c);
        const long long t = i / c;
        const int p = static_cast<int>(t % hw);
        const long long f = t / hw;
        out[(f * hw + p) * out_pitch + ch] = in[(f * c + ch) * hw + p];
    }
}

int launch_nchw_to_rows_f32(const float* in, float* out, int out_pitch, int n, int h, int w, int c, cudaStream_t s) {
    const long long total = 1LL * n * c * h * w;
    const int blocks = static_cast<int>(total / 256 + 1 < 148 * 16 ? total / 256 + 1 : 148 * 16);
    nchw_to_rows_f32_kernel<<<blocks, 256, 0, s>>>(in, out, out_pitch, n, h * w, c);
    return cudaPeekAtLastError() == cudaSuccess ? 0 : -1;  // (peek: the caller reports the reason)
}

}  // namespace fd
