// pre.cu — frame ingest kernels (HBM-bound; coalesced / vectorised byte traffic, no tensor cores).
//
//   normalise_f32_nchw : reference server/detector.py:133-134  (u8 HWC -> x/255 in f64 -> f32 -> NCHW)
//   letterbox_u8       : extension (the reference rejects non-net-sized frames, detector.py:131-132)
//   conv0_u8           : the same normalisation fused into the first convolution (Cin = 3), so the f32
//                        NCHW tensor the reference materialises never exists on the serving path.
#include <stdlib.h>

#include "act.cuh"
#include "conv_tc.h"
#include "kernels.h"
#include "ptx.cuh"

namespace fd {

// float32(k / 255.0): the reference divides in float64 and rounds once to float32.
__device__ __forceinline__ float norm_u8(int k) { return static_cast<float>(static_cast<double>(k) / 255.0); }

__global__ void __launch_bounds__(256)
normalise_f32_nchw_kernel(const uint8_t* __restrict__ frames, float* __restrict__ out, int n, int hw) {
    __shared__ float lut[256];
    lut[threadIdx.x] = norm_u8(threadIdx.x);
    __syncthreads();
    const long long quads_per_frame = hw / 4;  // host guarantees hw % 4 == 0 on this path
    const long long total = quads_per_frame * n;
    for (long long q = blockIdx.x * 256LL + threadIdx.x; q < total; q += 256LL * gridDim.x) {
        const long long f = q / quads_per_frame;
        const long long p = (q - f * quads_per_frame) * 4;  // first pixel of the quad inside the frame
        const uint32_t* src = reinterpret_cast<const uint32_t*>(frames + (f * hw + p) * 3);
        const uint32_t a = __ldg(src), b = __ldg(src + 1), c = __ldg(src + 2);  // 12 bytes = 4 RGB pixels
        // bytes: a = r0 g0 b0 r1 | b = g1 b1 r2 g2 | c = b2 r3 g3 b3
        const float4 r = make_float4(lut[a & 255], lut[a >> 24], lut[(b >> 16) & 255], lut[(c >> 8) & 255]);
        const float4 g = make_float4(lut[(a >> 8) & 255], lut[b & 255], lut[b >> 24], lut[(c >> 16) & 255]);
        const float4 bl = make_float4(lut[(a >> 16) & 255], lut[(b >> 8) & 255], lut[c & 255], lut[c >> 24]);
        float* o = out + f * 3 * hw + p;
        *reinterpret_cast<float4*>(o) = r;
        *reinterpret_cast<float4*>(o + hw) = g;
        *reinterpret_cast<float4*>(o + 2LL * hw) = bl;
    }
}

__global__ void __launch_bounds__(256)
normalise_f32_nchw_scalar_kernel(const uint8_t* __restrict__ frames, float* __restrict__ out, int n, int hw) {
    const long long total = 1LL * n * hw;
    for (long long i = blockIdx.x * 256LL + threadIdx.x; i < total; i += 256LL * gridDim.x) {
        const long long f = i / hw, p = i - f * hw;
        const uint8_t* s = frames + i * 3;
        float* o = out + f * 3 * hw + p;
        o[0] = norm_u8(s[0]);
        o[hw] = norm_u8(s[1]);
        o[2LL * hw] = norm_u8(s[2]);
    }
}

int launch_normalise_f32_nchw(const uint8_t* frames, float* out, int n, int h, int w, cudaStream_t s) {
    const int hw = h * w;
    const bool vec = (hw % 4 == 0) && ((reinterpret_cast<uintptr_t>(frames) & 3) == 0) &&
                     ((reinterpret_cast<uintptr_t>(out) & 15) == 0);
    const long long work = vec ? 1LL * n * hw / 4 : 1LL * n * hw;
    const int blocks = static_cast<int>(work / 256 + 1 < 148 * 16 ? work / 256 + 1 : 148 * 16);
    if (vec) normalise_f32_nchw_kernel<<<blocks, 256, 0, s>>>(frames, out, n, hw);
    else normalise_f32_nchw_scalar_kernel<<<blocks, 256, 0, s>>>(frames, out, n, hw);
    return cudaPeekAtLastError() == cudaSuccess ? 0 : -1;  // (peek: the caller reports the reason)
}

// ------------------------------------------------------------------------------------ letterbox
__device__ __forceinline__ void lb_axis(int d, int n_dst, int n_src, int* i0, int* i1, int* fr) {
    long long pos = ((2LL * d + 1) * n_src * 65536LL) / (2LL * n_dst) - 32768LL;
    const long long hi = (n_src - 1) * 65536LL;
    pos = pos < 0 ? 0 : (pos > hi ? hi : pos);
    *i0 = static_cast<int>(pos >> 16);
    *fr = static_cast<int>(pos & 0xFFFF);
    *i1 = *i0 + 1 < n_src ? *i0 + 1 : n_src - 1;
}

__global__ void __launch_bounds__(256)
letterbox_u8_kernel(const uint8_t* __restrict__ src, uint8_t* __restrict__ dst, int n, int sh, int sw, int h, int w,
                    int new_w, int new_h, int off_x, int off_y, int fill) {
    const long long total = 1LL * n * h * w;
    for (long long i = blockIdx.x * 256LL + threadIdx.x; i < total; i += 256LL * gridDim.x) {
        const int f = static_cast<int>(i / (1LL * h * w));
        const int rem = static_cast<int>(i - 1LL * f * h * w);
        const int y = rem / w, x = rem - y * w;
        uint8_t* o = dst + i * 3;
        const int dx = x - off_x, dy = y - off_y;
        if (dx < 0 || dx >= new_w || dy < 0 || dy >= new_h) {
            o[0] = o[1] = o[2] = static_cast<uint8_t>(fill);
            continue;
        }
        int x0, x1, fx, y0, y1, fy;
        lb_axis(dx, new_w, sw, &x0, &x1, &fx);
        lb_axis(dy, new_h, sh, &y0, &y1, &fy);
        const uint8_t* base = src + 1LL * f * sh * sw * 3;
        const uint8_t* p00 = base + (1LL * y0 * sw + x0) * 3;
        const uint8_t* p01 = base + (1LL * y0 * sw + x1) * 3;
        const uint8_t* p10 = base + (1LL * y1 * sw + x0) * 3;
        const uint8_t* p11 = base + (1LL * y1 * sw + x1) * 3;
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            const long long top = 1LL * p00[c] * (65536 - fx) + 1LL * p01[c] * fx;
            const long long bot = 1LL * p10[c] * (65536 - fx) + 1LL * p11[c] * fx;
            o[c] = static_cast<uint8_t>((top * (65536 - fy) + bot * fy + (1LL << 31)) >> 32);
        }
    }
}

int launch_letterbox_u8(const uint8_t* src, uint8_t* dst, int n, int sh, int sw, int h, int w, int fill,
                        cudaStream_t s) {
    int new_w, new_h;
    if (1LL * sw * h >= 1LL * sh * w) {
        new_w = w;
        new_h = static_cast<int>((1LL * sh * w + sw / 2) / sw);
        if (new_h < 1) new_h = 1;
    } else {
        new_h = h;
        new_w = static_cast<int>((1LL * sw * h + sh / 2) / sh);
        if (new_w < 1) new_w = 1;
    }
    const int off_x = (w - new_w) / 2, off_y = (h - new_h) / 2;
    const long long total = 1LL * n * h * w;
    const int blocks = static_cast<int>(total / 256 + 1 < 148 * 16 ? total / 256 + 1 : 148 * 16);
    letterbox_u8_kernel<<<blocks, 256, 0, s>>>(src, dst, n, sh, sw, h, w, new_w, new_h, off_x, off_y, fill);
    return cudaPeekAtLastError() == cudaSuccess ? 0 : -1;  // (peek: the caller reports the reason)
}

// ------------------------------------------------------------------------------------ first conv
// Tile: 32 x 16 output pixels per CTA of 128 threads; each thread owns a 4-pixel horizontal strip and
// walks the output channels 8 at a time, so every 2 broadcast LDS.128 of weights feed 32 FMAs.
static constexpr int C0_TW = 32, C0_TH = 16, C0_THREADS = 128;

__device__ __forceinline__ uint32_t c0_pack(float a, float b) {
    __nv_bfloat162 v = __floats2bfloat162_rn(a, b);
    return *reinterpret_cast<uint32_t*>(&v);
}
__device__ __forceinline__ uint32_t c0_max(uint32_t a, uint32_t b) {  // bf16x2 maximum
    const __nv_bfloat162 r = __hmax2(*reinterpret_cast<const __nv_bfloat162*>(&a), *reinterpret_cast<const __nv_bfloat162*>(&b));
    return *reinterpret_cast<const uint32_t*>(&r);
}

// MISH: Mish (act.cuh) instead of LeakyReLU(alpha) when act is set
template <bool MISH = false>
__global__ void __launch_bounds__(C0_THREADS)
conv0_u8_kernel(const uint8_t* __restrict__ frames, const float* __restrict__ wgt, const float* __restrict__ bias,
                __nv_bfloat16* __restrict__ out, int h, int wd, int cout, int out_pitch, int act, float alpha) {
    extern __shared__ __align__(16) uint8_t c0_smem[];
    float* lut = reinterpret_cast<float*>(c0_smem);             // 256
    float* in_s = lut + 256;                                     // (TH+2) x (TW+2) x 3
    float* w_s = in_s + (C0_TH + 2) * (C0_TW + 2) * 3 + 4;       // 27 x cout   (+4 keeps 16-byte alignment)
    float* b_s = w_s + 27 * cout;                                // cout
    __nv_bfloat16* o_s = reinterpret_cast<__nv_bfloat16*>(b_s + cout);  // TH*TW x cout

    const int tid = threadIdx.x;
    const int x0 = blockIdx.x * C0_TW, y0 = blockIdx.y * C0_TH, f = blockIdx.z;
    for (int i = tid; i < 256; i += C0_THREADS) lut[i] = norm_u8(i);
    for (int i = tid; i < 27 * cout; i += C0_THREADS) w_s[i] = __ldg(wgt + i);
    for (int i = tid; i < cout; i += C0_THREADS) b_s[i] = __ldg(bias + i);
    __syncthreads();
    const uint8_t* fr = frames + 1LL * f * h * wd * 3;
    constexpr int ROW = (C0_TW + 2) * 3;
    for (int i = tid; i < (C0_TH + 2) * ROW; i += C0_THREADS) {
        const int yy = i / ROW, rem = i - yy * ROW;
        const int xx = rem / 3;
        const int gy = y0 - 1 + yy, gx = x0 - 1 + xx;
        float v = 0.f;  // zero padding of the *normalised* input, as Conv pads=1 does
        if (gy >= 0 && gy < h && gx >= 0 && gx < wd) v = lut[__ldg(fr + (1LL * gy * wd + x0 - 1) * 3 + rem)];
        in_s[i] = v;
    }
    __syncthreads();

    const int tx = tid & 7, ty = tid >> 3;
    float xin[3][6][3];
#pragma unroll
    for (int r = 0; r < 3; ++r)
#pragma unroll
        for (int c = 0; c < 6; ++c)
#pragma unroll
            for (int ci = 0; ci < 3; ++ci) xin[r][c][ci] = in_s[((ty + r) * (C0_TW + 2) + 4 * tx + c) * 3 + ci];

    for (int co0 = 0; co0 < cout; co0 += 8) {
        float acc[4][8];
#pragma unroll
        for (int p = 0; p < 4; ++p)
#pragma unroll
            for (int j = 0; j < 8; ++j) acc[p][j] = b_s[co0 + j];
#pragma unroll
        for (int r = 0; r < 3; ++r)
#pragma unroll
            for (int s = 0; s < 3; ++s)
#pragma unroll
                for (int ci = 0; ci < 3; ++ci) {
                    const float4 w0 = *reinterpret_cast<const float4*>(w_s + ((r * 3 + s) * 3 + ci) * cout + co0);
                    const float4 w1 = *reinterpret_cast<const float4*>(w_s + ((r * 3 + s) * 3 + ci) * cout + co0 + 4);
#pragma unroll
                    for (int p = 0; p < 4; ++p) {
                        const float x = xin[r][p + s][ci];
                        acc[p][0] = fmaf(x, w0.x, acc[p][0]); acc[p][1] = fmaf(x, w0.y, acc[p][1]);
                        acc[p][2] = fmaf(x, w0.z, acc[p][2]); acc[p][3] = fmaf(x, w0.w, acc[p][3]);
                        acc[p][4] = fmaf(x, w1.x, acc[p][4]); acc[p][5] = fmaf(x, w1.y, acc[p][5]);
                        acc[p][6] = fmaf(x, w1.z, acc[p][6]); acc[p][7] = fmaf(x, w1.w, acc[p][7]);
                    }
                }
#pragma unroll
        for (int p = 0; p < 4; ++p) {
            if (MISH) {
#pragma unroll
                for (int j = 0; j < 8; ++j) acc[p][j] = mish_f32(acc[p][j]);
            } else if (act) {
#pragma unroll
                for (int j = 0; j < 8; ++j) acc[p][j] = acc[p][j] > 0.f ? acc[p][j] : acc[p][j] * alpha;
            }
            uint4 q;
            q.x = c0_pack(acc[p][0], acc[p][1]); q.y = c0_pack(acc[p][2], acc[p][3]);
            q.z = c0_pack(acc[p][4], acc[p][5]); q.w = c0_pack(acc[p][6], acc[p][7]);
            *reinterpret_cast<uint4*>(o_s + (ty * C0_TW + 4 * tx + p) * cout + co0) = q;
        }
    }
    __syncthreads();
    // coalesced write-out: consecutive threads -> consecutive 16-byte chunks of consecutive pixels
    const int chunks = cout / 8;
    for (int i = tid; i < C0_TH * C0_TW * chunks; i += C0_THREADS) {
        const int pix = i / chunks, ch = i - pix * chunks;
        const int py = pix / C0_TW, px = pix - py * C0_TW;
        const int gy = y0 + py, gx = x0 + px;
        if (gy < h && gx < wd) {
            const uint4 v = *reinterpret_cast<const uint4*>(o_s + pix * cout + ch * 8);
            *reinterpret_cast<uint4*>(out + ((1LL * f * h + gy) * wd + gx) * out_pitch + ch * 8) = v;
        }
    }
}

// ------------------------------------------------------------------------------------ first conv, im2col by descriptor
// The production first layer (Cout 16 / 32): im2col done by the tensor core's operand addressing instead of by threads.
//   * The CTA keeps a bf16 halo patch of the input in shared memory, one 16-byte unit per pixel
//     (R, G, B, 0, 0, 0, 0, 0): patch[18 rows][10 pixels] for a tile of 16 rows x 8 columns of output pixels.
//   * In the un-swizzled K-major operand layout a "core matrix" is 8 rows x 16 bytes with the rows 16 bytes apart,
//     the next 8-row group SBO bytes further, the next 16-byte K chunk LBO bytes further.  With the patch above,
//     8 consecutive pixels ARE a core matrix; SBO = one patch row (160 B) walks down the tile's 16 image rows, and
//     LBO = 16 B steps to the next pixel, i.e. the next filter tap of the same filter row.  So the A operand of the
//     MMA for filter row r, taps (s, s+1) is just the patch viewed from pixel (r, s): no per-pixel gather at all
//     (a version whose threads built the im2col rows spent ~54 shared-memory loads per output pixel on it: 391 us).
//   * K per filter row = 4 taps x 8 channels (tap 3 and channels 3..7 meet zero weights): 6 MMAs of 128 x Cout x 16
//     per tile, ~45 cycles each (dev/mma_rate.cu), against the 64 B/pixel the layer has to write to HBM.
//   * Epilogue: each warp drains its TMEM lane quarter (lane = pixel), bias + LeakyReLU in registers, bf16 rows staged
//     in shared memory and written by one TMA store per warp (box = Cout x 8 pixels x 4 rows).
//
// Stride 2 (YOLOv4-tiny: 416 -> 208) keeps the same trick with PAIR units: a 16-byte unit holds the RGB of input columns
// (2u, 2u+1) and two zero slots.  Output column x reads columns 2x-1 (tap 0: unit x-1's second half) and 2x, 2x+1
// (taps 1, 2: unit x), so K chunk 0 of filter row r is unit x-1 and chunk 1 unit x: LBO = 16 B again, 8 consecutive
// output pixels are 8 consecutive units, and SBO = TWO patch rows walks down the output rows.  K = 16 per filter row:
// 3 MMAs per 128 outputs; the patch of a 16 x 8 output tile is 33 rows x 9 units, no slack needed.
static constexpr int C0D_TW = 8, C0D_TH = 16;
template <int S> struct C0Geom;
template <> struct C0Geom<1> {
    static constexpr int PW = C0D_TW + 2, PH = C0D_TH + 2;     // halo patch, pixels
    static constexpr int PATCH_BYTES = (PH * PW + 8) * 16;     // + slack: tap 3 of the last pixels reads past the end
    static constexpr int MMAS = 6;                             // per tile: 3 filter rows x 2 K steps (taps 0-1, 2-3)
};
template <> struct C0Geom<2> {
    static constexpr int PW = C0D_TW + 1, PH = 2 * C0D_TH + 1;  // halo patch, pair units
    static constexpr int PATCH_BYTES = PH * PW * 16;
    static constexpr int MMAS = 3;                              // per tile: one per filter row
};

// Warp-specialised: a lock-step version (build -> sync -> MMA -> wait -> drain per tile) spent most of a tile's ~5000
// cycles waiting at its barriers (ncu: barrier + load-use stalls), so the three stages run decoupled over rings:
//   warps 13..20 builders: warp b owns patch slot b and every 8th tile; it gathers the 180 halo pixels of a tile (6 per
//                lane, the bytes of its next two tiles already in registers), converts through the LUT, publishes the patch
//   warp 12      issues the 6 MMAs of a tile into a ring of 8 TMEM accumulators
//   warps 0..11  three epilogue groups (tiles it % 3; TMEM lane quarter = warp % 4): bias + LeakyReLU, bf16 rows
//                staged in shared memory, one TMA store per warp and tile
static constexpr int C0W_GROUPS = 3;                       // epilogue groups of 4 warps
static constexpr int C0W_EPI_WARPS = 4 * C0W_GROUPS;       // warps 0 .. 11
static constexpr int C0W_MMA_WARP = C0W_EPI_WARPS;         // warp 12
static constexpr int C0W_BUILD_WARPS = 8;                  // one per patch slot
static constexpr int C0W_THREADS = (C0W_EPI_WARPS + 1 + C0W_BUILD_WARPS) * 32, C0W_PATCHES = 8, C0W_ACCS = 8;  // ring depth: the
// publish -> MMA -> drain -> release round trip is ~3000 cycles, so 4 slots capped the kernel at ~800 cycles per tile
// q = x / d for 0 <= x < 2^24 and d < 2^12 as one 64-bit multiply: m = ceil(2^40 / d)
__device__ __forceinline__ int div_magic(int x, unsigned long long m) { return static_cast<int>((static_cast<unsigned long long>(x) * m) >> 40); }

// h, wd: the input frame; the output map is (h / S, wd / S) (stride 2: h and wd even)
// MISH: the activation is Mish (act.cuh); act / alpha are not read
template <int S, bool MISH = false>
__global__ void __launch_bounds__(C0W_THREADS)
conv0_ws_kernel(const uint8_t* __restrict__ frames, const float* __restrict__ wgt, const float* __restrict__ bias,
                const __grid_constant__ CUtensorMap tm_out, int n, int h, int wd, int cout, int act, float alpha,
                unsigned long long m_per_frame, unsigned long long m_tiles_x, int pool2) {
    using G = C0Geom<S>;
    constexpr int C0D_PATCH_BYTES = G::PATCH_BYTES;
    constexpr int C0W_PPL = (G::PH * G::PW + 31) / 32;  // patch units per builder lane
    extern __shared__ __align__(1024) uint8_t c0w_dyn[];        // patch ring
    uint8_t (*s_patch)[C0D_PATCH_BYTES] = reinterpret_cast<uint8_t (*)[C0D_PATCH_BYTES]>(c0w_dyn);
    __shared__ __align__(1024) uint8_t s_w[12 * 32 * 16];       // B: [K chunk 0..11][32 filters][16 B]
    __shared__ __align__(1024) uint8_t s_out[C0W_EPI_WARPS][2048];  // per epilogue warp: one staging tile of 32 pixels x 64 B
    __shared__ uint16_t lut[256];
    __shared__ __align__(8) uint64_t patch_full[C0W_PATCHES], patch_empty[C0W_PATCHES], acc_full[C0W_ACCS], acc_empty[C0W_ACCS];
    __shared__ uint32_t tmem_slot;

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    for (int i = tid; i < 256; i += C0W_THREADS) {
        const __nv_bfloat16 v = __float2bfloat16(norm_u8(i));
        lut[i] = *reinterpret_cast<const uint16_t*>(&v);
    }
    if constexpr (S == 1) {
        for (int i = tid; i < 12 * 32; i += C0W_THREADS) {
            const int c = i >> 5, f = i & 31, r = c >> 2, sx = c & 3;
            float w0 = 0.f, w1 = 0.f, w2 = 0.f;
            if (sx < 3 && f < cout) {
                const float* wp = wgt + ((r * 3 + sx) * 3) * cout + f;
                w0 = __ldg(wp); w1 = __ldg(wp + cout); w2 = __ldg(wp + 2 * cout);
            }
            *reinterpret_cast<uint4*>(s_w + i * 16) = make_uint4(c0_pack(w0, w1), c0_pack(w2, 0.f), 0u, 0u);
        }
    } else {
        // chunk 2r: slots 3..5 = tap (r, 0) (the second pixel of unit x-1); chunk 2r+1: slots 0..2 = tap (r, 1), 3..5 = tap (r, 2)
        for (int i = tid; i < 6 * 32; i += C0W_THREADS) {
            const int c = i >> 5, f = i & 31, r = c >> 1;
            float w[6] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
            if (f < cout) {
#pragma unroll
                for (int j = 0; j < 6; ++j) {
                    const int sx = (c & 1) ? 1 + j / 3 : 0;
                    if ((c & 1) || j >= 3) w[j] = __ldg(wgt + ((r * 3 + sx) * 3 + j % 3) * cout + f);
                }
            }
            *reinterpret_cast<uint4*>(s_w + i * 16) = make_uint4(c0_pack(w[0], w[1]), c0_pack(w[2], w[3]), c0_pack(w[4], w[5]), 0u);
        }
    }
    for (int i = tid; i < C0W_PATCHES * C0D_PATCH_BYTES / 16; i += C0W_THREADS) reinterpret_cast<uint4*>(c0w_dyn)[i] = make_uint4(0u, 0u, 0u, 0u);
    if (tid == 0) {
        for (int i = 0; i < C0W_PATCHES; ++i) { ptx::mbar_init(&patch_full[i], 1); ptx::mbar_init(&patch_empty[i], 1); }
        for (int i = 0; i < C0W_ACCS; ++i) { ptx::mbar_init(&acc_full[i], 1); ptx::mbar_init(&acc_empty[i], 4); }
        ptx::fence_barrier_init();
        ptx::tma_prefetch_desc(&tm_out);
    }
    if (warp == C0W_MMA_WARP) {
        ptx::tmem_alloc(&tmem_slot, 32 * C0W_ACCS);
        ptx::tmem_relinquish();
    }
    ptx::fence_proxy_async();  // the weight tile and the zeroed patch slack are read by the tensor core
    ptx::tc_fence_before();
    __syncthreads();
    ptx::tc_fence_after();
    const uint32_t tmem = tmem_slot;
    ptx::grid_dep_launch();  // the next layer may start its set-up on SMs as they drain (it waits before reading)

    const int tiles_x = (wd / S + C0D_TW - 1) / C0D_TW, tiles_y = (h / S + C0D_TH - 1) / C0D_TH;
    const int per_frame = tiles_x * tiles_y;
    const int total = n * per_frame;  // < 2^31 by far
    const int my_tiles = (total > static_cast<int>(blockIdx.x)) ? (total - 1 - static_cast<int>(blockIdx.x)) / static_cast<int>(gridDim.x) + 1 : 0;

    if (warp > C0W_MMA_WARP) {
        // ---------------------------------------------------------------- builders: u8 halo patch -> bf16, 16 B per pixel
        // warp s of this role owns patch slot s and every 8th tile; a lane handles 6 fixed patch pixels, whose
        // offsets inside a tile are computed once (one warp's dependent-instruction latency per tile is what bounds
        // this role, so the per-tile work is kept to the loads, the LUT and the stores)
        // (stride 2: a unit is 2 pixels = 6 bytes at an even offset, loaded as 3 u16; the frames are 2-byte aligned)
        const int slot = warp - C0W_MMA_WARP - 1;
        int pq[C0W_PPL], ppy[C0W_PPL], ppx[C0W_PPL], poff[C0W_PPL];
#pragma unroll
        for (int k = 0; k < C0W_PPL; ++k) {
            const int q = lane + 32 * k;  // patch unit
            pq[k] = q < G::PH * G::PW ? q : -1;
            ppy[k] = q / G::PW;
            ppx[k] = q - ppy[k] * G::PW;
            poff[k] = (ppy[k] * wd + S * ppx[k]) * 3;
        }
        // two register sets: the bytes of this warp's next TWO tiles are in flight while it converts the current one
        // (the loads come from DRAM: one tile of look-ahead left the warp waiting on them)
        uint32_t raw_a[3 * C0W_PPL], raw_b[3 * C0W_PPL], inside_a = 0, inside_b = 0;
#pragma unroll
        for (int i = 0; i < 3 * C0W_PPL; ++i) raw_a[i] = raw_b[i] = 0;
        auto fetch = [&](int it, uint32_t (&raw)[3 * C0W_PPL], uint32_t& inside) {  // no arithmetic on the bytes here: it would wait for the loads
            const int tile = blockIdx.x + it * gridDim.x;
            const int f = div_magic(tile, m_per_frame);
            const int rem = tile - f * per_frame;
            const int ty = div_magic(rem, m_tiles_x), tx = rem - ty * tiles_x;
            const int y0 = ty * C0D_TH * S - 1, x0 = tx * C0D_TW - 1;  // first patch row (input) and unit (input pixel or pair)
            const uint8_t* origin = frames + (1LL * f * h * wd + 1LL * y0 * wd + S * x0) * 3;  // may point before the frame: only used when inside
            inside = 0;
#pragma unroll
            for (int k = 0; k < C0W_PPL; ++k) {
                const int gy = y0 + ppy[k], gx = x0 + ppx[k];
                if (pq[k] >= 0 && gy >= 0 && gy < h && gx >= 0 && gx < wd / S) {  // outside: zero padding of the normalised input
                    const uint8_t* sp = origin + poff[k];
                    inside |= 1u << k;
                    if constexpr (S == 1) {
                        raw[3 * k] = __ldg(sp);
                        raw[3 * k + 1] = __ldg(sp + 1);
                        raw[3 * k + 2] = __ldg(sp + 2);
                    } else {
                        const uint16_t* sp16 = reinterpret_cast<const uint16_t*>(sp);
                        raw[3 * k] = __ldg(sp16);
                        raw[3 * k + 1] = __ldg(sp16 + 1);
                        raw[3 * k + 2] = __ldg(sp16 + 2);
                    }
                }
            }
        };
        auto publish = [&](const uint32_t (&raw)[3 * C0W_PPL], uint32_t inside, uint32_t phase) {
            ptx::mbar_wait(&patch_empty[slot], phase ^ 1);
#pragma unroll
            for (int k = 0; k < C0W_PPL; ++k) {
                if (pq[k] >= 0) {
                    uint4 v = make_uint4(0u, 0u, 0u, 0u);
                    if (inside & (1u << k)) {
                        if constexpr (S == 1) {
                            v.x = static_cast<uint32_t>(lut[raw[3 * k]]) | (static_cast<uint32_t>(lut[raw[3 * k + 1]]) << 16);
                            v.y = static_cast<uint32_t>(lut[raw[3 * k + 2]]);
                        } else {  // (R0 G0) (B0 R1) (G1 B1): byte pairs in memory order
                            v.x = static_cast<uint32_t>(lut[raw[3 * k] & 255]) | (static_cast<uint32_t>(lut[raw[3 * k] >> 8]) << 16);
                            v.y = static_cast<uint32_t>(lut[raw[3 * k + 1] & 255]) | (static_cast<uint32_t>(lut[raw[3 * k + 1] >> 8]) << 16);
                            v.z = static_cast<uint32_t>(lut[raw[3 * k + 2] & 255]) | (static_cast<uint32_t>(lut[raw[3 * k + 2] >> 8]) << 16);
                        }
                    }
                    *reinterpret_cast<uint4*>(&s_patch[slot][pq[k] * 16]) = v;
                }
            }
        };
        auto signal = [&]() {
            ptx::fence_proxy_async();  // generic-proxy writes of the patch -> visible to the tensor core
            __syncwarp();
            if (lane == 0) ptx::mbar_arrive(&patch_full[slot]);
        };
        uint32_t phase = 0;
        if (slot < my_tiles) fetch(slot, raw_a, inside_a);
        if constexpr (S == 2) {
            // one register set: 10 units per lane (30 loads in flight) leave no room for a second one in 80 registers
            for (int it = slot; it < my_tiles; it += C0W_PATCHES) {
                publish(raw_a, inside_a, phase);
                if (it + C0W_PATCHES < my_tiles) fetch(it + C0W_PATCHES, raw_a, inside_a);
                signal();
                phase ^= 1;
            }
        } else {
            if (slot + C0W_PATCHES < my_tiles) fetch(slot + C0W_PATCHES, raw_b, inside_b);
            for (int it = slot; it < my_tiles; it += 2 * C0W_PATCHES) {
                publish(raw_a, inside_a, phase);
                if (it + 2 * C0W_PATCHES < my_tiles) fetch(it + 2 * C0W_PATCHES, raw_a, inside_a);
                signal();
                phase ^= 1;
                if (it + C0W_PATCHES >= my_tiles) break;
                publish(raw_b, inside_b, phase);
                if (it + 3 * C0W_PATCHES < my_tiles) fetch(it + 3 * C0W_PATCHES, raw_b, inside_b);
                signal();
                phase ^= 1;
            }
        }
    } else if (warp == C0W_MMA_WARP) {
        // ---------------------------------------------------------------- MMA issuer
        // This warp's issue rate bounds the kernel (6 MMAs + 2 commits per 128 pixels), so everything it needs is a
        // warp-uniform value prepared outside the loop and the elected lane only issues (an `if (lane == 0)` body made
        // the compiler wrap every tcgen05.mma in an ELECT loop: ~950 cycles per tile).
        const uint32_t idesc = ptx::make_idesc_bf16_f32(128, cout);
        // un-swizzled K-major descriptors: LBO (K chunk stride) and SBO (8-row group stride), in 16-byte units
        auto desc = [](uint32_t addr, uint32_t lbo, uint32_t sbo) -> uint64_t {
            return static_cast<uint64_t>((addr >> 4) & 0x3FFF) | (static_cast<uint64_t>((lbo >> 4) & 0x3FFF) << 16) |
                   (static_cast<uint64_t>((sbo >> 4) & 0x3FFF) << 32) | (static_cast<uint64_t>(1) << 46);
        };
        const uint32_t w_addr = __shfl_sync(0xffffffffu, ptx::smem_u32(s_w), 0);
        const uint32_t p_addr0 = __shfl_sync(0xffffffffu, ptx::smem_u32(&s_patch[0][0]), 0);
        const uint32_t bar_pe = __shfl_sync(0xffffffffu, ptx::smem_u32(&patch_empty[0]), 0);
        const uint32_t bar_pf = __shfl_sync(0xffffffffu, ptx::smem_u32(&patch_full[0]), 0);
        const uint32_t bar_af = __shfl_sync(0xffffffffu, ptx::smem_u32(&acc_full[0]), 0);
        const uint32_t bar_ae = __shfl_sync(0xffffffffu, ptx::smem_u32(&acc_empty[0]), 0);
        const uint32_t tmem_u = __shfl_sync(0xffffffffu, tmem, 0);
        const uint64_t a0 = desc(p_addr0, 16, S * G::PW * 16);
        uint64_t bd[G::MMAS], aoff[G::MMAS];
#pragma unroll
        for (int j = 0; j < G::MMAS; ++j) {
            if constexpr (S == 1) {
                const int r = j >> 1, s0 = (j & 1) * 2;  // filter row, first of the two taps of this K step
                bd[j] = desc(w_addr + (r * 4 + s0) * 512, 512, 128);
                aoff[j] = static_cast<uint64_t>(r * G::PW + s0);  // 16-byte units
            } else {
                bd[j] = desc(w_addr + 2 * j * 512, 512, 128);  // filter row j: chunks 2j, 2j + 1
                aoff[j] = static_cast<uint64_t>(j * G::PW);    // patch row j, unit 0 (= output column -1 of the tile)
            }
        }
        const bool issuer = ptx::elect_one();
        uint32_t slot = 0, phase = 0;
        for (int it = 0; it < my_tiles; ++it) {
            ptx::mbar_wait_addr(bar_ae + 8u * slot, phase ^ 1);
            ptx::mbar_wait_addr(bar_pf + 8u * slot, phase);
            ptx::tc_fence_after();
            const uint64_t ad = a0 + slot * (C0D_PATCH_BYTES / 16);
            const uint32_t d = tmem_u + slot * 32;
            if (issuer) {
#pragma unroll
                for (int j = 0; j < G::MMAS; ++j) ptx::umma_bf16(d, ad + aoff[j], bd[j], idesc, j ? 1u : 0u);
                ptx::umma_commit_addr(bar_pe + 8u * slot);
                ptx::umma_commit_addr(bar_af + 8u * slot);
            }
            __syncwarp();
            if (++slot == C0W_ACCS) { slot = 0; phase ^= 1; }  // C0W_PATCHES == C0W_ACCS: one index walks both rings
        }
    } else {
        // ---------------------------------------------------------------- epilogue group g: tiles it = g, g + groups, ...
        static_assert(C0W_PATCHES == C0W_ACCS && C0W_ACCS == 8 && C0W_BUILD_WARPS == C0W_PATCHES, "ring indexing below assumes 8 + 8");
        const int group = warp >> 2, quarter = warp & 3;  // TMEM lane quarter = warp % 4
        float bv[32];
#pragma unroll
        for (int c = 0; c < 32; ++c) bv[c] = (c < cout) ? __ldg(bias + c) : 0.f;
        const float alpha_eff = act ? alpha : 1.0f;
        for (int it = group; it < my_tiles; it += C0W_GROUPS) {
            const int as = it & 7;
            const uint32_t aphase = (it >> 3) & 1;
            const int tile = blockIdx.x + it * gridDim.x;
            const int f = div_magic(tile, m_per_frame);
            const int rem = tile - f * per_frame;
            const int ty = div_magic(rem, m_tiles_x), tx = rem - ty * tiles_x;
            ptx::mbar_wait(&acc_full[as], aphase);
            ptx::tc_fence_after();
            uint32_t acc[32];
            ptx::tmem_ld_32x32(tmem + as * 32 + (static_cast<uint32_t>(quarter * 32) << 16), acc);
            ptx::tmem_ld_wait();
            ptx::tc_fence_before();
            __syncwarp();
            if (lane == 0) ptx::mbar_arrive(&acc_empty[as]);
            // lane = pixel (tile rows 4q .. 4q+3, 8 pixels each); bias + LeakyReLU as max(x, alpha x)
            uint32_t pk[16];
            const float2 a2 = make_float2(alpha_eff, alpha_eff);
#pragma unroll
            for (int c = 0; c < 16; ++c) {  // two columns per FADD2 / FMUL2
                float2 x = __fadd2_rn(make_float2(__uint_as_float(acc[2 * c]), __uint_as_float(acc[2 * c + 1])), make_float2(bv[2 * c], bv[2 * c + 1]));
                if constexpr (MISH) {
                    x = make_float2(mish_f32(x.x), mish_f32(x.y));
                } else if (act != 2) {
                    const float2 m = __fmul2_rn(x, a2);
                    x.x = fmaxf(x.x, m.x);
                    x.y = fmaxf(x.y, m.y);
                } else {
                    x.x = x.x > 0.f ? x.x : x.x * alpha;
                    x.y = x.y > 0.f ? x.y : x.y * alpha;
                }
                pk[c] = c0_pack(x.x, x.y);
            }
            // MaxPool(2, 2) of the activation (YOLOv3-tiny's first pool), in place: the 2x2 window of lane l = (row l >> 3,
            // column l & 7) is lanes l, l^1, l^8, l^9; lanes with even row and column keep the maximum
            if (pool2) {
#pragma unroll
                for (int c = 0; c < 16; ++c) {
                    uint32_t v = c0_max(pk[c], __shfl_xor_sync(0xffffffffu, pk[c], 1));
                    pk[c] = c0_max(v, __shfl_xor_sync(0xffffffffu, v, 8));
                }
            }
            uint8_t* so = s_out[warp];
            if (lane == 0) ptx::tma_store_wait_read<0>();  // this warp's previous store (two tiles ago) has finished reading the buffer
            __syncwarp();
            if (pool2) {
                // pooled box [2 rows][4 pixels x cout]: the 8 surviving pixels, dense
                const int pp = (lane >> 4) * 4 + ((lane & 7) >> 1);
                if ((lane & 9) == 0) {
                    if (cout == 32) {
#pragma unroll
                        for (int c = 0; c < 4; ++c)
                            *reinterpret_cast<uint4*>(so + pp * 64 + (c << 4)) = make_uint4(pk[4 * c], pk[4 * c + 1], pk[4 * c + 2], pk[4 * c + 3]);
                    } else {
#pragma unroll
                        for (int c = 0; c < 2; ++c)
                            *reinterpret_cast<uint4*>(so + pp * 32 + (c << 4)) = make_uint4(pk[4 * c], pk[4 * c + 1], pk[4 * c + 2], pk[4 * c + 3]);
                    }
                }
                ptx::fence_proxy_async();
                __syncwarp();
                if (lane == 0) {
                    ptx::tma_store_3d(&tm_out, so, tx * (C0D_TW / 2) * cout, ty * (C0D_TH / 2) + 2 * quarter, f);  // clipped at the frame edges
                    ptx::tma_store_commit();
                }
                continue;
            }
            // dense rows [4 image rows][8 pixels][cout]: with pitch == cout the 8 pixels of an image row are one contiguous
            // 8*cout*2-byte run in global memory: the TMA store moves 4 wide rows
            if (cout == 32) {
#pragma unroll
                for (int c = 0; c < 4; ++c)  // (un-swizzled: 4-way bank conflicts on 4 stores per tile, noise)
                    *reinterpret_cast<uint4*>(so + lane * 64 + (c << 4)) = make_uint4(pk[4 * c], pk[4 * c + 1], pk[4 * c + 2], pk[4 * c + 3]);
            } else {
#pragma unroll
                for (int c = 0; c < 2; ++c)
                    *reinterpret_cast<uint4*>(so + lane * 32 + (c << 4)) = make_uint4(pk[4 * c], pk[4 * c + 1], pk[4 * c + 2], pk[4 * c + 3]);
            }
            ptx::fence_proxy_async();
            __syncwarp();
            if (lane == 0) {
                ptx::tma_store_3d(&tm_out, so, tx * C0D_TW * cout, ty * C0D_TH + 4 * quarter, f);  // clipped at the frame edges
                ptx::tma_store_commit();
            }
        }
        if (lane == 0) ptx::tma_store_wait<0>();
    }
    ptx::tc_fence_before();
    __syncthreads();
    if (warp == C0W_MMA_WARP) {
        ptx::tc_fence_after();
        ptx::tmem_dealloc(tmem, 32 * C0W_ACCS);
    }
}

template <bool MISH>
static bool conv0_smem_attrs() {
    return cudaFuncSetAttribute(conv0_u8_kernel<MISH>, cudaFuncAttributeMaxDynamicSharedMemorySize, 100 * 1024) == cudaSuccess &&
           cudaFuncSetAttribute(conv0_ws_kernel<1, MISH>, cudaFuncAttributeMaxDynamicSharedMemorySize, C0W_PATCHES * C0Geom<1>::PATCH_BYTES) == cudaSuccess &&
           cudaFuncSetAttribute(conv0_ws_kernel<2, MISH>, cudaFuncAttributeMaxDynamicSharedMemorySize, C0W_PATCHES * C0Geom<2>::PATCH_BYTES) == cudaSuccess;
}

int kernels_init() { return conv0_smem_attrs<false>() && conv0_smem_attrs<true>() ? 0 : -1; }

int launch_conv0_u8(const uint8_t* frames, const float* w, const float* bias, __nv_bfloat16* out, int n, int h,
                    int wd, int cout, int stride, int out_pitch, int act, float alpha, int pool2, cudaStream_t s) {
    const bool mish = act == 2;
    const int act_mode = act ? ((alpha >= 0.f && alpha <= 1.f) ? 1 : 2) : 0;
    if (stride != 1 && stride != 2) return -1;
    // stride 2: tensor cores only (even input, dense Cout 16 / 32 rows, 2-byte aligned frames for the pair loads)
    if (stride == 2 && (((h | wd) & 1) || pool2 || (reinterpret_cast<uintptr_t>(frames) & 1))) return -1;
    const int sh = h / stride, sw = wd / stride;  // the convolution's output map
    const long long tiles = 1LL * n * ((sw + C0D_TW - 1) / C0D_TW) * ((sh + C0D_TH - 1) / C0D_TH);
    const int tx = (sw + C0D_TW - 1) / C0D_TW, per_frame = tx * ((sh + C0D_TH - 1) / C0D_TH);
    if ((cout == 16 || cout == 32) && out_pitch == cout && (reinterpret_cast<uintptr_t>(out) & 15) == 0 &&
        tiles < (1LL << 24) && per_frame < 65536) {  // (ranges of the multiply-shift division)
        // dense NHWC output: an image row is one run of W*C elements; TMA store box = 8 pixels x 4 rows
        CUtensorMap tm;
        // (pooled: the output map is (h/2, wd/2) and a warp's box its 2 x 4 surviving pixels)
        const int oh = pool2 ? h / 2 : sh, ow = pool2 ? wd / 2 : sw;
        if (pool2 && ((h | wd) & 1)) return -1;
        const unsigned long long dims[3] = {static_cast<unsigned long long>(cout) * ow, static_cast<unsigned long long>(oh),
                                            static_cast<unsigned long long>(n)};
        const unsigned long long strides[2] = {2ULL * cout * ow, 2ULL * cout * ow * oh};
        const unsigned box[3] = {static_cast<unsigned>(cout) * (pool2 ? C0D_TW / 2 : C0D_TW), pool2 ? 2u : 4u, 1};
        if (encode_tiled_bf16(&tm, out, 3, dims, strides, box, 0)) return -1;
        const int blocks = static_cast<int>(tiles < 148LL ? tiles : 148LL);
        const unsigned long long one40 = 1ULL << 40;
        const unsigned long long mf = (one40 + per_frame - 1) / per_frame, mx = (one40 + tx - 1) / tx;
        if (stride == 2 && mish)
            conv0_ws_kernel<2, true><<<blocks, C0W_THREADS, C0W_PATCHES * C0Geom<2>::PATCH_BYTES, s>>>(frames, w, bias, tm, n, h, wd, cout, act_mode, alpha, mf, mx, 0);
        else if (stride == 2)
            conv0_ws_kernel<2><<<blocks, C0W_THREADS, C0W_PATCHES * C0Geom<2>::PATCH_BYTES, s>>>(frames, w, bias, tm, n, h, wd, cout, act_mode, alpha, mf, mx, 0);
        else if (mish)
            conv0_ws_kernel<1, true><<<blocks, C0W_THREADS, C0W_PATCHES * C0Geom<1>::PATCH_BYTES, s>>>(frames, w, bias, tm, n, h, wd, cout, act_mode, alpha, mf, mx, pool2);
        else
            conv0_ws_kernel<1><<<blocks, C0W_THREADS, C0W_PATCHES * C0Geom<1>::PATCH_BYTES, s>>>(frames, w, bias, tm, n, h, wd, cout, act_mode, alpha, mf, mx, pool2);
        return cudaPeekAtLastError() == cudaSuccess ? 0 : -1;  // (peek: the caller reports the reason)
    }
    // any other stride-1 first layer (Cout up to 64, any pitch): CUDA cores
    if (pool2 || stride != 1) return -1;  // (the planner fuses the pool, and takes stride 2, only for shapes the kernel above takes)
    const size_t smem = (256 + (C0_TH + 2) * (C0_TW + 2) * 3 + 4 + 27 * cout + cout) * sizeof(float) +
                        static_cast<size_t>(C0_TH) * C0_TW * cout * 2;
    dim3 grid((wd + C0_TW - 1) / C0_TW, (h + C0_TH - 1) / C0_TH, n);
    if (mish) conv0_u8_kernel<true><<<grid, C0_THREADS, smem, s>>>(frames, w, bias, out, h, wd, cout, out_pitch, act, alpha);
    else conv0_u8_kernel<<<grid, C0_THREADS, smem, s>>>(frames, w, bias, out, h, wd, cout, out_pitch, act, alpha);
    return cudaPeekAtLastError() == cudaSuccess ? 0 : -1;  // (peek: the caller reports the reason)
}

}  // namespace fd
