// conv_tc.cu — persistent, warp-specialised implicit-GEMM convolution on tcgen05 / TMEM / TMA.
//
//   D[M = N*Ho*Wo, Cout] = im2col(X)[M, K = kh*kw*Cin] * W[Cout, K]^T     (bf16 x bf16 -> fp32)
//   epilogue: + bias (BatchNorm folded) -> LeakyReLU -> (+ residual) -> bf16 NHWC slice | fp32 head rows
//
// Stands in for the Conv/BatchNormalization/LeakyRelu/Add (and the Resize+Concat that follow a
// branch conv) nodes ONNX Runtime executes at reference server/detector.py:135.
//
// CTA = 12 warps: warp 0  TMA producer (A: 2D tiled map for 1x1, im2col map for 3x3; B: 2D tiled)
//                 warp 1  tcgen05.mma issuer (128 x BLOCK_N x 16 per instruction; 256 x 256 x 16 for a CTA pair)
//                 warp 2  TMEM allocator
//                 warps 4..11  epilogue: all eight on the same tile (TMEM lane quarter = warp % 4, the two warps of a
//                              quarter split the tile's columns)
// Kernel instantiations: <BLOCK_N, TWO, SWAP, STRIP> — single CTA tiles (32..256 columns), CTA pairs (cta_group::2),
// the swapped form for 128-channel outputs, and the strip form of the pair kernel for 3x3 / stride 1 / pad 1 layers
// (ConvParams::strip: one zero-padded flat pixel strip per channel block, the nine taps by descriptor row offsets).
// Pipelines: smem ring (full/empty mbarriers, num_stages deep) between TMA and MMA; two TMEM accumulator stages
// (tmem_full/tmem_empty) between MMA and epilogue, so a tile's epilogue overlaps the next tile's main loop.
// Epilogue: tcgen05.ld (next chunk in flight) -> bias from the constant bank + max(x, alpha x) on packed fp32 pairs ->
// (+ residual, 256-bit row loads) -> bf16 rows staged with the 128-byte swizzle -> TMA stores; fp32 head rows the same
// way; strip mode stores rows directly (its rows are scattered over the image).  The production flag combinations have
// compile-time copies of the epilogue (STRIP / FAST / PLAIN): short-K layers run at the epilogue's instruction count.
#include "conv_tc.h"
#include "act.cuh"
#include "options.h"
#include "ptx.cuh"

#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <type_traits>

namespace fd {

// Developer instrumentation (per-role cycle counters in ConvParams::prof, the ConvParams::debug switches that skip loads /
// MMAs / stores) exists only in builds with -DFASTDET_DEV (csrc/dev/test_conv); the library's kernels carry none of it.
#ifdef FASTDET_DEV
static constexpr bool kDev = true;
#else
static constexpr bool kDev = false;
#endif

static constexpr int BLOCK_M = 128;
static constexpr int NUM_THREADS = 384;
static constexpr int MAX_STAGES = 32;
// dynamic shared memory map (after aligning the base to 1024 B):
//   [0, 1024)       full[32] + empty[32] + tmem_full[2] + tmem_empty[2] mbarriers, TMEM base slot
//   [1024, 33792)   epilogue staging: 8 warps x 4 KB (two 32-row x 64-byte bf16 chunk buffers each)
//   [33792, ...)    operand ring: num_stages x (A stage | B stage), every stage 1024-byte aligned
static constexpr int SMEM_STAGING_OFF = 1024;
static constexpr int SMEM_RING_OFF = 1024 + 8 * 4096;
static constexpr int SMEM_LIMIT = 227 * 1024;

template <int BLOCK_N>
struct TileCfg {
    static constexpr int TMEM_COLS = (2 * BLOCK_N < 32) ? 32 : 2 * BLOCK_N;  // 64,128,256,512: powers of two
};

__device__ __forceinline__ uint32_t pack_bf16(float a, float b) {
    __nv_bfloat162 v = __floats2bfloat162_rn(a, b);
    return *reinterpret_cast<uint32_t*>(&v);
}
__device__ __forceinline__ float bf16_lo(uint32_t u) { return __uint_as_float(u << 16); }
__device__ __forceinline__ float bf16_hi(uint32_t u) { return __uint_as_float(u & 0xFFFF0000u); }

// bias + activation on two accumulator columns at once (FADD2 / FMUL2 are two fp32 lanes per instruction).
// Branch-free for the two cases YOLO has: LeakyReLU with 0 <= alpha <= 1 is max(x, alpha*x), and a linear layer is
// the same expression with alpha = 1 (x*1 = x exactly).  GENERIC (alpha outside [0,1]) uses the select form.
template <bool GENERIC>
__device__ __forceinline__ float2 bias_act2(uint32_t a0, uint32_t a1, float b0, float b1, float2 alpha2) {
    float2 x = __fadd2_rn(make_float2(__uint_as_float(a0), __uint_as_float(a1)), make_float2(b0, b1));
    if (GENERIC) {
        x.x = x.x > 0.f ? x.x : x.x * alpha2.x;
        x.y = x.y > 0.f ? x.y : x.y * alpha2.x;
    } else {
        const float2 m = __fmul2_rn(x, alpha2);
        x.x = fmaxf(x.x, m.x);
        x.y = fmaxf(x.y, m.y);
    }
    return x;
}

// One accumulator tile (128 rows x BLOCK_N columns of this CTA's TMEM) -> global memory.
//   taddr0     TMEM address of the warp's lane quarter at the accumulator stage's first column
//   m_base     global output-pixel index of the warp's first row
//   empty_addr shared address of the tmem_empty barrier to arrive on once the accumulator is drained
//              (for a CTA pair: the leader's barrier, reached through the shared::cluster window)
// Shared-memory LOADS cost ~500 cycles here (the LSU queues behind the TMA fills and the tensor core's operand
// reads — measured), and two epilogue warps per scheduler cannot hide that, so the path has none: the bias comes
// from the constant bank (kernel parameter), the residual is read row-major straight from global memory one chunk
// ahead, the bf16 rows are staged with fire-and-forget stores and leave through a TMA store, and the TMEM load of
// chunk c+1 is in flight while chunk c is processed.
//   p.epi_mode 0: bf16 NHWC slice via TMA store (+ residual)   1: fp32 head rows, direct stores
//              2: bf16 with x2 nearest upsampling (2 layers): staged, re-read transposed, 4 coalesced stores per row
// STRIP / RES: compile-time copies for the strip-mode kernel (RES = the layer has a residual input); with STRIP = false the
// residual, the store mode and the activation form are run-time properties of the launch.  The strip kernel's epilogue is
// its critical path (the strips took the main loop off it), so every flag it does not need is compiled out.
// FAST: the common production path of the other kernels — bf16 output through 128-byte TMA stores, max(x, alpha x)
// activation, whole-K tiles — with the same flags fixed at compile time (1x1 layers have K loops of 4-16 K blocks, shorter
// than one epilogue: they run at the epilogue's speed, which is its instruction count).
// MISH: the kernel's activation is Mish (act.cuh) in every copy; the copies without it keep max(x, alpha x) / the select form.
template <int BLOCK_N, bool STRIP = false, bool RES = false, bool FAST = false, bool MISH = false>
__device__ __forceinline__ void epilogue_tile(const ConvParams& p, const CUtensorMap* tm_out, uint32_t taddr0,
                                              uint8_t* stage, int& sbuf, long long m_base, int n0, int lane, int half,
                                              uint32_t full_addr, uint32_t aphase, uint32_t empty_addr, long long* t_acc,
                                              int tile = 0, int part = 0, int region = 0) {
    // the two warps that share a TMEM lane quarter split the tile's columns: all 8 epilogue warps work on the same
    // tile, which halves the time the last tile of a launch (nothing left to overlap with) spends here
    constexpr int HALF_N = BLOCK_N >= 64 ? BLOCK_N / 2 : BLOCK_N;
    // (a 32-column tile is one chunk: there the two warps take alternate tiles instead, see the kernel)
    const int c_begin = (BLOCK_N >= 64) ? half * HALF_N : 0;
    const int c_end = c_begin + HALF_N;
    constexpr bool FIXED = STRIP || FAST;
    const int mode = FIXED ? 0 : p.epi_mode;
    const bool generic_act = !FIXED && p.act == 2;
    const float alpha_eff = p.act ? p.alpha : 1.0f;
    const float2 alpha2 = make_float2(alpha_eff, alpha_eff);
    long long m_own = m_base + lane;  // the pixel row this lane holds
    bool own_ok = m_own < p.M;
    if (STRIP) {  // m_base counts zero-padded flat positions: back to the pixel row, pad positions hold nothing
        const int q = static_cast<int>(m_own), plane = p.strip_wp * p.strip_hp;
        const int img = q / plane, rem = q - img * plane, yp = rem / p.strip_wp, xp = rem - yp * p.strip_wp;
        own_ok = q < p.strip_total_q && yp >= 1 && yp <= p.ho && xp >= 1 && xp <= p.wo;
        m_own = own_ok ? (static_cast<long long>(img) * p.ho + (yp - 1)) * p.wo + (xp - 1) : 0;
    }
    const bool has_res = FIXED ? RES : (mode == 0 && p.residual != nullptr);
    const __nv_bfloat16* res_row = p.residual + m_own * p.res_pitch + n0;
    ptx::U32x8 rnext[2];
    // this lane's 64 bytes of the residual row for chunk c0, as two 32-byte loads: every L2 sector is requested once
    // (16-byte loads would fetch each sector twice, and this kernel is bound by L2 -> SM traffic)
    auto fetch_res = [&](int c0) {
#pragma unroll
        for (int i = 0; i < 2; ++i) {
#pragma unroll
            for (int e = 0; e < 8; ++e) rnext[i].v[e] = 0u;
            if (!(has_res && own_ok && n0 + c0 + 16 * i < p.cout)) continue;
            if (p.res_v8) {
                rnext[i] = ptx::ld_nc_v8(res_row + c0 + 16 * i);
            } else {  // slices that are only 16-byte aligned
                const uint4 lo = ptx::ld_nc_v4(reinterpret_cast<const uint4*>(res_row + c0 + 16 * i));
                const uint4 hi = ptx::ld_nc_v4(reinterpret_cast<const uint4*>(res_row + c0 + 16 * i + 8));
                rnext[i].v[0] = lo.x; rnext[i].v[1] = lo.y; rnext[i].v[2] = lo.z; rnext[i].v[3] = lo.w;
                rnext[i].v[4] = hi.x; rnext[i].v[5] = hi.y; rnext[i].v[6] = hi.z; rnext[i].v[7] = hi.w;
            }
        }
    };
    fetch_res(c_begin);  // independent of the accumulator: in flight while the MMAs finish

    const long long ta0 = t_acc ? clock64() : 0;
    ptx::mbar_wait_addr(full_addr, aphase);
    if (t_acc) *t_acc += clock64() - ta0;
    ptx::tc_fence_after();
    long long tp = t_acc ? clock64() : 0;  // developer phase timers: t_acc[1] TMEM load, [2] math, [3] staging + stores
    auto lap = [&](int slot) {
        if (t_acc) { const long long now = clock64(); t_acc[slot] += now - tp; tp = now; }
    };

    // one 32-column chunk held in `acc` (its TMEM load already waited for)
    auto chunk = [&](const uint32_t (&acc)[32], int c0) {
        ptx::U32x8 rcur[2];
        rcur[0] = rnext[0];
        rcur[1] = rnext[1];
        if (c0 + 32 < c_end) fetch_res(c0 + 32);
        const float* bias = p.bias_c + n0 + c0;  // constant bank, warp-uniform index
        float2 x[16];
        if constexpr (MISH) {
#pragma unroll
            for (int g = 0; g < 16; ++g) x[g] = bias_mish2(acc[2 * g], acc[2 * g + 1], bias[2 * g], bias[2 * g + 1]);
        } else if (!generic_act) {
#pragma unroll
            for (int g = 0; g < 16; ++g) x[g] = bias_act2<false>(acc[2 * g], acc[2 * g + 1], bias[2 * g], bias[2 * g + 1], alpha2);
        } else {
#pragma unroll
            for (int g = 0; g < 16; ++g) x[g] = bias_act2<true>(acc[2 * g], acc[2 * g + 1], bias[2 * g], bias[2 * g + 1], alpha2);
        }
        if (mode == 1 && p.head_tma) {
            // head tensors: the lane's 32 fp32 columns (128 B) go into a 32-row staging tile (128-byte swizzle) and leave
            // through a TMA store.  Direct stores made every warp instruction touch 32 half-used sectors: the 52x52 head
            // spent 4x its MMA time storing.
            if (lane == 0) ptx::tma_store_wait_read<0>();  // the previous chunk's store has finished reading the tile
            __syncwarp();
#pragma unroll
            for (int c = 0; c < 8; ++c)
                *reinterpret_cast<float4*>(stage + lane * 128 + ((c ^ (lane & 7)) << 4)) =
                    make_float4(x[2 * c].x, x[2 * c].y, x[2 * c + 1].x, x[2 * c + 1].y);
            ptx::fence_proxy_async();
            __syncwarp();
            if (lane == 0) {
                ptx::tma_store_2d(tm_out, stage, n0 + c0, static_cast<int>(m_base));  // rows >= M, columns >= pitch are clipped
                ptx::tma_store_commit();
            }
            lap(3);
            return;
        }
        if (mode == 1) {
            // fallback: fp32 rows straight from the registers
            if (own_ok) {
                float* op = reinterpret_cast<float*>(p.out) + m_own * p.out_pitch + n0 + c0;
#pragma unroll
                for (int g = 0; g < 8; ++g)
                    if (n0 + c0 + 4 * g < p.n_store_limit)
                        *reinterpret_cast<float4*>(op + 4 * g) = make_float4(x[2 * g].x, x[2 * g].y, x[2 * g + 1].x, x[2 * g + 1].y);
            }
            lap(2);
            return;
        }
        if (has_res) {  // ONNX Add after LeakyRelu, in fp32 like the reference graph: ONE rounding, of the sum (rounding the branch value first
                        // and the bf16 sum again doubled the rounding noise of every residual layer)
#pragma unroll
            for (int g = 0; g < 16; ++g) {
                const uint32_t r = rcur[g >> 3].v[g & 7];
                x[g] = __fadd2_rn(x[g], make_float2(__uint_as_float(r << 16), __uint_as_float(r & 0xFFFF0000u)));
            }
        }
        uint32_t pk[16];
#pragma unroll
        for (int g = 0; g < 16; ++g) pk[g] = pack_bf16(x[g].x, x[g].y);
        lap(2);
        if (STRIP && !RES) {
            // The lane's rows are scattered over the image (pad positions in between), so no TMA box fits them: 64 bytes
            // per lane straight from the registers (measured faster than the staged form below when nothing else loads)
            if (own_ok) {
                __nv_bfloat16* op = reinterpret_cast<__nv_bfloat16*>(p.out) + m_own * p.out_pitch + n0 + c0;
#pragma unroll
                for (int c = 0; c < 4; ++c)
                    if (n0 + c0 + 8 * c < p.cout)
                        *reinterpret_cast<uint4*>(op + 8 * c) = make_uint4(pk[4 * c], pk[4 * c + 1], pk[4 * c + 2], pk[4 * c + 3]);
            }
            lap(3);
            return;
        }
        if (STRIP) {
            // With a residual the row-per-lane loads and stores (32 LSU wavefronts per instruction each) get in each
            // other's way: two chunks are staged as 32 rows x 128 B (128-byte swizzle), read back with 8 lanes per row, and
            // stored with every instruction covering 4 whole 128-byte lines.
            const bool second = ((c0 - c_begin) & 32) != 0;
#pragma unroll
            for (int c = 0; c < 4; ++c)
                *reinterpret_cast<uint4*>(stage + lane * 128 + (((c + (second ? 4 : 0)) ^ (lane & 7)) << 4)) =
                    make_uint4(pk[4 * c], pk[4 * c + 1], pk[4 * c + 2], pk[4 * c + 3]);
            if (second) {
                __syncwarp();
                const int sub = lane >> 3, ch = lane & 7;
                const int row32 = own_ok ? static_cast<int>(m_own) : -1;
                uint4 v[8];
                int mrow[8];
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                    const int r = 4 * i + sub;
                    v[i] = *reinterpret_cast<const uint4*>(stage + r * 128 + ((ch ^ (r & 7)) << 4));
                    mrow[i] = __shfl_sync(0xffffffffu, row32, r);
                }
                const int col = n0 + c0 - 32 + 8 * ch;
#pragma unroll
                for (int i = 0; i < 8; ++i)
                    if (mrow[i] >= 0 && col < p.cout)
                        *reinterpret_cast<uint4*>(reinterpret_cast<__nv_bfloat16*>(p.out) + static_cast<long long>(mrow[i]) * p.out_pitch + col) = v[i];
                __syncwarp();  // the staging tile is rewritten by the next pair of chunks
            }
            lap(3);
            return;
        }
        if (mode == 0 && HALF_N >= 64 && (FAST || p.store64)) {
            // two chunks share one staging tile of 32 rows x 128 B (128-byte swizzle: 16-byte chunk k of row r at slot
            // k ^ (r & 7)) and leave through ONE TMA store: half the store requests (the TMA engine moves about one
            // row per 3 cycles whatever its width) and half the proxy fences of the 64-byte form
            const bool second = ((c0 - c_begin) & 32) != 0;
            if (!second) {
                if (lane == 0) ptx::tma_store_wait_read<0>();  // the previous pair's store has finished reading the tile
                __syncwarp();
            }
#pragma unroll
            for (int c = 0; c < 4; ++c)
                *reinterpret_cast<uint4*>(stage + lane * 128 + (((c + (second ? 4 : 0)) ^ (lane & 7)) << 4)) =
                    make_uint4(pk[4 * c], pk[4 * c + 1], pk[4 * c + 2], pk[4 * c + 3]);
            if (second) {
                ptx::fence_proxy_async();  // generic-proxy writes -> visible to the TMA engine
                __syncwarp();
                if (lane == 0) {
                    ptx::tma_store_2d(tm_out, stage, n0 + c0 - 32, static_cast<int>(m_base));  // rows >= M are clipped by the map
                    ptx::tma_store_commit();
                }
            }
            lap(3);
            return;
        }
        // stage the bf16 row (64 B = 4 x 16 B) with the 64-byte swizzle (chunk c of row r at slot c ^ ((r >> 1) & 3)):
        // conflict-free for these stores, and the layout a SWIZZLE_64B tensor map reads back
        uint8_t* buf = stage + (sbuf & 1) * 2048;
        if (mode == 0) {
            // the TMA store that last read this buffer (two chunks ago) must have finished reading it
            if (lane == 0) ptx::tma_store_wait_read<1>();
            __syncwarp();
        }
#pragma unroll
        for (int c = 0; c < 4; ++c)
            *reinterpret_cast<uint4*>(buf + lane * 64 + ((c ^ ((lane >> 1) & 3)) << 4)) =
                make_uint4(pk[4 * c], pk[4 * c + 1], pk[4 * c + 2], pk[4 * c + 3]);
        if (mode == 0) {
            ptx::fence_proxy_async();  // generic-proxy writes -> visible to the TMA engine
            __syncwarp();
            if (lane == 0) {
                ptx::tma_store_2d(tm_out, buf, n0 + c0, static_cast<int>(m_base));  // rows >= M are clipped by the map
                ptx::tma_store_commit();
            }
            ++sbuf;
            lap(3);
            return;
        }
        // mode 2 (x2 upsampling): re-read transposed so that 4 lanes cover the 64 contiguous bytes of one pixel row
        __syncwarp();
        const int hw = p.ho * p.wo;
        const int sub = lane >> 2, j = lane & 3;
        const int ch = n0 + c0 + 8 * j;
        const long long w2p = 2LL * p.wo * p.out_pitch;
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const int r = 8 * i + sub;
            const long long m = m_base + r;
            const uint4 q = *reinterpret_cast<const uint4*>(buf + r * 64 + ((j ^ ((r >> 1) & 3)) << 4));
            if (m >= p.M || ch >= p.n_store_limit) continue;
            const int img = static_cast<int>(m / hw);
            const int rem = static_cast<int>(m - static_cast<long long>(img) * hw);
            const int oy = rem / p.wo;
            const int ox = rem - oy * p.wo;
            const long long orow = (static_cast<long long>(img) * 2 * p.ho + 2 * oy) * (2LL * p.wo) + 2 * ox;
            __nv_bfloat16* op = reinterpret_cast<__nv_bfloat16*>(p.out) + orow * p.out_pitch + ch;
            *reinterpret_cast<uint4*>(op) = q;  // the 2x2 nearest-neighbour block
            *reinterpret_cast<uint4*>(op + p.out_pitch) = q;
            *reinterpret_cast<uint4*>(op + w2p) = q;
            *reinterpret_cast<uint4*>(op + w2p + p.out_pitch) = q;
        }
        __syncwarp();  // staging tile is rewritten by the next chunk
        lap(3);
    };
    auto release_tmem = [&]() {  // all TMEM reads of this accumulator stage done: hand it back to the MMA warp
        ptx::tc_fence_before();
        __syncwarp();
        if (lane == 0) ptx::mbar_arrive_cluster_addr(empty_addr);
    };

    uint32_t acc_a[32], acc_b[32];
    if (!FIXED && p.split_k > 1) {
        // ---- split-K: this launch computed only part `part` of the tile's K range
        const int S = p.split_k;
        // partial regions: [tile][part][region = CTA rank * 4 + lane quarter][column / 4][32 lanes][4] fp32: a warp's
        // 16-byte accesses are 512 contiguous bytes (row-major rows made every access 32 separate lines: 20x slower)
        const size_t region_elems = static_cast<size_t>(32) * BLOCK_N;
        float* mine = p.ws + ((static_cast<size_t>(tile) * S + part) * 8 + region) * region_elems + lane * 4;
        for (int c0 = c_begin; c0 < c_end; c0 += 32) {
            ptx::tmem_ld_32x32(taddr0 + c0, acc_a);
            ptx::tmem_ld_wait();
            if (c0 + 32 >= c_end) release_tmem();
#pragma unroll
            for (int g = 0; g < 8; ++g)
                *reinterpret_cast<uint4*>(mine + (c0 / 4 + g) * 128) = make_uint4(acc_a[4 * g], acc_a[4 * g + 1], acc_a[4 * g + 2], acc_a[4 * g + 3]);
        }
        __threadfence();
        __syncwarp();
        int* counter = p.counters + (tile * 8 + region) * 2 + half;
        int old = 0;
        if (lane == 0) old = atomicAdd(counter, 1);
        old = __shfl_sync(0xffffffffu, old, 0);
        if (old != S - 1) return;  // another part's warp will find the counter full and finish this region
        __threadfence();
        fetch_res(c_begin);
        for (int c0 = c_begin; c0 < c_end; c0 += 32) {
            float sum[32];
#pragma unroll
            for (int e = 0; e < 32; ++e) sum[e] = 0.f;
            // parts are added in part order (the result does not depend on which part arrived last); the loads of up to
            // four parts x 16 columns are issued together so that their latencies overlap
            for (int sp0 = 0; sp0 < S; sp0 += 4) {
#pragma unroll
                for (int hcol = 0; hcol < 2; ++hcol) {
                    float4 v[4][4];
#pragma unroll
                    for (int k = 0; k < 4; ++k) {
                        const float* src = p.ws + ((static_cast<size_t>(tile) * S + sp0 + k) * 8 + region) * region_elems + lane * 4 + (c0 / 4 + 4 * hcol) * 128;
#pragma unroll
                        for (int g = 0; g < 4; ++g) v[k][g] = (sp0 + k < S) ? ptx::ld_cg_f4(src + g * 128) : make_float4(0.f, 0.f, 0.f, 0.f);
                    }
#pragma unroll
                    for (int k = 0; k < 4; ++k) {
                        if (sp0 + k >= S) break;
#pragma unroll
                        for (int g = 0; g < 4; ++g) {
                            float* d4 = sum + 16 * hcol + 4 * g;
                            d4[0] += v[k][g].x; d4[1] += v[k][g].y; d4[2] += v[k][g].z; d4[3] += v[k][g].w;
                        }
                    }
                }
            }
#pragma unroll
            for (int e = 0; e < 32; ++e) acc_a[e] = __float_as_uint(sum[e]);
            chunk(acc_a, c0);
        }
        if (lane == 0) *counter = 0;  // ready for the next launch that uses this workspace
        return;
    }
    ptx::tmem_ld_32x32(taddr0 + c_begin, acc_a);
#pragma unroll 1
    for (int c0 = c_begin; c0 < c_end; c0 += 64) {
        ptx::tmem_ld_wait();
        if (HALF_N > 32) ptx::tmem_ld_32x32(taddr0 + c0 + 32, acc_b);  // in flight during chunk c0
        else release_tmem();
        lap(1);
        if (!(kDev && (p.debug & 1))) chunk(acc_a, c0);
        if (HALF_N > 32) {
            ptx::tmem_ld_wait();
            if (c0 + 64 < c_end) ptx::tmem_ld_32x32(taddr0 + c0 + 64, acc_a);
            else release_tmem();
            lap(1);
            if (!(kDev && (p.debug & 1))) chunk(acc_b, c0 + 32);
        }
    }
}

// Swapped mode (narrow layers, Cout <= 128): the accumulator holds channels on the TMEM lanes and 256 output pixels on
// the columns (a tcgen05.mma costs ~150 cycles at M = 128 whatever its N, so N must be 256 to use the whole array and
// a narrow Cout cannot be N).  Lane = channel: bias is a per-lane scalar; a 32-pixel column chunk is staged to shared
// memory transposed ([pixel][32 channels] bf16) and re-read so that 4 lanes cover the 64 contiguous bytes this warp
// owns of one pixel row.
// PLAIN: compile-time copy for the production case (bf16 slice through TMA stores, no residual, max(x, alpha x)).
// MISH: Mish instead of max(x, alpha x) / the select form, in both copies.
template <bool PLAIN = false, bool MISH = false>
__device__ __forceinline__ void epilogue_tile_swapped(const ConvParams& p, const CUtensorMap* tm_out, int& sbuf, uint32_t taddr0,
                                                      float* stage_buf, int ch_warp, long long pix0, int lane, int half,
                                                      uint32_t full_addr, uint32_t aphase, uint32_t empty_addr, long long* t_acc) {
    const int hw = p.ho * p.wo;
    const int sub = lane >> 2, j = lane & 3;
    const bool warp_has_channels = ch_warp < p.cout;
    const int ch_own = ch_warp + lane;                      // row-major phase: this lane's channel
    const float bias_own = (ch_own < p.cout) ? __ldg(p.bias + ch_own) : 0.f;
    const int ch = ch_warp + 8 * j;                         // transposed phase: this lane's 8 channels
    const bool has_res = !PLAIN && p.residual != nullptr;
    const bool generic_act = !PLAIN && p.act == 2;
    const float alpha_eff = p.act ? p.alpha : 1.0f;
    const float2 alpha2 = make_float2(alpha_eff, alpha_eff);
    const bool tma_path = PLAIN || (p.epi_mode == 0 && !has_res && p.swap_tma);  // plain bf16 slice: staged rows leave through TMA stores

    const long long ta0 = t_acc ? clock64() : 0;
    ptx::mbar_wait_addr(full_addr, aphase);
    if (t_acc) *t_acc += clock64() - ta0;
    ptx::tc_fence_after();
    long long tp = t_acc ? clock64() : 0;
    auto lap = [&](int slot) {
        if (t_acc) { const long long now = clock64(); t_acc[slot] += now - tp; tp = now; }
    };

    const int c_end = half * 128 + 128;  // the two warps of a lane quarter take 128 of the tile's 256 pixels each
#pragma unroll 1
    for (int c0 = half * 128; c0 < c_end; c0 += 32) {
        uint32_t acc[32];
        if (warp_has_channels) ptx::tmem_ld_32x32(taddr0 + c0, acc);
        // pixels of this chunk handled by this lane in the transposed phase, and their residual values
        long long orow[4];
        bool ok[4];
        uint4 res[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            if (PLAIN || tma_path) { ok[i] = false; orow[i] = 0; res[i] = make_uint4(0u, 0u, 0u, 0u); continue; }
            const long long m = pix0 + c0 + 8 * i + sub;
            ok[i] = warp_has_channels && m < p.M && ch < p.cout;
            orow[i] = m;
            res[i] = make_uint4(0u, 0u, 0u, 0u);
            if (has_res && ok[i]) res[i] = __ldg(reinterpret_cast<const uint4*>(p.residual + m * p.res_pitch + ch));
            if (p.upsample2x && ok[i]) {
                const int img = static_cast<int>(m / hw);
                const int rem = static_cast<int>(m - static_cast<long long>(img) * hw);
                const int oy = rem / p.wo;
                const int ox = rem - oy * p.wo;
                orow[i] = (static_cast<long long>(img) * 2 * p.ho + 2 * oy) * (2LL * p.wo) + 2 * ox;
            }
        }
        if (warp_has_channels) ptx::tmem_ld_wait();
        if (c0 + 32 >= c_end) {
            ptx::tc_fence_before();
            __syncwarp();
            if (lane == 0) ptx::mbar_arrive_cluster_addr(empty_addr);
        }
        lap(1);
        if (!warp_has_channels || (kDev && (p.debug & 1))) continue;
        if (tma_path) {
            // lane = channel: element (pixel q, channel lane) goes to row q of a 32-pixel x 64-byte bf16 tile (64-byte
            // swizzle: 16-byte chunk (lane >> 3) of row q sits at slot (lane >> 3) ^ ((q >> 1) & 3)) that one TMA store
            // writes out — no shared-memory loads, no per-thread global stores
            uint8_t* buf = reinterpret_cast<uint8_t*>(stage_buf) + (sbuf & 1) * 2048;
            if (lane == 0) ptx::tma_store_wait_read<1>();  // the store that last read this buffer (two chunks ago) is done with it
            __syncwarp();
            const uint32_t lane_chunk = static_cast<uint32_t>(lane) >> 3, lane_byte = (static_cast<uint32_t>(lane) & 7u) * 2u;
#pragma unroll
            for (int q = 0; q < 32; q += 2) {
                float2 x;
                if constexpr (MISH) x = bias_mish2(acc[q], acc[q + 1], bias_own, bias_own);
                else x = generic_act ? bias_act2<true>(acc[q], acc[q + 1], bias_own, bias_own, alpha2)
                                     : bias_act2<false>(acc[q], acc[q + 1], bias_own, bias_own, alpha2);
                const uint32_t slot = (lane_chunk ^ ((static_cast<uint32_t>(q) >> 1) & 3u)) << 4;  // rows q and q+1 share (q >> 1)
                *reinterpret_cast<__nv_bfloat16*>(buf + q * 64 + slot + lane_byte) = __float2bfloat16(x.x);
                *reinterpret_cast<__nv_bfloat16*>(buf + (q + 1) * 64 + slot + lane_byte) = __float2bfloat16(x.y);
            }
            ptx::fence_proxy_async();
            __syncwarp();
            if (lane == 0) {
                ptx::tma_store_2d(tm_out, buf, ch_warp, static_cast<int>(pix0 + c0));  // pixels >= M / channels >= Cout are clipped
                ptx::tma_store_commit();
            }
            ++sbuf;
            lap(3);
            continue;
        }
        if (PLAIN) continue;
        // channel-major phase: + bias, LeakyReLU; element (pixel q, channel lane) -> stage_buf[q][lane] (fp32: one
        // conflict-free 128-byte row per store instruction)
        if constexpr (MISH) {
#pragma unroll
            for (int q = 0; q < 32; q += 2) {
                const float2 x = bias_mish2(acc[q], acc[q + 1], bias_own, bias_own);
                stage_buf[q * 32 + lane] = x.x;
                stage_buf[(q + 1) * 32 + lane] = x.y;
            }
        } else if (!generic_act) {
#pragma unroll
            for (int q = 0; q < 32; q += 2) {
                const float2 x = bias_act2<false>(acc[q], acc[q + 1], bias_own, bias_own, alpha2);
                stage_buf[q * 32 + lane] = x.x;
                stage_buf[(q + 1) * 32 + lane] = x.y;
            }
        } else {
#pragma unroll
            for (int q = 0; q < 32; q += 2) {
                const float2 x = bias_act2<true>(acc[q], acc[q + 1], bias_own, bias_own, alpha2);
                stage_buf[q * 32 + lane] = x.x;
                stage_buf[(q + 1) * 32 + lane] = x.y;
            }
        }
        __syncwarp();
        lap(2);
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const int q = 8 * i + sub;
            float4 lo = *reinterpret_cast<const float4*>(stage_buf + q * 32 + 8 * j);
            float4 hi = *reinterpret_cast<const float4*>(stage_buf + q * 32 + 8 * j + 4);
            if (has_res) {  // same arithmetic as the normal mode: fp32 sum, rounded once
                const uint4 rr = res[i];
                lo.x += __uint_as_float(rr.x << 16); lo.y += __uint_as_float(rr.x & 0xFFFF0000u);
                lo.z += __uint_as_float(rr.y << 16); lo.w += __uint_as_float(rr.y & 0xFFFF0000u);
                hi.x += __uint_as_float(rr.z << 16); hi.y += __uint_as_float(rr.z & 0xFFFF0000u);
                hi.z += __uint_as_float(rr.w << 16); hi.w += __uint_as_float(rr.w & 0xFFFF0000u);
            }
            const uint4 v = make_uint4(pack_bf16(lo.x, lo.y), pack_bf16(lo.z, lo.w), pack_bf16(hi.x, hi.y), pack_bf16(hi.z, hi.w));
            if (!ok[i]) continue;
            __nv_bfloat16* op = reinterpret_cast<__nv_bfloat16*>(p.out) + orow[i] * p.out_pitch + ch;
            *reinterpret_cast<uint4*>(op) = v;
            if (p.upsample2x) {
                const long long w2p = 2LL * p.wo * p.out_pitch;
                *reinterpret_cast<uint4*>(op + p.out_pitch) = v;
                *reinterpret_cast<uint4*>(op + w2p) = v;
                *reinterpret_cast<uint4*>(op + w2p + p.out_pitch) = v;
            }
        }
        __syncwarp();
        lap(3);
    }
}

template <int KS, bool TWO>
__device__ __forceinline__ void issue_mmas(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, bool acc0) {
#pragma unroll
    for (int k = 0; k < KS; ++k) {
        if (TWO) ptx::umma2_bf16(tmem_d, adesc + 2 * k, bdesc + 2 * k, idesc, (acc0 || k > 0) ? 1u : 0u);
        else ptx::umma_bf16(tmem_d, adesc + 2 * k, bdesc + 2 * k, idesc, (acc0 || k > 0) ? 1u : 0u);
    }
}

// TWO = false: one CTA per 128 x BLOCK_N tile (tcgen05 cta_group::1).
// TWO = true : a cluster of two CTAs (one TPC) per 256 x 256 tile (cta_group::2): CTA r owns output rows
//              [128r, 128r+128) and stages B rows [128r, 128r+128); the leader (rank 0) issues the MMAs, which
//              read both CTAs' shared memory.  Per SM and K block this needs 16 KB of A + 16 KB of B instead of
//              16 + 32 KB, which is what the L2->SM fill latency x shared-memory capacity product can sustain.
// MISH: every epilogue copy applies Mish (ConvParams::act 3); a separate instantiation, so the LeakyReLU kernels are unchanged.
template <int BLOCK_N, bool TWO, bool SWAP = false, bool STRIP = false, bool MISH = false>
__global__ void __launch_bounds__(NUM_THREADS, 1)
conv_tc_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
               const __grid_constant__ CUtensorMap tmOut, const __grid_constant__ ConvParams p) {
    using Cfg = TileCfg<BLOCK_N>;
    static_assert(!TWO || BLOCK_N == 256, "the CTA-pair kernel is built for 256-wide tiles");
    static_assert(!SWAP || (BLOCK_N == 256 && !TWO), "the swapped mode is a single-CTA 128 x 256 kernel");
    constexpr int B_ROWS = TWO ? BLOCK_N / 2 : BLOCK_N;  // B rows this CTA stages per K block
    const int STAGES = p.num_stages;

    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem);
    uint64_t* empty_bar = full_bar + MAX_STAGES;
    uint64_t* tmem_full_bar = empty_bar + MAX_STAGES;
    uint64_t* tmem_empty_bar = tmem_full_bar + 2;
    uint64_t* bres_bar = tmem_empty_bar + 2;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bres_bar + 1);
    // "B resident": when the whole filter bank of the (single) N tile fits, it is loaded into shared memory once per
    // CTA and the ring carries only A — narrow layers are bound by the TMA issue rate, and this halves it.
    const bool b_res = !TWO && p.b_resident != 0;
    // swapped mode: slot 0 (the MMA's M side, 128 rows) holds filter rows, slot 1 (N side, 256 rows) holds pixels
    constexpr bool swap = SWAP;
    static_assert(!STRIP || (TWO && BLOCK_N == 256 && !SWAP), "strip mode belongs to the CTA-pair kernel");
    constexpr bool strip = STRIP;  // A comes from per-channel-block strips (see ConvParams::strip), the ring carries B only
    uint64_t* strip_full_bar = reinterpret_cast<uint64_t*>(smem + 640);
    uint64_t* strip_empty_bar = strip_full_bar + 2;
    const uint32_t a_bytes = strip ? 0u : BLOCK_M * p.block_k * 2;
    const uint32_t b_bytes = B_ROWS * p.block_k * 2;
    uint8_t* bres = smem + SMEM_RING_OFF;
    uint8_t* ring = bres + (b_res ? b_bytes * p.num_k_blocks : 0u);
    const uint32_t sub_bytes = a_bytes + (b_res ? 0u : b_bytes);  // one K block: A then B, both multiples of 1024
    const int kps = p.kb_per_stage;                   // K blocks sharing one ring stage / one barrier round
    const uint32_t stage_bytes = sub_bytes * kps;

    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    const int num_tiles = (kDev && (p.debug & 32)) ? 0 : p.num_m_tiles * p.num_n_tiles;  // TWO: m tiles are 256 rows
    // work items: (tile, part) with the tile's K blocks cut into split_k parts (1 = whole tiles); every role walks
    // items unit, unit + units, ... and derives the same K-block range [kb_lo, kb_hi) for each
    const int split_k = p.split_k;
    const uint32_t cta_rank = TWO ? ptx::cluster_ctarank() : 0u;    // rank inside the pair
    const int unit = TWO ? (blockIdx.x >> 1) : blockIdx.x;            // tile-stream index of this CTA / pair
    const int units = TWO ? (gridDim.x >> 1) : gridDim.x;
    const int num_items = num_tiles * split_k;
    auto tile_of = [&](int item) { return item / split_k; };

    if (warp == 0 && lane == 0) {
        ptx::tma_prefetch_desc(&tmA);
        ptx::tma_prefetch_desc(&tmB);
    }
    if (warp == 4 && lane == 0 && (p.epi_mode == 0 || p.head_tma)) ptx::tma_prefetch_desc(&tmOut);  // (a valid map in every mode)
    if (warp == 1 && lane == 0) {
        for (int i = 0; i < STAGES; ++i) {
            ptx::mbar_init(&full_bar[i], 1);
            ptx::mbar_init(&empty_bar[i], 1);
        }
        for (int i = 0; i < 2; ++i) {
            ptx::mbar_init(&tmem_full_bar[i], 1);
            ptx::mbar_init(&tmem_empty_bar[i], TWO ? 16 : (BLOCK_N < 64 ? 4 : 8));  // one arrive per epilogue warp (of both CTAs) draining the stage
        }
        ptx::mbar_init(bres_bar, 1);
        for (int i = 0; i < 2; ++i) {
            ptx::mbar_init(&strip_full_bar[i], 1);
            ptx::mbar_init(&strip_empty_bar[i], 1);
        }
        ptx::fence_barrier_init();
    }
    if (warp == 2) {
        if (TWO) { ptx::tmem_alloc2(tmem_slot, Cfg::TMEM_COLS); ptx::tmem_relinquish2(); }
        else { ptx::tmem_alloc(tmem_slot, Cfg::TMEM_COLS); ptx::tmem_relinquish(); }
    }
    ptx::tc_fence_before();
    if (TWO) ptx::cluster_sync(); else __syncthreads();
    ptx::tc_fence_after();
    const uint32_t tmem_base_v = *tmem_slot;
    // Programmatic dependent launch: the next layer's CTAs may be scheduled from here on (they take an SM as soon as
    // this kernel's CTA leaves it and run their own set-up above while the rest of this grid finishes).  Warps that
    // touch activations call grid_dep_wait() first: the previous layer is complete and visible after it.
    ptx::grid_dep_launch();

    // Everything the single-thread producer / MMA loops need is copied into registers first: the inline-asm
    // "memory" clobbers would otherwise make the compiler re-read every p.* field from the constant bank on each
    // k-block, and integer divisions per k-block put ~700 dependent cycles in the producer's way (measured).
    const uint32_t bar_base_v = ptx::smem_u32(full_bar);       // full[i] at +8i, empty[i] at +8(MAX_STAGES+i)
    const uint32_t ring_base_v = ptx::smem_u32(ring);
    const uint32_t tmem_full_addr_v = ptx::smem_u32(tmem_full_bar), tmem_empty_addr_v = ptx::smem_u32(tmem_empty_bar);
    const int nkb = p.num_k_blocks, cin_blocks = p.cin_blocks, ksize = p.ksize, block_k = p.block_k;
    const int n_tiles_n = p.num_n_tiles;
    const bool prof = kDev && p.prof != nullptr;
    constexpr int TILE_M = TWO ? 2 * BLOCK_M : BLOCK_M;
    const uint32_t strip_stride = (static_cast<uint32_t>(p.strip_rows) * 128u + 1023u) & ~1023u;
    const uint32_t strips_base_v = ring_base_v + static_cast<uint32_t>(STAGES) * stage_bytes;  // two strip buffers behind the ring
    const uint32_t strip_bar_v = ptx::smem_u32(strip_full_bar);  // full[i] at +8i, empty[i] at +16+8i

    if (warp == 0) {
        // ------------------------------------------------------------------ TMA producer (both CTAs of a pair)
        // The whole warp walks the loop (warp-uniform control flow keeps addresses and coordinates in uniform
        // registers); one elected lane issues.
        const bool issuer = ptx::elect_one();
        const uint32_t ring_base = __shfl_sync(0xffffffffu, ring_base_v, 0);  // warp-uniform for the compiler (see the MMA warp)
        const uint32_t bar_base = __shfl_sync(0xffffffffu, bar_base_v, 0);
        const bool im2col = p.a_im2col != 0, load_a = !(kDev && (p.debug & 2));
        const int ho_wo = p.ho * p.wo, wo = p.wo, cstride = p.stride, pad = p.pad_lo;
        const uint32_t tx_bytes = ((load_a ? a_bytes : 0u) + (b_res ? 0u : b_bytes)) * (TWO ? 2u : 1u);
        const uint64_t mapA = reinterpret_cast<uint64_t>(&tmA), mapB = reinterpret_cast<uint64_t>(&tmB);
        int stage = 0;
        uint32_t phase = 0;
        long long t_wait = 0;
        if (b_res && issuer && unit < num_items) {
            const uint32_t bar = ptx::smem_u32(bres_bar);
            ptx::mbar_arrive_expect_tx_addr(bar, b_bytes * nkb);
            for (int kb = 0; kb < nkb; ++kb)
                ptx::tma_load_2d_addr(ptx::smem_u32(bres) + kb * b_bytes, mapB, bar, kb * block_k, 0);
        }
        // weights above are constants; everything below reads the previous layer's output: its whole grid has to be complete
        ptx::grid_dep_wait();
        const long long t_start = prof ? clock64() : 0;
        int sidx = 0;  // strips loaded so far (strip mode)
        const uint32_t strips_base = __shfl_sync(0xffffffffu, strips_base_v, 0), strip_bar = __shfl_sync(0xffffffffu, strip_bar_v, 0);
        for (int item = unit; item < num_items && !(kDev && (p.debug & 8)); item += units) {
            const int tile = tile_of(item), part = item - tile * split_k;
            const int kb_lo = (part * nkb) / split_k, kb_hi = ((part + 1) * nkb) / split_k;
            const int m_tile = tile / n_tiles_n;
            if (strip) {
                const int n0s = (tile - m_tile * n_tiles_n) * BLOCK_N + static_cast<int>(cta_rank) * B_ROWS;
                const int wp = p.strip_wp, plane = p.strip_wp * p.strip_hp;
                const int qs = p.strip_qfirst + m_tile * TILE_M + static_cast<int>(cta_rank) * BLOCK_M - wp - 1;  // first strip position
                const int simg = qs / plane, srem = qs - simg * plane, syp = srem / wp, sxp = srem - syp * wp;
                for (int cbi = 0; cbi < cin_blocks; ++cbi, ++sidx) {
                    const int sb = sidx & 1;
                    const uint32_t sfull = strip_bar + 8u * sb;
                    ptx::mbar_wait_addr(sfull + 16u, ((sidx >> 1) & 1) ^ 1);  // the MMAs of two strips ago have retired
                    if (issuer && cta_rank == 0) ptx::mbar_arrive_expect_tx_addr(sfull, static_cast<uint32_t>(p.strip_rows) * 128u * 2u);
                    if (issuer)
                        ptx::tma2_load_im2col_4d_addr(strips_base + sb * strip_stride, mapA, sfull & ptx::kPeerBitMask, cbi * block_k, sxp - 1,
                                                      syp - 1, simg, 0, 0);
                    for (int tap = 0; tap < 9; ++tap) {
                        const uint32_t full_addr = bar_base + 8u * stage;
                        ptx::mbar_wait_addr(full_addr + 8u * MAX_STAGES, phase ^ 1);
                        if (issuer && cta_rank == 0) ptx::mbar_arrive_expect_tx_addr(full_addr, b_bytes * 2u);
                        if (issuer)
                            ptx::tma2_load_2d_addr(ring_base + stage * stage_bytes, mapB, full_addr & ptx::kPeerBitMask,
                                                   (tap * cin_blocks + cbi) * block_k, n0s);
                        if (++stage == STAGES) { stage = 0; phase ^= 1; }
                    }
                }
                continue;
            }
            // normal: m0 = first output pixel (M side), n0 = first output channel (N side)
            // swapped: m0 = first output pixel (N side, 256 per tile), n0 = first output channel (M side, 128 per tile)
            const int n0 = swap ? (tile - m_tile * n_tiles_n) * BLOCK_M
                                : (tile - m_tile * n_tiles_n) * BLOCK_N + static_cast<int>(cta_rank) * B_ROWS * (TWO ? 1 : 0);
            const int m0 = swap ? m_tile * 256 : m_tile * TILE_M + static_cast<int>(cta_rank) * BLOCK_M;
            int img = 0, base_w = 0, base_h = 0;
            if (im2col) {
                img = m0 / ho_wo;
                const int rem = m0 - img * ho_wo;
                const int oy = rem / wo;
                base_w = (rem - oy * wo) * cstride - pad;
                base_h = oy * cstride - pad;
            }
            const int tap0 = kb_lo / cin_blocks;
            int cb = kb_lo - tap0 * cin_blocks, tap_r = tap0 / ksize, tap_s = tap0 - (tap0 / ksize) * ksize, kcoord = kb_lo * block_k;
            for (int kb = kb_lo; kb < kb_hi; kb += kps) {
                const int nsub = (kb_hi - kb < kps) ? kb_hi - kb : kps;
                const uint32_t full_addr = bar_base + 8u * stage;
                const uint32_t lead_bar = TWO ? (full_addr & ptx::kPeerBitMask) : full_addr;
                const long long tw0 = prof ? clock64() : 0;
                ptx::mbar_wait_addr(full_addr + 8u * MAX_STAGES, phase ^ 1);
                if (prof) t_wait += clock64() - tw0;
                // transaction bytes of both CTAs of a pair land on the leader's barrier; only the leader arms it
                if (issuer && cta_rank == 0) ptx::mbar_arrive_expect_tx_addr(full_addr, tx_bytes * nsub);
                for (int sb = 0; sb < nsub; ++sb) {
                    const uint32_t dst = ring_base + stage * stage_bytes + sb * sub_bytes;
                    if (!issuer) {
                    } else if (TWO) {
                        if (load_a) {
                            if (im2col)
                                ptx::tma2_load_im2col_4d_addr(dst, mapA, lead_bar, cb * block_k, base_w, base_h, img,
                                                              static_cast<uint16_t>(tap_s), static_cast<uint16_t>(tap_r));
                            else
                                ptx::tma2_load_2d_addr(dst, mapA, lead_bar, cb * block_k, m0);
                        }
                        ptx::tma2_load_2d_addr(dst + a_bytes, mapB, lead_bar, kcoord, n0);
                    } else {
                        // pixels go to the slot of the side they occupy in the MMA (slot 0 = M side, slot 1 = N side)
                        const uint32_t dst_x = swap ? dst + a_bytes : dst, dst_w = swap ? dst : dst + a_bytes;
                        if (load_a) {
                            if (im2col)
                                ptx::tma_load_im2col_4d_addr(dst_x, mapA, full_addr, cb * block_k, base_w, base_h, img,
                                                             static_cast<uint16_t>(tap_s), static_cast<uint16_t>(tap_r));
                            else
                                ptx::tma_load_2d_addr(dst_x, mapA, full_addr, cb * block_k, m0);
                        }
                        if (!b_res) ptx::tma_load_2d_addr(dst_w, mapB, full_addr, kcoord, n0);
                    }
                    kcoord += block_k;
                    if (++cb == cin_blocks) {
                        cb = 0;
                        if (++tap_s == ksize) { tap_s = 0; ++tap_r; }
                    }
                }
                if (++stage == STAGES) { stage = 0; phase ^= 1; }
            }
        }
        if (prof && lane == 0) { p.prof[blockIdx.x * 16 + 0] = clock64() - t_start; p.prof[blockIdx.x * 16 + 1] = t_wait; }
    } else if (warp == 1 && cta_rank == 0) {
        // ------------------------------------------------------------------ MMA issuer (leader CTA only)
        const uint32_t idesc = ptx::make_idesc_bf16_f32(TILE_M, BLOCK_N);
        // swizzle span = one K block: 128 B (block_k 64), 64 B (32) or 32 B (16)
        const uint32_t layout = (block_k == 64) ? 2u : (block_k == 32 ? 4u : 6u);
        const uint32_t sbo = 16u * block_k;  // 8 rows x swizzle span
        const int k_steps = (kDev && (p.debug & 4)) ? 0 : block_k / 16;
        // shared-memory / TMEM base addresses are the same in every lane, but the compiler cannot see that (they come
        // from a cvta and a shared-memory load): a broadcast shuffle marks them warp-uniform
        const uint32_t ring_base = __shfl_sync(0xffffffffu, ring_base_v, 0);
        const uint32_t bar_base = __shfl_sync(0xffffffffu, bar_base_v, 0);
        const uint32_t tmem_base = __shfl_sync(0xffffffffu, tmem_base_v, 0);
        const uint32_t tmem_full_addr = __shfl_sync(0xffffffffu, tmem_full_addr_v, 0);
        const uint32_t tmem_empty_addr = __shfl_sync(0xffffffffu, tmem_empty_addr_v, 0);
        const uint64_t desc0 = ptx::make_kmajor_desc(ring_base, sbo, layout);  // stage 0, A operand
        const uint32_t stage_units = stage_bytes >> 4, sub_units = sub_bytes >> 4, a_units = a_bytes >> 4;
        const bool issuer = ptx::elect_one();
        const uint64_t bres_desc0 = ptx::make_kmajor_desc(__shfl_sync(0xffffffffu, ptx::smem_u32(bres), 0), sbo, layout);
        const uint32_t b_units = b_bytes >> 4;
        if (b_res && unit < num_items) {
            ptx::mbar_wait(bres_bar, 0);
            ptx::tc_fence_after();
        }
        long long t_full = 0, t_tmem = 0, t_start = prof ? clock64() : 0;
        const bool skip_full_wait = kDev && (p.debug & 8) != 0;  // developer: MMA-only run (operands = whatever is in smem)
        // The loop is walked by the whole warp with every address / descriptor a warp-uniform value computed OUTSIDE the
        // elected lane's branch: that keeps them in uniform registers, so a tcgen05.mma costs one UIADD3.64 per operand
        // instead of a chain of R2UR moves (the narrow layers are bound by this warp's issue rate: ~150 cycles per MMA
        // before, against 48 the tensor core needs at N = 64 — dev/mma_rate.cu).
        auto run = [&](auto ks_tag) {
            constexpr int KS = decltype(ks_tag)::value;  // MMAs (16-wide K steps) per K block
            int stage = 0, it = 0, sidx = 0;
            uint32_t phase = 0, stage_off = 0;
            const uint32_t strip_bar = __shfl_sync(0xffffffffu, strip_bar_v, 0);
            const uint64_t strip_desc0 = ptx::make_kmajor_desc(__shfl_sync(0xffffffffu, strips_base_v, 0), 1024u, 2u);
            const uint32_t strip_units = strip_stride >> 4, wp_units = static_cast<uint32_t>(p.strip_wp) * 8u;  // 128-byte rows in 16-byte units
            for (int item = unit; item < num_items; item += units, ++it) {
                const int part = item % split_k;
                const int kb_lo = (part * nkb) / split_k, kb_hi = ((part + 1) * nkb) / split_k;
                const int as = it & 1;
                const uint32_t aphase = (it >> 1) & 1;
                const long long tq0 = prof ? clock64() : 0;
                ptx::mbar_wait_addr(tmem_empty_addr + 8u * as, aphase ^ 1);
                if (prof) t_tmem += clock64() - tq0;
                ptx::tc_fence_after();
                const uint32_t tmem_d = tmem_base + as * BLOCK_N;
                uint32_t accumulate = 0, bres_off = kb_lo * b_units;
                if (strip) {
                    for (int cbi = 0; cbi < cin_blocks; ++cbi, ++sidx) {
                        const int sb = sidx & 1;
                        const long long ts0 = prof ? clock64() : 0;
                        ptx::mbar_wait_addr(strip_bar + 8u * sb, (sidx >> 1) & 1);
                        if (prof) t_full += clock64() - ts0;
                        const uint64_t sdesc = strip_desc0 + sb * strip_units;
                        uint32_t tap_off = 0;
                        for (int ky = 0; ky < 3; ++ky, tap_off += wp_units) {
                            for (int kx = 0; kx < 3; ++kx) {
                                const uint32_t full_addr = bar_base + 8u * stage;
                                const long long tf0 = prof ? clock64() : 0;
                                ptx::mbar_wait_addr(full_addr, phase);
                                if (prof) t_full += clock64() - tf0;
                                ptx::tc_fence_after();
                                if (issuer) {
                                    issue_mmas<KS, TWO>(tmem_d, sdesc + tap_off + 8u * kx, desc0 + stage_off, idesc, accumulate != 0);
                                    ptx::umma2_commit_mcast_addr(full_addr + 8u * MAX_STAGES, 3);
                                }
                                accumulate = 1;
                                __syncwarp();
                                stage_off += stage_units;
                                if (++stage == STAGES) { stage = 0; stage_off = 0; phase ^= 1; }
                            }
                        }
                        if (issuer) ptx::umma2_commit_mcast_addr(strip_bar + 16u + 8u * sb, 3);  // strip buffer free in both CTAs
                        __syncwarp();
                    }
                    if (issuer) ptx::umma2_commit_mcast_addr(tmem_full_addr + 8u * as, 3);
                    __syncwarp();
                    continue;
                }
                for (int kb = kb_lo; kb < kb_hi; kb += kps) {
                    const int nsub = (kb_hi - kb < kps) ? kb_hi - kb : kps;
                    const uint32_t full_addr = bar_base + 8u * stage;
                    const long long tf0 = prof ? clock64() : 0;
                    if (!skip_full_wait) ptx::mbar_wait_addr(full_addr, phase);
                    if (prof) t_full += clock64() - tf0;
                    ptx::tc_fence_after();
                    uint64_t adesc = desc0 + stage_off;
                    for (int sb = 0; sb < nsub; ++sb) {
                        const uint64_t bdesc = b_res ? bres_desc0 + bres_off : adesc + a_units;
                        // 16 elements (32 B) along K inside the swizzle span per MMA: +2 in 16-byte units
                        if (issuer) issue_mmas<KS, TWO>(tmem_d, adesc, bdesc, idesc, accumulate != 0);
                        accumulate = 1;
                        adesc += sub_units;
                        bres_off += b_units;
                    }
                    if (issuer) {  // smem slot free (in both CTAs) once these MMAs retire
                        if (TWO) ptx::umma2_commit_mcast_addr(full_addr + 8u * MAX_STAGES, 3);
                        else ptx::umma_commit_addr(full_addr + 8u * MAX_STAGES);
                    }
                    __syncwarp();
                    stage_off += stage_units;
                    if (++stage == STAGES) { stage = 0; stage_off = 0; phase ^= 1; }
                }
                // accumulator complete (each CTA of a pair drains its own 128 rows)
                if (issuer) {
                    if (TWO) ptx::umma2_commit_mcast_addr(tmem_full_addr + 8u * as, 3);
                    else ptx::umma_commit_addr(tmem_full_addr + 8u * as);
                }
                __syncwarp();
            }
        };
        if (k_steps == 4) run(std::integral_constant<int, 4>{});
        else if (k_steps == 2) run(std::integral_constant<int, 2>{});
        else if (k_steps == 1) run(std::integral_constant<int, 1>{});
        else run(std::integral_constant<int, 0>{});
        if (prof && lane == 0) { p.prof[blockIdx.x * 16 + 2] = clock64() - t_start; p.prof[blockIdx.x * 16 + 3] = t_full; p.prof[blockIdx.x * 16 + 4] = t_tmem; }
    } else if (warp >= 4) {
        // ------------------------------------------------------------------ epilogue
        const int half = (warp - 4) >> 2;   // which half of the tile's columns this warp drains
        const int quarter = warp & 3;       // TMEM lanes [32*quarter, 32*quarter + 32)
        uint8_t* stage = smem + SMEM_STAGING_OFF + (warp - 4) * 4096;  // two 2 KB chunk buffers (swapped mode: one 4 KB)
        const uint32_t tmem_full_addr = tmem_full_addr_v, tmem_empty_addr = tmem_empty_addr_v;
        const uint32_t tlane = tmem_base_v + (static_cast<uint32_t>(quarter * 32) << 16);
        // the MMA issuer that waits for "accumulator drained" lives in the leader CTA
        const uint32_t empty_mask = TWO ? ptx::kPeerBitMask : 0xFFFFFFFFu;
        int it = 0;
        int sbuf = 0;
        // the production configuration takes the copy of the epilogue that has its flags compiled in
        const bool fast_epi = !STRIP && !swap && p.epi_mode == 0 && p.store64 && p.split_k == 1 && p.act != 2 && !(kDev && p.debug);
        // residual reads / output writes must not overtake the previous layer
        ptx::grid_dep_wait();
        long long t_acc[8] = {0, 0, 0, 0, 0, 0, 0, 0}, t_start = prof ? clock64() : 0;
        for (int item = unit; item < num_items; item += units, ++it) {
            const int tile = tile_of(item), part = item - tile * split_k;
            const int as = it & 1;  // accumulator stage
            if (BLOCK_N < 64 && as != half) continue;  // one-chunk tiles: the two warps of a lane quarter alternate tiles
            const uint32_t aphase = (it >> 1) & 1;
            const uint32_t taddr0 = tlane + as * BLOCK_N;
            const uint32_t full_addr = tmem_full_addr + 8u * as, empty_addr = (tmem_empty_addr + 8u * as) & empty_mask;
            const int m_tile = tile / n_tiles_n;
            if (swap) {
                const int ch_warp = (tile - m_tile * n_tiles_n) * BLOCK_M + quarter * 32;
                if (p.epi_mode == 0 && !p.residual && p.swap_tma && p.act != 2 && !(kDev && p.debug))
                    epilogue_tile_swapped<true, MISH>(p, &tmOut, sbuf, taddr0, reinterpret_cast<float*>(stage), ch_warp, static_cast<long long>(m_tile) * 256,
                                                lane, half, full_addr, aphase, empty_addr, prof ? t_acc : nullptr);
                else
                    epilogue_tile_swapped<false, MISH>(p, &tmOut, sbuf, taddr0, reinterpret_cast<float*>(stage), ch_warp, static_cast<long long>(m_tile) * 256,
                                                 lane, half, full_addr, aphase, empty_addr, prof ? t_acc : nullptr);
                continue;
            }
            const int n0 = (tile - m_tile * n_tiles_n) * BLOCK_N;
            const long long m_base = (strip ? p.strip_qfirst : 0) + static_cast<long long>(m_tile) * TILE_M + cta_rank * BLOCK_M + quarter * 32;
            if constexpr (STRIP) {
                if (p.residual)
                    epilogue_tile<BLOCK_N, true, true, false, MISH>(p, &tmOut, taddr0, stage, sbuf, m_base, n0, lane, half, full_addr, aphase, empty_addr,
                                                       prof ? t_acc : nullptr, tile, part, static_cast<int>(cta_rank) * 4 + quarter);
                else
                    epilogue_tile<BLOCK_N, true, false, false, MISH>(p, &tmOut, taddr0, stage, sbuf, m_base, n0, lane, half, full_addr, aphase, empty_addr,
                                                        prof ? t_acc : nullptr, tile, part, static_cast<int>(cta_rank) * 4 + quarter);
            } else if (BLOCK_N >= 128 && fast_epi) {
                if (p.residual)
                    epilogue_tile<BLOCK_N, false, true, true, MISH>(p, &tmOut, taddr0, stage, sbuf, m_base, n0, lane, half, full_addr, aphase, empty_addr,
                                                              prof ? t_acc : nullptr, tile, part, static_cast<int>(cta_rank) * 4 + quarter);
                else
                    epilogue_tile<BLOCK_N, false, false, true, MISH>(p, &tmOut, taddr0, stage, sbuf, m_base, n0, lane, half, full_addr, aphase, empty_addr,
                                                               prof ? t_acc : nullptr, tile, part, static_cast<int>(cta_rank) * 4 + quarter);
            } else {
                epilogue_tile<BLOCK_N, false, false, false, MISH>(p, &tmOut, taddr0, stage, sbuf, m_base, n0, lane, half, full_addr, aphase, empty_addr,
                                       prof ? t_acc : nullptr, tile, part, static_cast<int>(cta_rank) * 4 + quarter);
            }
        }
        if (lane == 0) ptx::tma_store_wait<0>();  // outstanding TMA stores read this CTA's shared memory
        if (prof && warp == 4 && lane == 0) {
            long long* o = p.prof + blockIdx.x * 16;
            o[5] = clock64() - t_start; o[6] = t_acc[0]; o[7] = t_acc[1]; o[8] = t_acc[2]; o[9] = t_acc[3]; o[10] = t_acc[4]; o[11] = t_acc[5];
        }
    }

    ptx::tc_fence_before();
    if (TWO) ptx::cluster_sync(); else __syncthreads();
    if (warp == 2) {
        ptx::tc_fence_after();
        if (TWO) ptx::tmem_dealloc2(tmem_base_v, Cfg::TMEM_COLS);
        else ptx::tmem_dealloc(tmem_base_v, Cfg::TMEM_COLS);
    }
}

// ------------------------------------------------------------------------------------------ host
namespace {

typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                    const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                    CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
typedef CUresult (*PFN_encodeIm2col)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                     const cuuint64_t*, const int*, const int*, cuuint32_t, cuuint32_t,
                                     const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                     CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

PFN_encodeTiled g_encodeTiled = nullptr;
PFN_encodeIm2col g_encodeIm2col = nullptr;
int g_driver_version = 0;

void set_err(char* err, size_t n, const char* fmt, long long a = 0, long long b = 0, long long c = 0) {
    if (err && n) snprintf(err, n, fmt, a, b, c);
}

template <int BN, bool TWO, bool SWAP = false, bool STRIP = false, bool MISH = false>
int set_smem_attr() {
    return cudaFuncSetAttribute(conv_tc_kernel<BN, TWO, SWAP, STRIP, MISH>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_LIMIT) == cudaSuccess
               ? 0
               : -1;
}

}  // namespace

int conv_tc_init(char* err, size_t errlen) {
    if (!g_encodeTiled) {
        cudaDriverEntryPointQueryResult q;
        void* f = nullptr;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &f, cudaEnableDefault, &q) != cudaSuccess || !f) {
            set_err(err, errlen, "cuTensorMapEncodeTiled entry point unavailable");
            return -1;
        }
        g_encodeTiled = reinterpret_cast<PFN_encodeTiled>(f);
        f = nullptr;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeIm2col", &f, cudaEnableDefault, &q) != cudaSuccess || !f) {
            set_err(err, errlen, "cuTensorMapEncodeIm2col entry point unavailable");
            return -1;
        }
        g_encodeIm2col = reinterpret_cast<PFN_encodeIm2col>(f);
        cudaDriverGetVersion(&g_driver_version);
    }
    if (set_smem_attr<32, false>() || set_smem_attr<64, false>() || set_smem_attr<128, false>() ||
        set_smem_attr<256, false>() || set_smem_attr<256, true>() || set_smem_attr<256, false, true>() ||
        set_smem_attr<256, true, false, true>() || set_smem_attr<32, false, false, false, true>() ||
        set_smem_attr<64, false, false, false, true>() || set_smem_attr<128, false, false, false, true>() ||
        set_smem_attr<256, false, false, false, true>() || set_smem_attr<256, true, false, false, true>() ||
        set_smem_attr<256, false, true, false, true>() || set_smem_attr<256, true, false, true, true>()) {
        set_err(err, errlen, "cudaFuncSetAttribute(MaxDynamicSharedMemorySize) failed: %lld",
                static_cast<long long>(cudaGetLastError()));
        return -1;
    }
    return 0;
}

int encode_tiled_bf16(CUtensorMap* out, void* base, int rank, const unsigned long long* dims,
                      const unsigned long long* strides_bytes, const unsigned* box, int swizzle) {
    if (!g_encodeTiled && conv_tc_init(nullptr, 0)) return -1;
    cuuint64_t d[5], st[4];
    cuuint32_t b[5], es[5];
    for (int i = 0; i < rank; ++i) { d[i] = dims[i]; b[i] = box[i]; es[i] = 1; }
    for (int i = 0; i + 1 < rank; ++i) st[i] = strides_bytes[i];
    const CUtensorMapSwizzle sw = swizzle == 3 ? CU_TENSOR_MAP_SWIZZLE_128B : swizzle == 2 ? CU_TENSOR_MAP_SWIZZLE_64B
                                  : swizzle == 1 ? CU_TENSOR_MAP_SWIZZLE_32B : CU_TENSOR_MAP_SWIZZLE_NONE;
    return g_encodeTiled(out, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, rank, base, d, st, b, es, CU_TENSOR_MAP_INTERLEAVE_NONE, sw,
                         CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS ? 0 : -1;
}

static int choose_block_n(int cout, long long m_tiles, int num_sms) {
    (void)m_tiles; (void)num_sms;
    // One 128 x N x 16 MMA reads A (4 KB) + B (N*32 B) from shared memory; at N = 128 that is exactly the
    // 128 B/clk/SM shared-memory bandwidth, so N = 256 is the only shape that keeps the tensor pipe fed
    // (measured: 1.15-1.22 PFLOP/s at N = 256 vs 0.68 at N = 128 on the hot 3x3 layers).
    if (cout <= 32) return 32;
    if (cout <= 64) return 64;
    if (cout <= 128) return 128;
    return 256;
}

int conv_tc_prepare(const ConvDesc& d, int num_sms, int block_n_hint, ConvLaunch* L, char* err, size_t errlen) {
    if (!g_encodeTiled && conv_tc_init(err, errlen)) return -1;
    memset(L, 0, sizeof(*L));
    const int k = d.ksize;
    if (!(k == 1 || k == 3)) { set_err(err, errlen, "conv_tc: unsupported kernel size %lld", k); return -1; }
    if (d.cin % 16 != 0) { set_err(err, errlen, "conv_tc: Cin=%lld is not a multiple of 16", d.cin); return -1; }
    if (d.in_pitch % 8 != 0 || d.out_pitch % 4 != 0 || (!d.out_fp32 && (d.out_pitch % 8 != 0 || d.cout % 8 != 0))) {
        set_err(err, errlen, "conv_tc: pitches/channels must keep 16-byte alignment (in_pitch=%lld out_pitch=%lld)",
                d.in_pitch, d.out_pitch);
        return -1;
    }
    if ((reinterpret_cast<uintptr_t>(d.in) & 15) || (reinterpret_cast<uintptr_t>(d.out) & 15) ||
        (reinterpret_cast<uintptr_t>(d.w) & 15) || (d.residual && (reinterpret_cast<uintptr_t>(d.residual) & 15))) {
        set_err(err, errlen, "conv_tc: pointers must be 16-byte aligned");
        return -1;
    }
    const int ho = (d.hi + d.pad_lo + d.pad_hi - k) / d.stride + 1;
    const int wo = (d.wi + d.pad_lo + d.pad_hi - k) / d.stride + 1;
    const long long M = 1LL * d.n * ho * wo;
    if (M <= 0 || M > 0x7fffffffLL) { set_err(err, errlen, "conv_tc: bad M=%lld", M); return -1; }
    const int block_k = (d.cin % 64 == 0) ? 64 : (d.cin % 32 == 0 ? 32 : 16);
    const int cin_blocks = d.cin / block_k;
    const int K = k * k * d.cin;
    long long m_tiles = (M + BLOCK_M - 1) / BLOCK_M;
    // swapped mode for narrow layers: channels on the MMA's M side (128-row tiles), 256 pixels on its N side
    // (only where Cout fills the 128 lanes: with fewer channels most epilogue warps idle and the normal mode wins)
    const Options& O = options();
    int swap = (d.cout > 64 && d.cout <= 128 && !d.out_fp32 && M >= 256) ? 1 : 0;
    if (block_n_hint == 1024) { swap = 1; block_n_hint = 0; }
    else if (block_n_hint) swap = 0;
    // Small batches: a layer whose 256-wide tiles would occupy less than a quarter of the SMs is cut into 128 x 64 (or
    // 128 x 128) single-CTA tiles instead — up to eight times as many CTAs, each with a proportionally shorter main loop.
    // A launch is as long as ONE CTA's work, and at batch 1 that is what a layer costs: full-416 batch 1 0.90 -> 0.64 ms.
    // 64-wide tiles where they still fit the GPU in one wave, 128-wide otherwise (measured: 64 everywhere makes batch 4
    // slower than the 256-wide default, 128 faster).
    if (!block_n_hint && !d.out_fp32 && O.strip != 2) {  // (strip = 2 forces the CTA-pair strip form wherever it is legal)
        const long long tiles256 = ((M + 255) / 256) * ((d.cout + 255) / 256);
        if (tiles256 * 4 <= num_sms) {
            const int lb = ((M + BLOCK_M - 1) / BLOCK_M) * ((d.cout + 63) / 64) <= num_sms ? 64 : 128;
            if (d.cout > lb) { swap = 0; block_n_hint = lb; }
        }
    }
    if (swap) block_n_hint = 257;
    int two = -1;  // -1: decide below
    if (block_n_hint == 512) { two = 1; block_n_hint = 256; }
    if (block_n_hint == 257) { two = 0; block_n_hint = 256; }
    int bn = block_n_hint ? block_n_hint : choose_block_n(d.cout, m_tiles, num_sms);
    if (!(bn == 32 || bn == 64 || bn == 128 || bn == 256)) { set_err(err, errlen, "conv_tc: bad block_n %lld", bn); return -1; }

    if (two < 0) two = (bn == 256 && block_k == 64 && m_tiles >= 2) ? 1 : 0;
    if (two && (bn != 256 || block_k != 64)) { set_err(err, errlen, "conv_tc: the CTA-pair kernel needs Cout > 128 and Cin %% 64 == 0"); return -1; }
    if (two) m_tiles = (M + 2 * BLOCK_M - 1) / (2 * BLOCK_M);
    // (clusters of two pairs sharing the filter tile through TMA multicast were built and measured in round 1: 812 instead
    // of 738 cycles per K block per CTA and only 32 clusters of 4 co-resident — removed, see DESIGN.md)
    if (swap) m_tiles = (M + 255) / 256;
    ConvParams& p = L->p;
    // strip mode (see ConvParams::strip): 3x3 / stride 1 / pad 1 layers of the CTA-pair kernel on maps where the pad
    // positions cost less than the operand bytes saved.  Option strip: 0 switches it off, 2 forces it wherever it is legal.
    {
        const int strip_env = O.strip;
        // one shared pad column between consecutive image rows and one shared pad row between consecutive images are
        // enough (the right neighbour of a row's last pixel IS the next row's left pad): (W+1)(H+1) positions per image
        const int wp = d.wi + 1, hp = d.hi + 1, rows = 128 + 2 * wp + 2;
        // the strip kernel compiles the max(x, alpha x) form and Mish, not the select form
        const bool plain_act = !d.act || d.act == 2 || (d.alpha >= 0.f && d.alpha <= 1.f);
        const bool legal = two && plain_act && k == 3 && d.stride == 1 && d.pad_lo == 1 && d.pad_hi == 1 && block_k == 64 && !d.out_fp32 &&
                           !d.upsample2x && rows <= 400 && static_cast<long long>(d.n) * wp * hp < (1LL << 30);  // 400 rows: two strip buffers + a 5-stage B ring still fit
        constexpr int STRIP_MIN_W = 12;  // (W+1)(H+1)/(WH) extra rows: 1.04 at 52x52, 1.08 at 26x26, 1.16 at 13x13
        const bool pays = d.wi >= STRIP_MIN_W;
        // small batches keep the im2col form: it can split K over idle CTA pairs, the strip form cannot
        const long long strip_tiles = (static_cast<long long>(d.n) * wp * hp - (wp + 1) + 2 * BLOCK_M - 1) / (2 * BLOCK_M) * ((d.cout + bn - 1) / bn);
        const bool fills = strip_tiles >= num_sms / 2;
        if (legal && strip_env && ((pays && fills) || strip_env == 2)) {
            p.strip = 1;
            p.strip_wp = wp; p.strip_hp = hp; p.strip_rows = rows;
            p.strip_qfirst = wp + 1;
            p.strip_total_q = static_cast<int>(d.n) * wp * hp;
            m_tiles = (p.strip_total_q - p.strip_qfirst + 2 * BLOCK_M - 1) / (2 * BLOCK_M);
        }
    }
    p.M = static_cast<int>(M);
    p.cout = d.cout;
    p.num_k_blocks = k * k * cin_blocks;
    p.cin_blocks = cin_blocks;
    p.ksize = k;
    p.stride = d.stride;
    p.pad_lo = d.pad_lo;
    p.ho = ho;
    p.wo = wo;
    p.block_k = block_k;
    p.a_im2col = !(k == 1 && d.stride == 1 && d.pad_lo == 0 && d.pad_hi == 0);
    p.num_m_tiles = static_cast<int>(m_tiles);
    p.num_n_tiles = swap ? (d.cout + BLOCK_M - 1) / BLOCK_M : (d.cout + bn - 1) / bn;
    p.swap = swap;
    if (d.cout > 1024) { set_err(err, errlen, "conv_tc: Cout=%lld exceeds the 1024-entry bias block", d.cout); return -1; }
    if (!d.bias_host) { set_err(err, errlen, "conv_tc: bias_host is required"); return -1; }
    memset(p.bias_c, 0, sizeof(p.bias_c));
    memcpy(p.bias_c, d.bias_host, sizeof(float) * d.cout);
    p.epi_mode = d.out_fp32 ? 1 : (d.upsample2x ? 2 : 0);
    p.res_v8 = (d.residual && (reinterpret_cast<uintptr_t>(d.residual) & 31) == 0 && d.res_pitch % 16 == 0 && d.cout % 16 == 0) ? 1 : 0;
    if (d.residual && p.epi_mode != 0 && !swap) { set_err(err, errlen, "conv_tc: a residual needs a plain bf16 output"); return -1; }
    p.bias = d.bias;
    p.act = d.act == 2 ? 3 : d.act ? ((d.alpha >= 0.f && d.alpha <= 1.f) ? 1 : 2) : 0;  // 1: max(x, alpha x); 2: select form; 3: Mish
    p.alpha = d.alpha;
    p.residual = d.residual;
    p.res_pitch = d.res_pitch;
    p.out = d.out;
    p.out_pitch = d.out_pitch;
    p.out_fp32 = d.out_fp32;
    p.upsample2x = d.upsample2x;
    p.n_store_limit = d.out_fp32 ? d.out_pitch : d.cout;
    if (d.upsample2x && d.out_fp32) { set_err(err, errlen, "conv_tc: upsample2x needs a bf16 output"); return -1; }

    const CUtensorMapSwizzle swz = (block_k == 64)   ? CU_TENSOR_MAP_SWIZZLE_128B
                                   : (block_k == 32) ? CU_TENSOR_MAP_SWIZZLE_64B
                                                     : CU_TENSOR_MAP_SWIZZLE_32B;
    CUresult r;
    if (!p.a_im2col) {
        cuuint64_t dims[2] = {static_cast<cuuint64_t>(d.cin), static_cast<cuuint64_t>(M)};
        cuuint64_t strides[1] = {static_cast<cuuint64_t>(d.in_pitch) * 2};
        cuuint32_t box[2] = {static_cast<cuuint32_t>(block_k), static_cast<cuuint32_t>(swap ? 256 : BLOCK_M)};
        cuuint32_t estr[2] = {1, 1};
        r = g_encodeTiled(&L->tmA, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<__nv_bfloat16*>(d.in), dims,
                          strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, swz, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                          CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    } else {
        cuuint64_t dims[4] = {static_cast<cuuint64_t>(d.cin), static_cast<cuuint64_t>(d.wi),
                              static_cast<cuuint64_t>(d.hi), static_cast<cuuint64_t>(d.n)};
        cuuint64_t strides[3] = {static_cast<cuuint64_t>(d.in_pitch) * 2,
                                 static_cast<cuuint64_t>(d.in_pitch) * 2 * d.wi,
                                 static_cast<cuuint64_t>(d.in_pitch) * 2 * d.wi * d.hi};
        int lower[2] = {-d.pad_lo, -d.pad_lo};
        int upper[2] = {d.pad_hi - (k - 1), d.pad_hi - (k - 1)};
        if (p.strip) { lower[0] = lower[1] = -1; upper[0] = upper[1] = 0; }  // traversal = the image with a pad column / row in front: W+1 x H+1
        cuuint32_t estr[4] = {1, static_cast<cuuint32_t>(d.stride), static_cast<cuuint32_t>(d.stride), 1};
        r = g_encodeIm2col(&L->tmA, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, const_cast<__nv_bfloat16*>(d.in), dims,
                           strides, lower, upper, static_cast<cuuint32_t>(block_k),
                           p.strip ? static_cast<cuuint32_t>(p.strip_rows) : (swap ? 256u : BLOCK_M), estr,
                           CU_TENSOR_MAP_INTERLEAVE_NONE, swz, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                           CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        // Same driver quirk CUTLASS works around for im2col maps over small tensors (< 128 KiB).
        const unsigned long long bytes = 2ULL * d.in_pitch * d.wi * d.hi * d.n;
        if (r == CUDA_SUCCESS && g_driver_version <= 13010 && bytes < 131072ULL)
            reinterpret_cast<uint64_t*>(&L->tmA)[1] &= ~(1ULL << 21);
    }
    if (r != CUDA_SUCCESS) { set_err(err, errlen, "conv_tc: tensor map A encode failed (CUresult %lld)", r); return -1; }
    {
        cuuint64_t dims[2] = {static_cast<cuuint64_t>(K), static_cast<cuuint64_t>(d.cout)};
        cuuint64_t strides[1] = {static_cast<cuuint64_t>(K) * 2};
        cuuint32_t box[2] = {static_cast<cuuint32_t>(block_k), static_cast<cuuint32_t>(swap ? BLOCK_M : (two ? bn / 2 : bn))};
        cuuint32_t estr[2] = {1, 1};
        r = g_encodeTiled(&L->tmB, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<__nv_bfloat16*>(d.w), dims,
                          strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, swz, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                          CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        if (r != CUDA_SUCCESS) { set_err(err, errlen, "conv_tc: tensor map B encode failed (CUresult %lld)", r); return -1; }
    }
    p.swap_tma = swap ? 1 : 0;
    if (p.epi_mode == 0 && (!swap || p.swap_tma)) {
        cuuint64_t dims[2] = {static_cast<cuuint64_t>(d.cout), static_cast<cuuint64_t>(M)};
        cuuint64_t strides[1] = {static_cast<cuuint64_t>(d.out_pitch) * 2};
        p.store64 = (bn >= 128 && !swap) ? 1 : 0;  // 128-byte store rows (two 32-column chunks per TMA store)
        cuuint32_t box[2] = {p.store64 ? 64u : 32u, 32};
        cuuint32_t estr[2] = {1, 1};
        r = g_encodeTiled(&L->tmOut, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, d.out, dims, strides, box, estr,
                          CU_TENSOR_MAP_INTERLEAVE_NONE, p.store64 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B,
                          CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        if (r != CUDA_SUCCESS) { set_err(err, errlen, "conv_tc: tensor map OUT encode failed (CUresult %lld)", r); return -1; }
    } else if (p.epi_mode == 1 && !swap) {
        // fp32 head rows [M][out_pitch]: 32 columns x 32 rows per store (128-byte rows, SWIZZLE_128B)
        cuuint64_t dims[2] = {static_cast<cuuint64_t>(d.out_pitch), static_cast<cuuint64_t>(M)};
        cuuint64_t strides[1] = {static_cast<cuuint64_t>(d.out_pitch) * 4};
        cuuint32_t box[2] = {32, 32};
        cuuint32_t estr[2] = {1, 1};
        r = g_encodeTiled(&L->tmOut, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, d.out, dims, strides, box, estr,
                          CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_NONE,
                          CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        if (r != CUDA_SUCCESS) { set_err(err, errlen, "conv_tc: fp32 tensor map OUT encode failed (CUresult %lld)", r); return -1; }
        p.head_tma = 1;
    } else {
        L->tmOut = L->tmB;  // unused by these modes; any valid map
    }
    L->block_n = bn;
    L->two_cta = two;
    // split-K for launches that cannot fill the GPU with whole tiles (small batches): parts of >= 4 K blocks
    p.split_k = 1;
    {
        const long long whole = m_tiles * p.num_n_tiles;
        const long long units_max = two ? num_sms / 2 : num_sms;
        // (a split costs ~8-10 us of fences, counter traffic and partial-sum reads, so it only pays on long K loops)
        constexpr int SPLIT_K_MIN_KB = 32, SPLIT_K_MAX = 4;
        if (d.allow_split_k && !swap && !p.strip && bn >= 64 && whole * 2 <= units_max && p.num_k_blocks >= SPLIT_K_MIN_KB) {
            long long sk = units_max / whole;
            if (sk > SPLIT_K_MAX) sk = SPLIT_K_MAX;
            if (sk > p.num_k_blocks / 4) sk = p.num_k_blocks / 4;
            if (sk >= 2) p.split_k = static_cast<int>(sk);
        }
    }
    L->ws_bytes = p.split_k > 1 ? static_cast<size_t>(m_tiles * p.num_n_tiles) * p.split_k * 8 * 32 * bn * sizeof(float) : 0;
    L->counter_ints = p.split_k > 1 ? static_cast<size_t>(m_tiles * p.num_n_tiles) * 16 : 0;
    const long long tiles = m_tiles * p.num_n_tiles * p.split_k;
    if (two) {
        const long long pairs = num_sms / 2;
        L->grid = 2 * static_cast<int>(tiles < pairs ? tiles : pairs);
    } else {
        L->grid = static_cast<int>(tiles < num_sms ? tiles : num_sms);
    }
    // operand ring.  One K block of a narrow layer is only a few hundred tensor-core cycles of work but costs a
    // full barrier round trip (~450 cycles of wait/fence/commit in the issuing warp), so narrow layers put several
    // K blocks into one stage; then as many stages as fit (bytes in flight hide the ~1.5 us L2->SM fill latency).
    const int b_total = bn * K * 2;  // the whole filter bank of one N tile
    const int b_res = (!two && !swap && p.num_n_tiles == 1 && b_total <= 65536) ? 1 : 0;
    p.b_resident = b_res;
    const int sub_bytes = ((p.strip ? 0 : BLOCK_M) + (b_res ? 0 : (two ? bn / 2 : bn))) * block_k * 2;
    const int strips_bytes = p.strip ? 2 * ((p.strip_rows * 128 + 1023) / 1024 * 1024) : 0;
    int kps = 1;
    const int ring_avail = SMEM_LIMIT - 1024 - SMEM_RING_OFF - (b_res ? b_total : 0);
    if (swap) {
        kps = 49152 / sub_bytes;  // 48 KB stages, 4 of them
        if (kps < 1) kps = 1;
        if (kps > p.num_k_blocks) kps = p.num_k_blocks;
    } else if (!two && bn <= 128 && sub_bytes <= 16384) {
        kps = ring_avail / (4 * sub_bytes);  // keep at least 4 stages in flight
        if (kps < 1) kps = 1;
        if (kps > 4) kps = 4;
        if (kps > p.num_k_blocks) kps = p.num_k_blocks;
        if (k == 3 && p.num_k_blocks % 3 == 0 && kps == 4) kps = 3;  // keep whole filter rows together
    }
    const int stage_bytes = sub_bytes * kps;
    int stages = (SMEM_LIMIT - 1024 - SMEM_RING_OFF - strips_bytes - (b_res ? bn * block_k * 2 * p.num_k_blocks : 0)) / stage_bytes;
    if (stages > MAX_STAGES) stages = MAX_STAGES;
    if (stages < 2) { set_err(err, errlen, "conv_tc: stage does not fit in shared memory"); return -1; }
    p.num_stages = stages;
    p.kb_per_stage = kps;
    L->smem_bytes = 1024 + SMEM_RING_OFF + (b_res ? bn * block_k * 2 * p.num_k_blocks : 0) + static_cast<size_t>(stages) * stage_bytes + strips_bytes;
    L->flops = 2.0 * double(M) * d.cout * K;
    return 0;
}

// the Mish instantiations of the same forms
static int launch_mish(const ConvLaunch& L, cudaLaunchConfig_t& cfg) {
    cudaError_t e;
    if (L.two_cta && L.p.strip) e = cudaLaunchKernelEx(&cfg, conv_tc_kernel<256, true, false, true, true>, L.tmA, L.tmB, L.tmOut, L.p);
    else if (L.two_cta) e = cudaLaunchKernelEx(&cfg, conv_tc_kernel<256, true, false, false, true>, L.tmA, L.tmB, L.tmOut, L.p);
    else if (L.p.swap) e = cudaLaunchKernelEx(&cfg, conv_tc_kernel<256, false, true, false, true>, L.tmA, L.tmB, L.tmOut, L.p);
    else switch (L.block_n) {
        case 32: e = cudaLaunchKernelEx(&cfg, conv_tc_kernel<32, false, false, false, true>, L.tmA, L.tmB, L.tmOut, L.p); break;
        case 64: e = cudaLaunchKernelEx(&cfg, conv_tc_kernel<64, false, false, false, true>, L.tmA, L.tmB, L.tmOut, L.p); break;
        case 128: e = cudaLaunchKernelEx(&cfg, conv_tc_kernel<128, false, false, false, true>, L.tmA, L.tmB, L.tmOut, L.p); break;
        case 256: e = cudaLaunchKernelEx(&cfg, conv_tc_kernel<256, false, false, false, true>, L.tmA, L.tmB, L.tmOut, L.p); break;
        default: return -1;
    }
    return e == cudaSuccess ? 0 : -1;
}

void conv_tc_bind_workspace(ConvLaunch* L, float* ws, int* counters) {
    L->p.ws = ws;
    L->p.counters = counters;
}

int conv_tc_launch(const ConvLaunch& L, cudaStream_t stream) {
    if (L.p.split_k > 1 && (!L.p.ws || !L.p.counters)) return -1;  // conv_tc_bind_workspace was not called
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(L.grid);
    cfg.blockDim = dim3(NUM_THREADS);
    cfg.dynamicSmemBytes = L.smem_bytes;
    cfg.stream = stream;
    cudaLaunchAttribute attr[2];
    int na = 0;
    if (L.two_cta) {
        attr[na].id = cudaLaunchAttributeClusterDimension;
        attr[na].val.clusterDim.x = 2;
        attr[na].val.clusterDim.y = 1;
        attr[na].val.clusterDim.z = 1;
        ++na;
    }
    // programmatic dependent launch: this kernel may start while its predecessor in the stream drains
    attr[na].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[na].val.programmaticStreamSerializationAllowed = 1;
    ++na;
    cfg.attrs = attr;
    cfg.numAttrs = na;
    cudaError_t e;
    if (L.p.act == 3) return launch_mish(L, cfg);
    if (L.two_cta && L.p.strip) e = cudaLaunchKernelEx(&cfg, conv_tc_kernel<256, true, false, true>, L.tmA, L.tmB, L.tmOut, L.p);
    else if (L.two_cta) e = cudaLaunchKernelEx(&cfg, conv_tc_kernel<256, true>, L.tmA, L.tmB, L.tmOut, L.p);
    else if (L.p.swap) e = cudaLaunchKernelEx(&cfg, conv_tc_kernel<256, false, true>, L.tmA, L.tmB, L.tmOut, L.p);
    else switch (L.block_n) {
        case 32: e = cudaLaunchKernelEx(&cfg, conv_tc_kernel<32, false>, L.tmA, L.tmB, L.tmOut, L.p); break;
        case 64: e = cudaLaunchKernelEx(&cfg, conv_tc_kernel<64, false>, L.tmA, L.tmB, L.tmOut, L.p); break;
        case 128: e = cudaLaunchKernelEx(&cfg, conv_tc_kernel<128, false>, L.tmA, L.tmB, L.tmOut, L.p); break;
        case 256: e = cudaLaunchKernelEx(&cfg, conv_tc_kernel<256, false>, L.tmA, L.tmB, L.tmOut, L.p); break;
        default: return -1;
    }
    return e == cudaSuccess ? 0 : -1;
}

}  // namespace fd
