// conv_halo.cu — 3x3 convolution (stride 1 or 2, pad 1) for NARROW inputs (Cin = 16, 32 or 64) on large feature maps, with the
// im2col done by the tensor core's operand addressing over a halo patch that is loaded ONCE per tile.
//
// Why a second conv kernel: conv_tc.cu feeds its A operand with im2col TMA loads, one "row" (pixel) per L2 request.
// The L2 takes about one request per 3 cycles per SM whatever its size, and a 32-channel pixel is only 64 bytes, so the
// 9 taps x 128 pixels = 1152 requests of a tile starve the tensor core (YOLOv3's conv2 / conv4: 341 / 346 us at batch
// 64 against an HBM bound of ~160 / 135 us).  Here every input pixel of a tile is fetched once, by coalesced 16-byte
// cp.async copies (8 pixels x 64 B = one 512-byte run per instruction), into a layout the MMA can read all 9 taps from:
//
//   * un-swizzled K-major operand: a "core matrix" is 8 rows x 16 bytes with the rows 16 bytes apart; the next 8-row
//     group is SBO bytes further, the next 16-byte K chunk LBO bytes further (same scheme as pre.cu's first layer);
//   * the patch is stored as chunk planes: plane c holds channels 8c..8c+7 of every patch pixel, 16 bytes per pixel, in
//     row-major pixel order.  8 consecutive pixels of an image row are then one core matrix, SBO = one patch row walks
//     down the 16 image rows of the tile (M = 128 = 16 rows x 8 pixels), LBO = one plane steps to the next 8 channels;
//   * tap (r, s) of the filter is the same patch viewed from pixel (r, s): only the descriptor's start address moves;
//   * stride 2: the patch is split into 4 parity sub-planes (row parity, column parity), so that the pixels
//     2*ox + s for consecutive ox are again 16 bytes apart.
//
// Roles (17 warps): 8 epilogue warps in two groups (even / odd tiles; TMEM lane quarter = warp % 4), 1 MMA warp, 8
// builder warps in two teams (even / odd tiles) that never wait for a copy: the copies of every free patch slot (8 at
// stride 1, 4 at stride 2) are in flight at once and arrive on the slot's barrier asynchronously.
// Replaces the same Conv+BatchNormalization+LeakyRelu(+Add) node groups as conv_tc.cu (reference server/detector.py:135).
#include "conv_halo.h"

#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include "conv_tc.h"
#include "ptx.cuh"

namespace fd {

namespace {

constexpr int TW = 8, TH = 16;           // output tile (pixels): 16 rows x 8 columns = the 128 rows of one MMA
constexpr int EPI_WARPS = 8, MMA_WARP = 8, BUILD_WARPS = 8;
constexpr int THREADS = (EPI_WARPS + 1 + BUILD_WARPS) * 32;
constexpr int ACCS = 4;
constexpr int SMEM_LIMIT = 227 * 1024;

template <int STRIDE>
struct Geo {
    // full patch in input pixels
    static constexpr int PH = STRIDE == 1 ? TH + 2 : 2 * TH + 1;
    static constexpr int PW = STRIDE == 1 ? TW + 2 : 2 * TW + 1;
    // parity sub-plane (stride 2) / the whole patch (stride 1)
    static constexpr int SPH = STRIDE == 1 ? PH : TH + 1;
    static constexpr int SPW = STRIDE == 1 ? PW : TW + 1;
    static constexpr int PLANE_PIX = (STRIDE == 1 ? 1 : 4) * SPH * SPW;
    static constexpr int PLANE_BASE = ((PLANE_PIX * 16 + 127) / 128) * 128;
    static constexpr int SBO = SPW * 16;
};
// Plane stride.  The builders' cp.async items run chunk-fastest (8 lanes = one 128-byte shared-memory wavefront cover
// 8 / NCH pixels x NCH chunks), so chunk planes a multiple of 128 bytes apart put the NCH chunks of a pixel on the same
// banks: an NCH-way conflict on every copy (ncu, conv2: 87 % of the shared-memory pipe).  Skewing the planes by 128 / NCH
// bytes spreads the 8 items of a quarter warp over the 8 distinct 16-byte slots of a wavefront.
template <int CIN, int STRIDE>
struct Plane { static constexpr int BYTES = Geo<STRIDE>::PLANE_BASE + 128 / (CIN / 8); };
// patch ring depth: the copies of SLOTS tiles are in flight at once (the ~3 us DRAM/L2 round trip of a patch is what has
// to be covered: conv4 moved 4.2 TB/s with 8 slots = 94 KB in flight per SM, exactly latency x concurrency).  Bounded by
// shared memory: 32-channel stride-2 patches are 39 KB each; with 64 input channels the resident filter bank (up to
// 147 KB) leaves room for two 23 KB patches.
template <int CIN, int STRIDE>
struct Ring { static constexpr int SLOTS = CIN == 64 ? 2 : (STRIDE == 1 ? 12 : 4); };

__device__ __forceinline__ int div_magic(int x, unsigned long long m) {
    return static_cast<int>((static_cast<unsigned long long>(x) * m) >> 40);
}
__device__ __forceinline__ uint32_t pack2(float a, float b) {
    __nv_bfloat162 v = __floats2bfloat162_rn(a, b);
    return *reinterpret_cast<uint32_t*>(&v);
}
__device__ __forceinline__ uint32_t max_bf16x2(uint32_t a, uint32_t b) {
    const __nv_bfloat162 r = __hmax2(*reinterpret_cast<const __nv_bfloat162*>(&a), *reinterpret_cast<const __nv_bfloat162*>(&b));
    return *reinterpret_cast<const uint32_t*>(&r);
}
__device__ __forceinline__ uint32_t add_bf16x2(uint32_t a, uint32_t b) {
    const __nv_bfloat162 r = __hadd2(*reinterpret_cast<const __nv_bfloat162*>(&a), *reinterpret_cast<const __nv_bfloat162*>(&b));
    return *reinterpret_cast<const uint32_t*>(&r);
}
// un-swizzled K-major shared-memory descriptor: start, LBO (K chunk stride), SBO (8-row group stride), all bytes
__device__ __forceinline__ uint64_t desc_kmajor(uint32_t addr, uint32_t lbo, uint32_t sbo) {
    return static_cast<uint64_t>((addr >> 4) & 0x3FFF) | (static_cast<uint64_t>((lbo >> 4) & 0x3FFF) << 16) |
           (static_cast<uint64_t>((sbo >> 4) & 0x3FFF) << 32) | (static_cast<uint64_t>(1) << 46);
}

template <int CIN, int STRIDE>
__global__ void __launch_bounds__(THREADS, 1)
conv_halo_kernel(const __grid_constant__ CUtensorMap tm_out, const __grid_constant__ HaloParams p) {
    using G = Geo<STRIDE>;
    constexpr int NCH = CIN / 8;                    // 16-byte channel chunks per pixel
    constexpr int PLANE_BYTES = Plane<CIN, STRIDE>::BYTES;
    constexpr int PATCH_BYTES = NCH * PLANE_BYTES;
    constexpr int KSTEPS = CIN / 16;                // MMAs per filter tap
    constexpr int SLOTS = Ring<CIN, STRIDE>::SLOTS;
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    // [0, 1024) barriers | staging 8 warps x 4 KB | weights 9*NCH*cout*16 | patch ring SLOTS x PATCH_BYTES
    uint64_t* patch_full = reinterpret_cast<uint64_t*>(smem);
    uint64_t* patch_empty = patch_full + SLOTS;
    uint64_t* acc_full = patch_empty + SLOTS;
    uint64_t* acc_empty = acc_full + ACCS;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(acc_empty + ACCS);
    uint8_t* s_stage = smem + 1024;
    uint8_t* s_w = s_stage + EPI_WARPS * 4096;
    const int cout = p.cout;
    uint8_t* s_patch = s_w + ((9 * NCH * cout * 16 + 1023) & ~1023);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    // weights (a constant of the layer: before the dependency wait): global [cout][9*CIN] -> smem [K chunk][filter][16 B]
    for (int i = tid; i < 9 * NCH * cout; i += THREADS) {
        const int kc = i / cout, f = i - kc * cout;
        *reinterpret_cast<uint4*>(s_w + i * 16) = __ldg(reinterpret_cast<const uint4*>(p.w + static_cast<size_t>(f) * 9 * CIN + kc * 8));
    }
    if (tid == 0) {
        for (int i = 0; i < SLOTS; ++i) { ptx::mbar_init(&patch_full[i], 128); ptx::mbar_init(&patch_empty[i], 1); }  // full: one asynchronous arrive per thread of a builder team
        for (int i = 0; i < ACCS; ++i) { ptx::mbar_init(&acc_full[i], 1); ptx::mbar_init(&acc_empty[i], 4); }
        ptx::fence_barrier_init();
        ptx::tma_prefetch_desc(&tm_out);
    }
    const uint32_t acc_cols = cout <= 32 ? 32u : (cout <= 64 ? 64u : 128u);
    if (warp == MMA_WARP) {
        ptx::tmem_alloc(tmem_slot, ACCS * acc_cols);
        ptx::tmem_relinquish();
    }
    ptx::fence_proxy_async();  // the weight tile is read by the tensor core
    ptx::tc_fence_before();
    __syncthreads();
    ptx::tc_fence_after();
    const uint32_t tmem = *tmem_slot;
    ptx::grid_dep_launch();

    const int tiles_x = p.tiles_x, per_frame = p.per_frame, total = p.total;
    const int my_tiles = (total > static_cast<int>(blockIdx.x)) ? (total - 1 - static_cast<int>(blockIdx.x)) / static_cast<int>(gridDim.x) + 1 : 0;

    if (warp > MMA_WARP) {
        // ---------------------------------------------------------------- builders
        // team t = 4 warps takes the tiles of parity t; a lane copies items q = pixel * NCH + chunk, q = ltid, ltid + 128,
        // ...: consecutive lanes take consecutive 16-byte chunks, i.e. whole pixels, i.e. 512-byte runs of an image row.
        // Nothing here waits for a copy: each thread's arrival on the slot's barrier is itself asynchronous
        // (cp.async.mbarrier.arrive), so the copies of every free slot are in flight at once.
        const int bw = warp - MMA_WARP - 1, team = bw >> 2, ltid = (bw & 3) * 32 + lane;
        constexpr int ITEMS = G::PH * G::PW * NCH;
        const uint32_t patch_base = ptx::smem_u32(s_patch);
        ptx::grid_dep_wait();
        for (int it = team; it < my_tiles; it += 2) {
            const int slot = it % SLOTS;
            const int tile = blockIdx.x + it * gridDim.x;
            const int f = div_magic(tile, p.m_per_frame);
            const int rem = tile - f * per_frame;
            const int ty = div_magic(rem, p.m_tiles_x), tx = rem - ty * tiles_x;
            const int y_org = ty * TH * STRIDE - 1, x_org = tx * TW * STRIDE - 1;
            const __nv_bfloat16* frame = p.in + static_cast<long long>(f) * p.hi * p.wi * p.in_pitch;
            const uint32_t dst0 = patch_base + slot * PATCH_BYTES;
            ptx::mbar_wait(&patch_empty[slot], ((it / SLOTS) & 1) ^ 1);
#pragma unroll 4
            for (int q = ltid; q < ITEMS; q += 128) {
                const int pix = q / NCH, c = q - pix * NCH;
                const int iy = pix / G::PW, ix = pix - iy * G::PW;
                const int gy = y_org + iy, gx = x_org + ix;
                const bool ok = gy >= 0 && gy < p.hi && gx >= 0 && gx < p.wi;
                const int idx = STRIDE == 1 ? pix : (((iy & 1) * 2 + (ix & 1)) * (G::SPH * G::SPW) + (iy >> 1) * G::SPW + (ix >> 1));
                const __nv_bfloat16* src = ok ? frame + (static_cast<long long>(gy) * p.wi + gx) * p.in_pitch + c * 8 : p.in;
                ptx::cp_async_16(dst0 + c * PLANE_BYTES + idx * 16, src, ok ? 16u : 0u);  // 0 bytes: zero fill (padding)
            }
            ptx::cp_async_arrive_noinc(&patch_full[slot]);
        }
    } else if (warp == MMA_WARP) {
        // ---------------------------------------------------------------- MMA issuer (all operands warp-uniform)
        const uint32_t idesc = ptx::make_idesc_bf16_f32(128, cout);
        const uint32_t w_addr = __shfl_sync(0xffffffffu, ptx::smem_u32(s_w), 0);
        const uint32_t p_addr0 = __shfl_sync(0xffffffffu, ptx::smem_u32(s_patch), 0);
        const uint32_t bar0 = __shfl_sync(0xffffffffu, ptx::smem_u32(patch_full), 0);  // full, empty, acc_full, acc_empty: 8-byte steps
        const uint32_t tmem_u = __shfl_sync(0xffffffffu, tmem, 0);
        const uint64_t a0 = desc_kmajor(p_addr0, PLANE_BYTES, G::SBO);
        const uint64_t b0 = desc_kmajor(w_addr, cout * 16, 128);
        const uint32_t b_step = static_cast<uint32_t>(cout) * 2;  // two K chunks per MMA, in 16-byte units: 2 * cout * 16 / 16
        const bool issuer = ptx::elect_one();
        for (int it = 0; it < my_tiles; ++it) {
            const uint32_t slot = it % SLOTS, phase = (it / SLOTS) & 1, as = it & 3, aphase = (it >> 2) & 1;
            ptx::mbar_wait_addr(bar0 + 8u * (2 * SLOTS + ACCS + as), aphase ^ 1);  // acc_empty
            ptx::mbar_wait_addr(bar0 + 8u * slot, phase);                          // patch_full
            ptx::fence_proxy_async();  // the builders' cp.async writes (generic proxy), acquired through the barrier -> tensor core
            ptx::tc_fence_after();
            const uint64_t ad = a0 + slot * (PATCH_BYTES / 16);
            const uint32_t d = tmem_u + as * acc_cols;
            if (issuer) {
#pragma unroll
                for (int t = 0; t < 9; ++t) {
                    const int r = t / 3, s = t - 3 * r;
                    const int start = STRIDE == 1 ? (r * G::PW + s)
                                                  : (((r & 1) * 2 + (s & 1)) * (G::SPH * G::SPW) + (r >> 1) * G::SPW + (s >> 1));
#pragma unroll
                    for (int j = 0; j < KSTEPS; ++j)
                        ptx::umma_bf16(d, ad + start + j * (2 * PLANE_BYTES / 16), b0 + (t * KSTEPS + j) * b_step, idesc,
                                       (t | j) ? 1u : 0u);
                }
                ptx::umma_commit_addr(bar0 + 8u * (SLOTS + slot));    // patch_empty
                ptx::umma_commit_addr(bar0 + 8u * (2 * SLOTS + as));  // acc_full
            }
            __syncwarp();
        }
    } else {
        // ---------------------------------------------------------------- epilogue group g: tiles it = g, g + 2, ...
        const int group = warp >> 2, quarter = warp & 3;
        uint8_t* stage = s_stage + warp * 4096;
        const float alpha_eff = p.act ? p.alpha : 1.0f;
        const float2 a2 = make_float2(alpha_eff, alpha_eff);
        const bool generic_act = p.act == 2;
        const bool has_res = p.residual != nullptr;
        int sbuf = 0;
        ptx::grid_dep_wait();
        for (int it = group; it < my_tiles; it += 2) {
            const int as = it & 3;
            const int tile = blockIdx.x + it * gridDim.x;
            const int f = div_magic(tile, p.m_per_frame);
            const int rem = tile - f * per_frame;
            const int ty = div_magic(rem, p.m_tiles_x), tx = rem - ty * tiles_x;
            const int oy = ty * TH + 4 * quarter + (lane >> 3), ox = tx * TW + (lane & 7);  // this lane's output pixel
            const bool inside = oy < p.ho && ox < p.wo;
            const __nv_bfloat16* res_row = p.residual + ((static_cast<long long>(f) * p.ho + oy) * p.wo + ox) * p.res_pitch;
            ptx::U32x8 rnext[2];
            auto fetch_res = [&](int c0) {
#pragma unroll
                for (int i = 0; i < 2; ++i) {
#pragma unroll
                    for (int e = 0; e < 8; ++e) rnext[i].v[e] = 0u;
                    if (has_res && inside && c0 + 16 * i < cout) rnext[i] = ptx::ld_nc_v8(res_row + c0 + 16 * i);
                }
            };
            fetch_res(0);
            if (has_res && it + 2 < my_tiles) {
                // pull the NEXT tile's residual rows (this lane's pixel, all channels) towards L2 now: no registers held,
                // and the loads above then come from L2 instead of DRAM (they were the epilogue's largest stall)
                const int tile2 = blockIdx.x + (it + 2) * gridDim.x;
                const int f2 = div_magic(tile2, p.m_per_frame);
                const int rem2 = tile2 - f2 * per_frame;
                const int ty2 = div_magic(rem2, p.m_tiles_x), tx2 = rem2 - ty2 * tiles_x;
                const int oy2 = ty2 * TH + 4 * quarter + (lane >> 3), ox2 = tx2 * TW + (lane & 7);
                if (oy2 < p.ho && ox2 < p.wo) {
                    const __nv_bfloat16* r2 = p.residual + ((static_cast<long long>(f2) * p.ho + oy2) * p.wo + ox2) * p.res_pitch;
                    asm volatile("prefetch.global.L2 [%0];" ::"l"(r2));
                    if (cout > 64) asm volatile("prefetch.global.L2 [%0];" ::"l"(r2 + 64));
                }
            }
            ptx::mbar_wait(&acc_full[as], (it >> 2) & 1);
            ptx::tc_fence_after();
            const uint32_t taddr = tmem + as * acc_cols + (static_cast<uint32_t>(quarter * 32) << 16);
            const bool rotate = cout > 64;  // wide outputs: two 2 KB staging buffers used in turn, one store per chunk
            if (!rotate) {
                if (lane == 0) ptx::tma_store_wait_read<0>();  // this warp's previous stores have finished reading the staging rows
                __syncwarp();
            }
            for (int c0 = 0; c0 < cout; c0 += 32) {
                uint32_t acc[32];
                ptx::tmem_ld_32x32(taddr + c0, acc);
                ptx::U32x8 rcur[2];
                rcur[0] = rnext[0];
                rcur[1] = rnext[1];
                if (c0 + 32 < cout) fetch_res(c0 + 32);
                ptx::tmem_ld_wait();
                if (c0 + 32 >= cout) {  // accumulator drained: hand the stage back to the MMA warp
                    ptx::tc_fence_before();
                    __syncwarp();
                    if (lane == 0) ptx::mbar_arrive(&acc_empty[as]);
                }
                const float* bias = p.bias_c + c0;  // constant bank, warp-uniform index
                uint32_t pk[16];
#pragma unroll
                for (int g = 0; g < 16; ++g) {
                    float2 x = __fadd2_rn(make_float2(__uint_as_float(acc[2 * g]), __uint_as_float(acc[2 * g + 1])),
                                          make_float2(bias[2 * g], bias[2 * g + 1]));
                    if (!generic_act) {
                        const float2 m = __fmul2_rn(x, a2);
                        x.x = fmaxf(x.x, m.x);
                        x.y = fmaxf(x.y, m.y);
                    } else {
                        x.x = x.x > 0.f ? x.x : x.x * p.alpha;
                        x.y = x.y > 0.f ? x.y : x.y * p.alpha;
                    }
                    pk[g] = pack2(x.x, x.y);
                }
                if (has_res) {  // (bf16x2 add: the fp32 form used by conv_tc.cu costs this kernel 20 % on its three residual layers, conv4 / conv7 / conv9)
#pragma unroll
                    for (int g = 0; g < 16; ++g) pk[g] = add_bf16x2(pk[g], rcur[g >> 3].v[g & 7]);
                }
                // MaxPool(2, 2) in place: lane = (row lane >> 3, column lane & 7) of the warp's 4 x 8 pixels, so a 2x2 window is
                // lanes l, l^1, l^8, l^9; the lane with even row and even column keeps the maximum (bf16 max is exact)
                if (p.pool2) {
#pragma unroll
                    for (int g = 0; g < 16; ++g) {
                        uint32_t v = max_bf16x2(pk[g], __shfl_xor_sync(0xffffffffu, pk[g], 1));
                        pk[g] = max_bf16x2(v, __shfl_xor_sync(0xffffffffu, v, 8));
                    }
                }
                // 32 pixels x 64 B with the 64-byte swizzle (chunk c of row r at slot c ^ ((r >> 1) & 3)): a SWIZZLE_64B box
                uint8_t* so = stage + ((rotate ? sbuf : (c0 >> 5)) & 1) * 2048;
                if (rotate) {
                    if (lane == 0) ptx::tma_store_wait_read<1>();  // the store that used this buffer two chunks ago is done with it
                    __syncwarp();
                }
                // pooled: the 8 surviving pixels [2 rows][4 columns] are rows 0..7 of the (smaller) box
                const int srow = p.pool2 ? ((lane >> 4) * 4 + ((lane & 7) >> 1)) : lane;
                if (!p.pool2 || (lane & 9) == 0) {
#pragma unroll
                    for (int c = 0; c < 4; ++c)
                        *reinterpret_cast<uint4*>(so + srow * 64 + ((c ^ ((srow >> 1) & 3)) << 4)) = make_uint4(pk[4 * c], pk[4 * c + 1], pk[4 * c + 2], pk[4 * c + 3]);
                }
                if (rotate) {
                    ptx::fence_proxy_async();
                    __syncwarp();
                    if (lane == 0) {
                        if (p.pool2) ptx::tma_store_4d(&tm_out, so, c0, tx * (TW / 2), ty * (TH / 2) + 2 * quarter, f);
                        else ptx::tma_store_4d(&tm_out, so, c0, tx * TW, ty * TH + 4 * quarter, f);
                        ptx::tma_store_commit();
                    }
                    ++sbuf;
                }
            }
            if (!rotate) {
                ptx::fence_proxy_async();
                __syncwarp();
                if (lane == 0) {
                    for (int c0 = 0; c0 < cout; c0 += 32) {
                        if (p.pool2) ptx::tma_store_4d(&tm_out, stage + (c0 >> 5) * 2048, c0, tx * (TW / 2), ty * (TH / 2) + 2 * quarter, f);
                        else ptx::tma_store_4d(&tm_out, stage + (c0 >> 5) * 2048, c0, tx * TW, ty * TH + 4 * quarter, f);  // clipped at the edges
                    }
                    ptx::tma_store_commit();
                }
            }
        }
        if (lane == 0) ptx::tma_store_wait<0>();
    }
    ptx::tc_fence_before();
    __syncthreads();
    if (warp == MMA_WARP) {
        ptx::tc_fence_after();
        ptx::tmem_dealloc(tmem, ACCS * acc_cols);
    }
}

template <int CIN, int STRIDE>
size_t smem_bytes(int cout) {
    return 1024 + 1024 + EPI_WARPS * 4096 + ((9 * (CIN / 8) * cout * 16 + 1023) & ~1023) +
           static_cast<size_t>(Ring<CIN, STRIDE>::SLOTS) * (CIN / 8) * Plane<CIN, STRIDE>::BYTES;
}

}  // namespace

bool conv_halo_supported(const HaloDesc& d) {
    if (!(d.cin == 64 || d.cin == 32 || d.cin == 16) || d.ksize != 3 || d.pad_lo != 1 || d.pad_hi > 1 || !(d.stride == 1 || d.stride == 2)) return false;
    if (!(d.cout == 32 || d.cout == 64 || d.cout == 128) || d.out_fp32 || d.upsample2x) return false;
    if (d.pool2 && (d.stride != 1 || d.residual || d.hi % 2 || d.wi % 2 || d.pad_hi != 1)) return false;
    if (d.cin == 64 && d.stride != 1) return false;  // the 78 KB stride-2 patch does not fit next to the resident filters
    if (d.in_pitch % 8 || d.out_pitch % 8 || (reinterpret_cast<uintptr_t>(d.in) & 15) || (reinterpret_cast<uintptr_t>(d.out) & 15) ||
        (reinterpret_cast<uintptr_t>(d.w) & 15))
        return false;
    if (d.residual && ((reinterpret_cast<uintptr_t>(d.residual) & 31) || d.res_pitch % 16)) return false;
    const int ho = (d.hi + d.pad_lo + d.pad_hi - 3) / d.stride + 1, wo = (d.wi + d.pad_lo + d.pad_hi - 3) / d.stride + 1;
    // worth it on large maps only: small ones waste too much of the fixed 16 x 8 tile
    if (ho < 64 || wo < 64) return false;
    const long long tiles = 1LL * d.n * ((wo + TW - 1) / TW) * ((ho + TH - 1) / TH);
    return tiles < (1LL << 24) && 1LL * ((wo + TW - 1) / TW) * ((ho + TH - 1) / TH) < (1 << 16);
}

int conv_halo_prepare(const HaloDesc& d, int num_sms, HaloLaunch* L, char* err, size_t errlen) {
    memset(L, 0, sizeof(*L));
    if (!conv_halo_supported(d)) { if (err && errlen) snprintf(err, errlen, "conv_halo: unsupported layer"); return -1; }
    HaloParams& p = L->p;
    p.in = d.in; p.n = d.n; p.hi = d.hi; p.wi = d.wi; p.in_pitch = d.in_pitch;
    p.stride = d.stride;
    p.ho = (d.hi + d.pad_lo + d.pad_hi - 3) / d.stride + 1;
    p.wo = (d.wi + d.pad_lo + d.pad_hi - 3) / d.stride + 1;
    p.w = d.w; p.cin = d.cin; p.cout = d.cout;
    p.act = d.act ? ((d.alpha >= 0.f && d.alpha <= 1.f) ? 1 : 2) : 0;
    p.alpha = d.alpha;
    p.residual = d.residual; p.res_pitch = d.res_pitch;
    p.pool2 = d.pool2;
    p.tiles_x = (p.wo + TW - 1) / TW;
    p.tiles_y = (p.ho + TH - 1) / TH;
    p.per_frame = p.tiles_x * p.tiles_y;
    p.total = d.n * p.per_frame;
    const unsigned long long one40 = 1ULL << 40;
    p.m_per_frame = (one40 + p.per_frame - 1) / p.per_frame;
    p.m_tiles_x = (one40 + p.tiles_x - 1) / p.tiles_x;
    memset(p.bias_c, 0, sizeof(p.bias_c));
    memcpy(p.bias_c, d.bias_host, sizeof(float) * d.cout);
    // output map: the conv's (ho, wo) grid, or the pooled (ho/2, wo/2) one; a warp's box = its 4 x 8 pixels (2 x 4 pooled)
    const int oh = d.pool2 ? p.ho / 2 : p.ho, ow = d.pool2 ? p.wo / 2 : p.wo;
    const unsigned long long dims[4] = {static_cast<unsigned long long>(d.cout), static_cast<unsigned long long>(ow),
                                        static_cast<unsigned long long>(oh), static_cast<unsigned long long>(d.n)};
    const unsigned long long strides[3] = {2ULL * d.out_pitch, 2ULL * d.out_pitch * ow, 2ULL * d.out_pitch * ow * oh};
    const unsigned box[4] = {32, d.pool2 ? TW / 2u : TW, d.pool2 ? 2u : 4u, 1};
    if (encode_tiled_bf16(&L->tm_out, d.out, 4, dims, strides, box, 2)) { if (err && errlen) snprintf(err, errlen, "conv_halo: output tensor map encode failed"); return -1; }
    L->stride = d.stride;
    L->cin = d.cin;
    L->smem_bytes = d.cin == 64 ? smem_bytes<64, 1>(d.cout)
                    : d.cin == 32 ? (d.stride == 1 ? smem_bytes<32, 1>(d.cout) : smem_bytes<32, 2>(d.cout))
                                  : (d.stride == 1 ? smem_bytes<16, 1>(d.cout) : smem_bytes<16, 2>(d.cout));
    if (L->smem_bytes > static_cast<size_t>(SMEM_LIMIT)) { if (err && errlen) snprintf(err, errlen, "conv_halo: %zu bytes of shared memory", L->smem_bytes); return -1; }
    L->grid = p.total < num_sms ? p.total : num_sms;
    L->flops = 2.0 * d.n * p.ho * p.wo * d.cout * 9.0 * d.cin;
    return 0;
}

// One-time per DEVICE (the attribute belongs to the device's context: a process that drives several GPUs must set it on
// each — a once-per-process guard here made every halo launch on the second and later GPUs of fd_server fail).
int conv_halo_init() {
    return (cudaFuncSetAttribute(conv_halo_kernel<32, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_LIMIT) == cudaSuccess &&
            cudaFuncSetAttribute(conv_halo_kernel<32, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_LIMIT) == cudaSuccess &&
            cudaFuncSetAttribute(conv_halo_kernel<64, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_LIMIT) == cudaSuccess &&
            cudaFuncSetAttribute(conv_halo_kernel<16, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_LIMIT) == cudaSuccess &&
            cudaFuncSetAttribute(conv_halo_kernel<16, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_LIMIT) == cudaSuccess)
               ? 0
               : -1;
}

int conv_halo_launch(const HaloLaunch& L, cudaStream_t stream) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(L.grid);
    cfg.blockDim = dim3(THREADS);
    cfg.dynamicSmemBytes = L.smem_bytes;
    cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    cudaError_t e;
    if (L.cin == 64) e = cudaLaunchKernelEx(&cfg, conv_halo_kernel<64, 1>, L.tm_out, L.p);
    else if (L.cin == 32) e = L.stride == 1 ? cudaLaunchKernelEx(&cfg, conv_halo_kernel<32, 1>, L.tm_out, L.p) : cudaLaunchKernelEx(&cfg, conv_halo_kernel<32, 2>, L.tm_out, L.p);
    else e = L.stride == 1 ? cudaLaunchKernelEx(&cfg, conv_halo_kernel<16, 1>, L.tm_out, L.p) : cudaLaunchKernelEx(&cfg, conv_halo_kernel<16, 2>, L.tm_out, L.p);
    return e == cudaSuccess ? 0 : -1;
}

}  // namespace fd
