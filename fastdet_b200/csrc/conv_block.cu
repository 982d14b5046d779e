// conv_block.cu — one residual block of the narrow, large-map stage in ONE kernel:
//   x (64 ch) -> conv 1x1 (64 -> 32) -> LeakyReLU -> conv 3x3 (32 -> 64, stride 1, pad 1) -> LeakyReLU -> + x -> bf16 NHWC.
//
// Why: as two kernels (YOLOv3's conv3 + conv4 at 208x208) the block reads x, writes the 32-channel tensor, reads it back
// and reads x again as the residual: 1.4 GB of HBM traffic per 64 frames for 0.30 ms.  Fused, the halo patch of x is loaded
// ONCE per tile (cp.async, chunk planes, as conv_halo.cu does for its input), the 1x1 convolution runs on the whole patch
// (a 1x1 needs no spatial order, so the patch is simply 180 consecutive "rows" of the MMA: two M = 128 blocks), its
// output goes through registers into the chunk planes the 3x3 reads its nine taps from, and the residual comes out of the
// x patch that is already in shared memory.  HBM sees x once and the block's output once.
//
// Per tile of 16 x 8 output pixels:
//   builders   (4 warps) cp.async the 18 x 10 x 64-channel patch of x into 8 chunk planes (zero fill outside the image); the
//              copies of every free slot are in flight at once and arrive on the slot's barrier asynchronously;
//   MMA warp   issues the 1x1 of tile t+1 (2 blocks x 4 MMAs, N = 32) and then the 3x3 of tile t (18 MMAs, N = 64, exactly
//              conv_halo.cu's stride-1 loop), so the tensor pipe has work while tile t's middle patch is finished;
//   epilogue A (8 warps: block b = warp / 4) drains the 1x1: bias, LeakyReLU, bf16, zero outside the image (the 3x3 pads
//              the 1x1's OUTPUT with zeros), 16-byte chunks into the middle patch's chunk planes;
//   epilogue B (8 warps, two groups on alternate tiles) drains the 3x3: bias, LeakyReLU, + x in fp32 (one rounding, like the reference's Add), bf16 rows
//              staged with the 64-byte swizzle, TMA stores; it releases the x patch (together with the 1x1's commit).
// Replaces the Conv+BN+LeakyRelu, Conv+BN+LeakyRelu, Add node group of YOLOv3's first residual block
// (reference server/detector.py:135).
#include "conv_block.h"

#include <stdio.h>
#include <string.h>

#include "conv_tc.h"
#include "ptx.cuh"

namespace fd {

namespace {

constexpr int TW = 8, TH = 16;                 // output tile: 16 rows x 8 columns = the 128 rows of one MMA
constexpr int CIN = 64, CMID = 32, COUT = 64;
constexpr int EPIA_WARPS = 8;                  // warps 0..7: block = warp / 4, TMEM lane quarter = warp % 4
constexpr int EPIB_WARPS = 8;                  // warps 8..15: two groups of 4, even / odd tiles (one warp's tile takes ~2000 cycles)
constexpr int MMA_WARP = EPIA_WARPS + EPIB_WARPS;  // warp 16
constexpr int BUILD_WARPS = 4;                 // warps 17..20
constexpr int THREADS = (MMA_WARP + 1 + BUILD_WARPS) * 32;
constexpr int PH = TH + 2, PW = TW + 2, NPIX = PH * PW;   // 18 x 10 halo patch, 180 pixels in row-major order
constexpr int NCH_IN = CIN / 8, NCH_MID = CMID / 8;       // 16-byte channel chunks per pixel
constexpr int BLOCKS_A = (NPIX + 127) / 128;              // 1x1: M blocks over the flat patch
// chunk planes: plane c holds channels 8c..8c+7 of every patch pixel, 16 bytes per pixel.  The input planes are skewed by
// 16 bytes (the builders' items run chunk-fastest: 8 lanes = the 8 chunks of a pixel must not share a bank group).
constexpr int PLANE_IN = ((NPIX * 16 + 127) / 128) * 128 + 16;
constexpr int IN_SLOT_BYTES = NCH_IN * PLANE_IN;
constexpr int IN_SLOTS = 5;
// block 1 of the 1x1 reads rows 128..255 of every plane: past the 180 pixels into the next plane, and past the last plane
// into the next slot or this tail — all of which hold zeros or activations (finite: the rows are never stored)
constexpr int IN_TAIL = ((BLOCKS_A * 128 * 16 - PLANE_IN + 127) / 128) * 128;
constexpr int PLANE_MID = ((NPIX * 16 + 127) / 128) * 128;
constexpr int MID_BYTES = NCH_MID * PLANE_MID;
constexpr int MID_SLOTS = 2;
constexpr int ACCBS = 4;
constexpr int TMEM_ACCB = 64, TMEM_COLS = 512;            // 1x1 accumulators: columns [0, 2 * 32); 3x3: [64, 64 + 4 * 64)
constexpr int WA_BYTES = NCH_IN * CMID * 16, WB_BYTES = 9 * NCH_MID * COUT * 16;
constexpr int OFF_WA = 1024, OFF_STAGE = 6144;
constexpr int OFF_WB = OFF_STAGE + EPIB_WARPS * 4096;
constexpr int OFF_MID = OFF_WB + WB_BYTES;
constexpr int OFF_IN = OFF_MID + MID_SLOTS * MID_BYTES;
constexpr int SMEM_BYTES = OFF_IN + IN_SLOTS * IN_SLOT_BYTES + IN_TAIL + 1024;  // + alignment slack
static_assert(WA_BYTES <= OFF_STAGE - OFF_WA && OFF_WB % 1024 == 0 && OFF_MID % 128 == 0 && OFF_IN % 128 == 0, "shared-memory layout");
static_assert(BLOCKS_A * 32 <= TMEM_ACCB && TMEM_ACCB + ACCBS * COUT <= TMEM_COLS, "TMEM columns");
static_assert(SMEM_BYTES <= 227 * 1024, "shared memory");
static_assert(BLOCKS_A == 2 && EPIA_WARPS == 4 * BLOCKS_A, "one epilogue-A group per 1x1 block");

__device__ __forceinline__ int div_magic(int x, unsigned long long m) {
    return static_cast<int>((static_cast<unsigned long long>(x) * m) >> 40);
}
__device__ __forceinline__ uint32_t pack2(float a, float b) {
    __nv_bfloat162 v = __floats2bfloat162_rn(a, b);
    return *reinterpret_cast<uint32_t*>(&v);
}
// un-swizzled K-major shared-memory descriptor: start, LBO (K chunk stride), SBO (8-row group stride), all bytes
__device__ __forceinline__ uint64_t desc_kmajor(uint32_t addr, uint32_t lbo, uint32_t sbo) {
    return static_cast<uint64_t>((addr >> 4) & 0x3FFF) | (static_cast<uint64_t>((lbo >> 4) & 0x3FFF) << 16) |
           (static_cast<uint64_t>((sbo >> 4) & 0x3FFF) << 32) | (static_cast<uint64_t>(1) << 46);
}
// bias + LeakyReLU as max(x, alpha x) (alpha in [0, 1]; 1 = linear) on two fp32 accumulator columns
__device__ __forceinline__ float2 bias_act(uint32_t a0, uint32_t a1, float b0, float b1, float2 alpha2) {
    const float2 x = __fadd2_rn(make_float2(__uint_as_float(a0), __uint_as_float(a1)), make_float2(b0, b1));
    const float2 m = __fmul2_rn(x, alpha2);
    return make_float2(fmaxf(x.x, m.x), fmaxf(x.y, m.y));
}

// developer switches / per-role cycle accounting (harness build only; the shipped kernel carries none of these branches)
#ifdef FASTDET_DEV
#define BLK_DBG(bit) ((p.debug & (bit)) != 0)
#define PROF_DECL long long prof_acc[4] = {0, 0, 0, 0}; const long long prof_t0 = clock64();
#define PROF_WAIT(slot, stmt) do { const long long t_ = clock64(); stmt; prof_acc[slot] += clock64() - t_; } while (0)
#define PROF_STORE(base, who) do { if (p.prof && (who)) { long long* o_ = p.prof + blockIdx.x * 16 + (base); o_[0] = clock64() - prof_t0; \
        o_[1] = prof_acc[0]; o_[2] = prof_acc[1]; o_[3] = prof_acc[2]; } } while (0)
#else
#define BLK_DBG(bit) false
#define PROF_DECL
#define PROF_WAIT(slot, stmt) stmt
#define PROF_STORE(base, who)
#endif

__global__ void __launch_bounds__(THREADS, 1)
conv_block_kernel(const __grid_constant__ CUtensorMap tm_out, const __grid_constant__ BlockParams p) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    uint64_t* in_full = reinterpret_cast<uint64_t*>(smem);
    uint64_t* in_empty = in_full + IN_SLOTS;
    uint64_t* acca_full = in_empty + IN_SLOTS;      // one per 1x1 block
    uint64_t* acca_empty = acca_full + BLOCKS_A;    // one for both blocks
    uint64_t* mid_full = acca_empty + 1;
    uint64_t* mid_empty = mid_full + MID_SLOTS;
    uint64_t* accb_full = mid_empty + MID_SLOTS;
    uint64_t* accb_empty = accb_full + ACCBS;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(accb_empty + ACCBS);
    uint8_t* s_wa = smem + OFF_WA;
    uint8_t* s_stage = smem + OFF_STAGE;
    uint8_t* s_wb = smem + OFF_WB;
    uint8_t* s_mid = smem + OFF_MID;
    uint8_t* s_in = smem + OFF_IN;

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    // ---- constants of the layer pair (before the dependency wait)
    // 1x1 filters: global [32][64] -> [K chunk][32 filters][16 B]
    for (int i = tid; i < NCH_IN * CMID; i += THREADS) {
        const int kc = i / CMID, f = i - kc * CMID;
        *reinterpret_cast<uint4*>(s_wa + i * 16) = __ldg(reinterpret_cast<const uint4*>(p.wa + static_cast<size_t>(f) * CIN + kc * 8));
    }
    // 3x3 filters: global [64][9 * 32] -> [K chunk = tap * 4 + channel chunk][64 filters][16 B]
    for (int i = tid; i < 9 * NCH_MID * COUT; i += THREADS) {
        const int kc = i / COUT, f = i - kc * COUT;
        *reinterpret_cast<uint4*>(s_wb + i * 16) = __ldg(reinterpret_cast<const uint4*>(p.wb + static_cast<size_t>(f) * 9 * CMID + kc * 8));
    }
    for (int i = tid; i < (MID_SLOTS * MID_BYTES + IN_SLOTS * IN_SLOT_BYTES + IN_TAIL) / 16; i += THREADS)
        reinterpret_cast<uint4*>(s_mid)[i] = make_uint4(0u, 0u, 0u, 0u);
    if (tid == 0) {
        for (int i = 0; i < IN_SLOTS; ++i) { ptx::mbar_init(&in_full[i], BUILD_WARPS * 32); ptx::mbar_init(&in_empty[i], 1 + 4); }
        for (int i = 0; i < BLOCKS_A; ++i) ptx::mbar_init(&acca_full[i], 1);
        ptx::mbar_init(acca_empty, EPIA_WARPS);
        for (int i = 0; i < MID_SLOTS; ++i) { ptx::mbar_init(&mid_full[i], EPIA_WARPS); ptx::mbar_init(&mid_empty[i], 1); }
        for (int i = 0; i < ACCBS; ++i) { ptx::mbar_init(&accb_full[i], 1); ptx::mbar_init(&accb_empty[i], 4); }
        ptx::fence_barrier_init();
        ptx::tma_prefetch_desc(&tm_out);
    }
    if (warp == MMA_WARP) {
        ptx::tmem_alloc(tmem_slot, TMEM_COLS);
        ptx::tmem_relinquish();
    }
    ptx::fence_proxy_async();  // filter tiles and the zeroed patches are read by the tensor core
    ptx::tc_fence_before();
    __syncthreads();
    ptx::tc_fence_after();
    const uint32_t tmem = *tmem_slot;
    ptx::grid_dep_launch();

    const int tiles_x = p.tiles_x, per_frame = p.per_frame, total = p.total;
    const int my_tiles = (total > static_cast<int>(blockIdx.x)) ? (total - 1 - static_cast<int>(blockIdx.x)) / static_cast<int>(gridDim.x) + 1 : 0;

    if (warp > MMA_WARP) {
        // ---------------------------------------------------------------- builders: the x patch, 8 chunk planes
        // a lane copies items q = pixel * 8 + chunk, q = ltid, ltid + 128, ...: consecutive lanes take consecutive 16-byte
        // chunks, i.e. whole pixels, i.e. 1280-byte runs of an image row.  Nothing here waits for a copy.
        const int ltid = (warp - MMA_WARP - 1) * 32 + lane;
        constexpr int ITEMS = NPIX * NCH_IN;
        const uint32_t in_base = ptx::smem_u32(s_in);
        PROF_DECL
        ptx::grid_dep_wait();
        for (int it = 0; it < my_tiles; ++it) {
            const int slot = it % IN_SLOTS;
            const int tile = blockIdx.x + it * gridDim.x;
            const int f = div_magic(tile, p.m_per_frame);
            const int rem = tile - f * per_frame;
            const int ty = div_magic(rem, p.m_tiles_x), tx = rem - ty * tiles_x;
            const int y_org = ty * TH - 1, x_org = tx * TW - 1;
            const __nv_bfloat16* frame = p.in + static_cast<long long>(f) * p.h * p.w * p.in_pitch;
            const uint32_t dst0 = in_base + slot * IN_SLOT_BYTES;
            PROF_WAIT(0, ptx::mbar_wait(&in_empty[slot], ((it / IN_SLOTS) & 1) ^ 1));
#pragma unroll 4
            for (int q = ltid; q < ITEMS; q += BUILD_WARPS * 32) {
                const int pix = q >> 3, c = q & 7;
                const int iy = pix / PW, ix = pix - iy * PW;
                const int gy = y_org + iy, gx = x_org + ix;
                const bool ok = gy >= 0 && gy < p.h && gx >= 0 && gx < p.w && !BLK_DBG(1);
                const __nv_bfloat16* src = ok ? frame + (static_cast<long long>(gy) * p.w + gx) * p.in_pitch + c * 8 : p.in;
                ptx::cp_async_16(dst0 + c * PLANE_IN + pix * 16, src, ok ? 16u : 0u);  // 0 bytes: zero fill (outside the image)
            }
            ptx::cp_async_arrive_noinc(&in_full[slot]);
        }
        PROF_STORE(0, ltid == 0);
    } else if (warp == MMA_WARP) {
        // ---------------------------------------------------------------- MMA issuer (all operands warp-uniform)
        const uint32_t idesc_a = ptx::make_idesc_bf16_f32(128, CMID), idesc_b = ptx::make_idesc_bf16_f32(128, COUT);
        const uint32_t bar0 = __shfl_sync(0xffffffffu, ptx::smem_u32(in_full), 0);  // all barriers: 8-byte steps from in_full
        const uint32_t tmem_u = __shfl_sync(0xffffffffu, tmem, 0);
        const uint64_t a_in = desc_kmajor(__shfl_sync(0xffffffffu, ptx::smem_u32(s_in), 0), PLANE_IN, 128);
        const uint64_t b_wa = desc_kmajor(__shfl_sync(0xffffffffu, ptx::smem_u32(s_wa), 0), CMID * 16, 128);
        const uint64_t a_mid = desc_kmajor(__shfl_sync(0xffffffffu, ptx::smem_u32(s_mid), 0), PLANE_MID, PW * 16);
        const uint64_t b_wb = desc_kmajor(__shfl_sync(0xffffffffu, ptx::smem_u32(s_wb), 0), COUT * 16, 128);
        constexpr uint32_t BAR_IN_EMPTY = IN_SLOTS, BAR_AA_FULL = 2 * IN_SLOTS, BAR_AA_EMPTY = BAR_AA_FULL + BLOCKS_A,
                           BAR_MID_FULL = BAR_AA_EMPTY + 1, BAR_MID_EMPTY = BAR_MID_FULL + MID_SLOTS,
                           BAR_AB_FULL = BAR_MID_EMPTY + MID_SLOTS, BAR_AB_EMPTY = BAR_AB_FULL + ACCBS;
        const bool issuer = ptx::elect_one();
        PROF_DECL
        for (int step = 0; step <= my_tiles; ++step) {
            if (step < my_tiles) {
                // 1x1 of tile `step`: the flat patch as 2 blocks of 128 rows, K = 64 in 4 MMAs each
                const int it = step;
                const uint32_t slot = it % IN_SLOTS;
                PROF_WAIT(0, ptx::mbar_wait_addr(bar0 + 8u * slot, (it / IN_SLOTS) & 1));  // in_full
                ptx::fence_proxy_async();  // the builders' cp.async writes (generic proxy), acquired through the barrier -> tensor core
                PROF_WAIT(1, ptx::mbar_wait_addr(bar0 + 8u * BAR_AA_EMPTY, (it & 1) ^ 1));  // the previous tile's 1x1 accumulators are drained
                ptx::tc_fence_after();
                const uint64_t ad = a_in + slot * (IN_SLOT_BYTES / 16);
                if (issuer) {
#pragma unroll
                    for (int b = 0; b < BLOCKS_A; ++b) {
#pragma unroll
                        for (int j = 0; j < CIN / 16; ++j)
                            if (!BLK_DBG(4)) ptx::umma_bf16(tmem_u + b * 32, ad + b * (128 * 16 / 16) + j * (2 * PLANE_IN / 16), b_wa + j * (2 * CMID), idesc_a, j ? 1u : 0u);
                        ptx::umma_commit_addr(bar0 + 8u * (BAR_AA_FULL + b));
                    }
                    ptx::umma_commit_addr(bar0 + 8u * (BAR_IN_EMPTY + slot));  // (1 of the slot's 5 releases: epilogue B still reads the residual)
                }
                __syncwarp();
            }
            if (step >= 1) {
                // 3x3 of tile `step - 1`: its middle patch has been finished by the epilogue-A warps meanwhile
                const int it = step - 1;
                const uint32_t c = it & 1, as = it & 3;
                PROF_WAIT(2, ptx::mbar_wait_addr(bar0 + 8u * (BAR_AB_EMPTY + as), ((it >> 2) & 1) ^ 1));
                PROF_WAIT(2, ptx::mbar_wait_addr(bar0 + 8u * (BAR_MID_FULL + c), (it >> 1) & 1));  // (the writers fenced: generic -> async proxy)
                ptx::tc_fence_after();
                const uint64_t ad = a_mid + c * (MID_BYTES / 16);
                const uint32_t d = tmem_u + TMEM_ACCB + as * COUT;
                if (issuer) {
#pragma unroll
                    for (int t = 0; t < 9; ++t) {
                        const int r = t / 3, s = t - 3 * r;
#pragma unroll
                        for (int j = 0; j < CMID / 16; ++j)
                            if (!BLK_DBG(8)) ptx::umma_bf16(d, ad + (r * PW + s) + j * (2 * PLANE_MID / 16), b_wb + (t * (CMID / 16) + j) * (2 * COUT), idesc_b, (t | j) ? 1u : 0u);
                    }
                    ptx::umma_commit_addr(bar0 + 8u * (BAR_MID_EMPTY + c));
                    ptx::umma_commit_addr(bar0 + 8u * (BAR_AB_FULL + as));
                }
                __syncwarp();
            }
        }
        PROF_STORE(4, lane == 0);
    } else if (warp < EPIA_WARPS) {
        // ---------------------------------------------------------------- epilogue A: 1x1 accumulators -> middle patch
        const int b = warp >> 2, quarter = warp & 3;      // TMEM lane quarter = warp % 4
        const int idx = 128 * b + 32 * quarter + lane;    // this lane's patch pixel (row-major in the 18 x 10 patch)
        const int py = idx / PW, px = idx - py * PW;
        const bool valid = idx < NPIX;
        const uint32_t mid_base = ptx::smem_u32(s_mid);
        const float2 alpha2 = make_float2(p.alpha_a, p.alpha_a);
        PROF_DECL
        for (int it = 0; it < my_tiles; ++it) {
            const int tile = blockIdx.x + it * gridDim.x;
            const int f = div_magic(tile, p.m_per_frame);
            const int rem = tile - f * per_frame;
            const int ty = div_magic(rem, p.m_tiles_x), tx = rem - ty * tiles_x;
            const int gy = ty * TH - 1 + py, gx = tx * TW - 1 + px;
            const bool inside = gy >= 0 && gy < p.h && gx >= 0 && gx < p.w;  // the 3x3's zero padding
            const int c = it & 1;
            PROF_WAIT(0, ptx::mbar_wait(&mid_empty[c], ((it >> 1) & 1) ^ 1));  // the 3x3 of the tile two back has read this patch
            PROF_WAIT(1, ptx::mbar_wait(&acca_full[b], it & 1));
            ptx::tc_fence_after();
            uint32_t acc[32];
            ptx::tmem_ld_32x32(tmem + b * 32 + (static_cast<uint32_t>(quarter * 32) << 16), acc);
            ptx::tmem_ld_wait();
            ptx::tc_fence_before();
            __syncwarp();
            if (lane == 0) ptx::mbar_arrive(acca_empty);
            if (!BLK_DBG(2)) {
                const uint32_t m = inside ? 0xFFFFFFFFu : 0u;
                const uint32_t dst = mid_base + c * MID_BYTES + idx * 16;
#pragma unroll
                for (int ch = 0; ch < NCH_MID; ++ch) {
                    uint32_t v[4];
#pragma unroll
                    for (int g = 0; g < 4; ++g) {
                        const float2 x = bias_act(acc[8 * ch + 2 * g], acc[8 * ch + 2 * g + 1], p.bias_a[8 * ch + 2 * g], p.bias_a[8 * ch + 2 * g + 1], alpha2);
                        v[g] = pack2(x.x, x.y) & m;
                    }
                    ptx::st_shared_v4_if(dst + ch * PLANE_MID, v[0], v[1], v[2], v[3], valid);
                }
            }
            ptx::fence_proxy_async();  // generic-proxy writes of the patch -> visible to the tensor core
            __syncwarp();
            if (lane == 0) ptx::mbar_arrive(&mid_full[c]);
        }
        PROF_STORE(8, warp == 0 && lane == 0);
    } else {
        // ---------------------------------------------------------------- epilogue B: 3x3 accumulators + x -> global memory
        const int quarter = warp & 3, group = (warp - EPIA_WARPS) >> 2;
        uint8_t* const stage = s_stage + (warp - EPIA_WARPS) * 4096;
        const uint32_t stage_u = ptx::smem_u32(stage);
        const uint32_t in_base = ptx::smem_u32(s_in);
        // this lane's output pixel (tile row 4q + lane / 8, column lane % 8) sits at patch pixel (row + 1, column + 1)
        const uint32_t res_off = ((4 * quarter + (lane >> 3) + 1) * PW + (lane & 7) + 1) * 16;
        const float2 alpha2 = make_float2(p.alpha_b, p.alpha_b);
        PROF_DECL
        ptx::grid_dep_wait();
        for (int it = group; it < my_tiles; it += 2) {
            const int as = it & 3, slot = it % IN_SLOTS;
            const int tile = blockIdx.x + it * gridDim.x;
            const int f = div_magic(tile, p.m_per_frame);
            const int rem = tile - f * per_frame;
            const int ty = div_magic(rem, p.m_tiles_x), tx = rem - ty * tiles_x;
            PROF_WAIT(0, ptx::mbar_wait(&accb_full[as], (it >> 2) & 1));
            ptx::tc_fence_after();
            const uint32_t taddr = tmem + TMEM_ACCB + as * COUT + (static_cast<uint32_t>(quarter * 32) << 16);
            const uint32_t buf = stage_u;
            if (lane == 0) PROF_WAIT(1, ptx::tma_store_wait_read<0>());  // this warp's previous stores (two tiles ago) have finished reading the buffer
            __syncwarp();
            // the x patch was written by the builders' cp.async: observe its barrier here too (long complete — the 1x1 ran on it —
            // but this warp's generic loads of the residual then have their own acquire on those writes)
            ptx::mbar_wait(&in_full[slot], (it / IN_SLOTS) & 1);
            const uint32_t res = in_base + slot * IN_SLOT_BYTES + res_off;
#pragma unroll
            for (int c0 = 0; c0 < COUT; c0 += 32) {
                uint32_t acc[32];
                ptx::tmem_ld_32x32(taddr + c0, acc);
                uint4 r[4];  // x, channels c0 .. c0 + 31 of this lane's pixel: four chunk planes
#pragma unroll
                for (int ch = 0; ch < 4; ++ch) r[ch] = ptx::ld_shared_v4(res + ((c0 >> 3) + ch) * PLANE_IN);
                ptx::tmem_ld_wait();
                if (c0 + 32 >= COUT) {  // accumulator drained: hand the stage back to the MMA warp
                    ptx::tc_fence_before();
                    __syncwarp();
                    if (lane == 0) ptx::mbar_arrive(&accb_empty[as]);
                }
                if (BLK_DBG(16)) continue;
                const uint32_t so = buf + (c0 >> 5) * 2048 + lane * 64;
#pragma unroll
                for (int ch = 0; ch < 4; ++ch) {
                    const uint32_t rr[4] = {r[ch].x, r[ch].y, r[ch].z, r[ch].w};
                    uint32_t v[4];
#pragma unroll
                    for (int g = 0; g < 4; ++g) {
                        const int col = 8 * ch + 2 * g;
                        float2 x = bias_act(acc[col], acc[col + 1], p.bias_b[c0 + col], p.bias_b[c0 + col + 1], alpha2);
                        // ONNX Add after LeakyRelu, in fp32: one rounding, of the sum
                        x = __fadd2_rn(x, make_float2(__uint_as_float(rr[g] << 16), __uint_as_float(rr[g] & 0xFFFF0000u)));
                        v[g] = pack2(x.x, x.y);
                    }
                    // 32 pixels x 64 B with the 64-byte swizzle (chunk c of row r at slot c ^ ((r >> 1) & 3)): a SWIZZLE_64B box
                    ptx::st_shared_v4(so + ((ch ^ ((lane >> 1) & 3)) << 4), v[0], v[1], v[2], v[3]);
                }
            }
            // the residual has been read (the loads above were consumed): this warp's share of the x patch is free
            __syncwarp();
            if (lane == 0) ptx::mbar_arrive(&in_empty[slot]);
            ptx::fence_proxy_async();
            __syncwarp();
            if (lane == 0 && !BLK_DBG(16)) {
#pragma unroll
                for (int c0 = 0; c0 < COUT; c0 += 32) ptx::tma_store_4d(&tm_out, stage + (c0 >> 5) * 2048, c0, tx * TW, ty * TH + 4 * quarter, f);  // clipped at the edges
                ptx::tma_store_commit();
            }
        }
        PROF_STORE(12, warp == EPIA_WARPS && lane == 0);
        if (lane == 0) ptx::tma_store_wait<0>();
    }
    ptx::tc_fence_before();
    __syncthreads();
    if (warp == MMA_WARP) {
        ptx::tc_fence_after();
        ptx::tmem_dealloc(tmem, TMEM_COLS);
    }
}

}  // namespace

bool conv_block_supported(const BlockDesc& d) {
    if (d.cin != CIN || d.cmid != CMID || d.cout != COUT) return false;
    if (d.act_a > 1 || d.act_b > 1) return false;  // LeakyReLU only (act 2, Mish, runs unfused)
    if (d.act_a && !(d.alpha_a >= 0.f && d.alpha_a <= 1.f)) return false;
    if (d.act_b && !(d.alpha_b >= 0.f && d.alpha_b <= 1.f)) return false;
    if (d.in_pitch % 8 || d.out_pitch % 8 || (reinterpret_cast<uintptr_t>(d.in) & 15) || (reinterpret_cast<uintptr_t>(d.out) & 15) ||
        (reinterpret_cast<uintptr_t>(d.wa) & 15) || (reinterpret_cast<uintptr_t>(d.wb) & 15))
        return false;
    if (d.h < 64 || d.w < 64) return false;  // worth it on large maps only
    const long long per_frame = 1LL * ((d.w + TW - 1) / TW) * ((d.h + TH - 1) / TH);
    return per_frame < (1 << 16) && d.n * per_frame < (1LL << 24);
}

int conv_block_prepare(const BlockDesc& d, int num_sms, BlockLaunch* L, char* err, size_t errlen) {
    memset(L, 0, sizeof(*L));
    if (!conv_block_supported(d)) { if (err && errlen) snprintf(err, errlen, "conv_block: unsupported layer pair"); return -1; }
    BlockParams& p = L->p;
    p.in = d.in; p.n = d.n; p.h = d.h; p.w = d.w; p.in_pitch = d.in_pitch;
    p.wa = d.wa; p.wb = d.wb;
    p.alpha_a = d.act_a ? d.alpha_a : 1.f;
    p.alpha_b = d.act_b ? d.alpha_b : 1.f;
    p.tiles_x = (d.w + TW - 1) / TW;
    p.per_frame = p.tiles_x * ((d.h + TH - 1) / TH);
    p.total = d.n * p.per_frame;
    const unsigned long long one40 = 1ULL << 40;
    p.m_per_frame = (one40 + p.per_frame - 1) / p.per_frame;
    p.m_tiles_x = (one40 + p.tiles_x - 1) / p.tiles_x;
    memcpy(p.bias_a, d.bias_a_host, sizeof(float) * CMID);
    memcpy(p.bias_b, d.bias_b_host, sizeof(float) * COUT);
    const unsigned long long dims[4] = {static_cast<unsigned long long>(COUT), static_cast<unsigned long long>(d.w),
                                        static_cast<unsigned long long>(d.h), static_cast<unsigned long long>(d.n)};
    const unsigned long long strides[3] = {2ULL * d.out_pitch, 2ULL * d.out_pitch * d.w, 2ULL * d.out_pitch * d.w * d.h};
    const unsigned box[4] = {32, TW, 4, 1};
    if (encode_tiled_bf16(&L->tm_out, d.out, 4, dims, strides, box, 2)) { if (err && errlen) snprintf(err, errlen, "conv_block: output tensor map encode failed"); return -1; }
    L->smem_bytes = SMEM_BYTES;
    L->grid = p.total < num_sms ? p.total : num_sms;
    L->flops = 2.0 * d.n * d.h * d.w * (1.0 * CMID * CIN + 1.0 * COUT * 9.0 * CMID);
    return 0;
}

int conv_block_init() {
    return cudaFuncSetAttribute(conv_block_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES) == cudaSuccess ? 0 : -1;
}

int conv_block_launch(const BlockLaunch& L, cudaStream_t stream) {
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
    return cudaLaunchKernelEx(&cfg, conv_block_kernel, L.tm_out, L.p) == cudaSuccess ? 0 : -1;
}

}  // namespace fd
