// conv_stem.cu — the network stem in ONE kernel: u8 frames -> /255 -> conv 3x3 (3 -> 32, stride 1) -> LeakyReLU ->
// conv 3x3 (32 -> 64, stride 2) -> LeakyReLU -> bf16 NHWC.
//
// Why: as two kernels the first convolution writes 709 MB per 64 frames of 416x416 (64 B per pixel) that the second reads
// straight back: 0.45 ms of a 4.4 ms forward pass for 3 % of its arithmetic, both kernels far from any tensor-core
// limit.  Fused, the 32-channel activation only ever exists as the halo patch of the second convolution's tile, in shared
// memory, in exactly the layout conv_halo.cu's stride-2 form reads its nine taps from.  The price is recomputing the first
// convolution on the patch overlap (33 x 17 conv1 pixels for 32 x 16 owned ones: 1.1x) and on the padding rows of the MMA
// blocks below; the kernel is bound by MMA issue (~45 cycles per tcgen05.mma whatever its N) and by its epilogues'
// instruction issue, not by HBM.  Measured at batch 64, 416x416: 224 us against 488 us for conv0_ws_kernel +
// conv_halo_kernel<32, 2> (dev/test_stem.cu; per-role cycle accounting in profiles/r02q_stem_role_cycles.txt).
//
// Per tile of 16 x 8 output pixels of the second convolution (M = 128 rows of its MMA):
//   builders   gather the 35 x 19 u8 halo patch of the frame, convert to bf16(float32(k / 255)) and store it with
//              8 bytes per pixel (R, G, B, 0).  In the un-swizzled K-major operand layout a core matrix is 8 rows x 16 B,
//              rows 16 B apart, the next K chunk LBO bytes further: with LBO = 16 B, row e of a group is the pixel pair
//              (2e, 2e+1) and its second K chunk the pair (2e+2, 2e+3) — ONE K = 16 MMA covers the taps 0..3 of a filter
//              row (tap 3 meets zero weights) for the output pixels 0, 2, 4, ... of the group: the operand addressing does
//              the im2col AND the column-parity split the stride-2 consumer wants.  Odd output columns need the same
//              bytes shifted by one pixel, so every patch row is stored three times, as three 160-byte "regions":
//              E0 (pixels 0..18 -> outputs 0, 2, .., 14), E1 (pixels 16..18 -> output 16), O (pixels 1..18 -> outputs
//              1, 3, .., 15).  Regions are 160 bytes apart throughout, so ANY 16 consecutive regions are one MMA block
//              (SBO = 160): 33 rows x 3 regions = 99 groups = 7 blocks of 3 MMAs (one per filter row; the next patch
//              row is 3 regions further).
//   MMA warp   issues conv1 of tile t+1 (21 MMAs, N = 32, into 7 TMEM accumulators) and then conv2 of tile t (18 MMAs,
//              N = 64, exactly conv_halo.cu's stride-2 loop), so the tensor pipe has work while tile t's patch is built.
//   epilogue 1 (16 warps) drains the conv1 accumulators: bias, LeakyReLU, bf16, zero outside the image (the second
//              convolution's padding is zero in conv1's OUTPUT domain), and stores each pixel's four 16-byte channel
//              chunks into the chunk planes / parity sub-planes of the conv2 patch (conv_halo.cu's layout).
//   epilogue 2 (4 warps) drains conv2: bias, LeakyReLU, bf16 rows staged with the 64-byte swizzle, TMA stores.
// Replaces the first two Conv+BatchNormalization+LeakyRelu groups of YOLOv3 and the `/255` in front of them
// (reference server/detector.py:133-135).
#include "conv_stem.h"

#include <stdio.h>
#include <string.h>

#include "conv_tc.h"
#include "ptx.cuh"

namespace fd {

namespace {

constexpr int TW = 8, TH = 16;                 // conv2 output tile: 16 rows x 8 columns = the 128 rows of one MMA
constexpr int C1 = 32, C2 = 64;
constexpr int EPI2_WARPS = 4;                  // warps 0..3
constexpr int EPI1_GROUPS = 4;                 // warps 4..19: group g drains blocks g, g + 4
constexpr int EPI1_WARPS = 4 * EPI1_GROUPS;
constexpr int MMA_WARP = EPI2_WARPS + EPI1_WARPS;  // warp 20
constexpr int BUILD_WARPS = 3;                 // warps 21..23 (24 warps: 80 registers per thread)
constexpr int THREADS = (MMA_WARP + 1 + BUILD_WARPS) * 32;
// conv1 output patch of a tile, split into (row parity, column parity) sub-planes per 8-channel chunk plane
constexpr int PH = 2 * TH + 1, PW = 2 * TW + 1;           // 33 x 17
constexpr int SPH = TH + 1, SPW = TW + 1;                 // 17 x 9
constexpr int SUB = SPH * SPW;                            // positions of one sub-plane
constexpr int NCH = C1 / 8;                               // 16-byte channel chunks per conv1 pixel
constexpr int PLANE_BYTES = ((4 * SUB * 16 + 127) / 128) * 128;
constexpr int C1_BYTES = NCH * PLANE_BYTES;
constexpr int C1_SLOTS = 2;
// input patch: 35 x 19 pixels, three 160-byte regions per row
constexpr int IH = PH + 2, IW = PW + 2;
constexpr int REGION = 160;
constexpr int ROW_BYTES = 3 * REGION;
constexpr int BLOCKS1 = (PH * 3 + 15) / 16;               // 7 MMA blocks of 16 regions
constexpr int IN_SLOT_BYTES = ((IH * ROW_BYTES + 127) / 128) * 128;
constexpr int IN_SLOTS = 4;
// the last block's padding groups (and the two filter rows below them) read past the slot: into the next slot or this tail,
// both of which only ever hold zeros or LUT values (finite: 0 x garbage must not be NaN)
constexpr int IN_TAIL = (((16 * BLOCKS1 + 6) * REGION + 16 - IH * ROW_BYTES + 127) / 128) * 128;
constexpr int A1_FULLS = (BLOCKS1 + 1) / 2;               // the MMA warp commits after every second conv1 block (sync instructions are its bottleneck)
constexpr int ACC2S = 4;
constexpr int TMEM_ACC2 = 256, TMEM_COLS = 512;           // conv1 accumulators: columns [0, 7 * 32); conv2: [256, 256 + 4 * 64)
constexpr int W2_BYTES = 9 * NCH * C2 * 16;
constexpr int OFF_W1 = 2048, OFF_STAGE = 6144;
constexpr int OFF_W2 = OFF_STAGE + EPI2_WARPS * 2 * 4096;
constexpr int OFF_C1 = OFF_W2 + W2_BYTES;
constexpr int OFF_IN = OFF_C1 + C1_SLOTS * C1_BYTES;
constexpr int SMEM_BYTES = OFF_IN + IN_SLOTS * IN_SLOT_BYTES + IN_TAIL + 1024;  // + alignment slack
static_assert(OFF_W2 % 1024 == 0 && OFF_C1 % 128 == 0 && OFF_IN % 128 == 0, "operand regions must stay 128-byte aligned");
static_assert(BLOCKS1 * 32 <= TMEM_ACC2 && TMEM_ACC2 + ACC2S * C2 <= TMEM_COLS, "TMEM columns");
static_assert(SMEM_BYTES <= 227 * 1024, "shared memory");
static_assert(6 * 32 * 16 <= OFF_STAGE - OFF_W1, "conv1 filter tile");

__device__ __forceinline__ int div_magic(int x, unsigned long long m) {
    return static_cast<int>((static_cast<unsigned long long>(x) * m) >> 40);
}
__device__ __forceinline__ uint32_t pack2(float a, float b) {
    __nv_bfloat162 v = __floats2bfloat162_rn(a, b);
    return *reinterpret_cast<uint32_t*>(&v);
}
// bf16(float32(k / 255.0)), the reference's normalisation rounded once more for the MMA, without a table: (2^23 + k) as a
// float is the bit pattern 0x4B000000 | k, and fma(2^23 + k, c, -2^23 c) = round(k c) with c = float32(1 / 255); the bf16
// rounding of that equals the bf16 rounding of float32(k / 255.0) for all 256 bytes (checked exhaustively:
// tests/test_native_cpu.py::test_stem_normalisation_formula)
__device__ __forceinline__ float norm_bits(uint32_t bits_2p23_plus_k) {
    constexpr float c = 1.0f / 255.0f;
    return fmaf(__uint_as_float(bits_2p23_plus_k), c, -8388608.0f * c);
}
// un-swizzled K-major shared-memory descriptor: start, LBO (K chunk stride), SBO (8-row group stride), all bytes
__device__ __forceinline__ uint64_t desc_kmajor(uint32_t addr, uint32_t lbo, uint32_t sbo) {
    return static_cast<uint64_t>((addr >> 4) & 0x3FFF) | (static_cast<uint64_t>((lbo >> 4) & 0x3FFF) << 16) |
           (static_cast<uint64_t>((sbo >> 4) & 0x3FFF) << 32) | (static_cast<uint64_t>(1) << 46);
}
// bias + LeakyReLU as max(x, alpha x) (alpha in [0, 1]; 1 = linear) on 32 fp32 accumulator columns -> 16 bf16 pairs
__device__ __forceinline__ void finish32(const uint32_t (&acc)[32], const float* bias, float alpha, uint32_t (&pk)[16]) {
    const float2 a2 = make_float2(alpha, alpha);
#pragma unroll
    for (int g = 0; g < 16; ++g) {
        float2 x = __fadd2_rn(make_float2(__uint_as_float(acc[2 * g]), __uint_as_float(acc[2 * g + 1])), make_float2(bias[2 * g], bias[2 * g + 1]));
        const float2 m = __fmul2_rn(x, a2);
        pk[g] = pack2(fmaxf(x.x, m.x), fmaxf(x.y, m.y));
    }
}

// developer switches (harness build only; the shipped kernel carries none of these branches)
#ifdef FASTDET_DEV
#define STEM_DBG(bit) ((p.debug & (bit)) != 0)
// per-role cycle accounting: PROF_WAIT(slot, stmt) adds the cycles `stmt` (a barrier wait) took to prof_acc[slot]
#define PROF_DECL long long prof_acc[4] = {0, 0, 0, 0}; const long long prof_t0 = clock64();
#define PROF_WAIT(slot, stmt) do { const long long t_ = clock64(); stmt; prof_acc[slot] += clock64() - t_; } while (0)
#define PROF_MARK(slot) const long long tm_##slot = clock64();
#define PROF_MARK_END(slot) prof_acc[slot] += clock64() - tm_##slot;
#define PROF_STORE(base, who) do { if (p.prof && (who)) { long long* o_ = p.prof + blockIdx.x * 16 + (base); o_[0] = clock64() - prof_t0; \
        o_[1] = prof_acc[0]; o_[2] = prof_acc[1]; o_[3] = prof_acc[2]; } } while (0)
#else
#define STEM_DBG(bit) false
#define PROF_DECL
#define PROF_WAIT(slot, stmt) stmt
#define PROF_MARK(slot)
#define PROF_MARK_END(slot)
#define PROF_STORE(base, who)
#endif

#define STEM_WAIT(addr, parity) ptx::mbar_wait_addr(addr, parity)

__global__ void __launch_bounds__(THREADS, 1)
conv_stem_kernel(const __grid_constant__ CUtensorMap tm_out, const __grid_constant__ StemParams p) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    uint64_t* in_full = reinterpret_cast<uint64_t*>(smem);
    uint64_t* in_empty = in_full + IN_SLOTS;
    uint64_t* acc1_full = in_empty + IN_SLOTS;      // one per pair of blocks
    uint64_t* acc1_empty = acc1_full + A1_FULLS;   // one barrier for the whole accumulator set
    uint64_t* c1_full = acc1_empty + 1;
    uint64_t* c1_empty = c1_full + C1_SLOTS;
    uint64_t* acc2_full = c1_empty + C1_SLOTS;
    uint64_t* acc2_empty = acc2_full + ACC2S;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(acc2_empty + ACC2S);
    uint8_t* s_w1 = smem + OFF_W1;
    uint8_t* s_stage = smem + OFF_STAGE;
    uint8_t* s_w2 = smem + OFF_W2;
    uint8_t* s_c1 = smem + OFF_C1;
    uint8_t* s_in = smem + OFF_IN;

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    // ---- constants of the layer pair (before any dependency wait)
    // conv1 filters: [filter row r][K chunk kc][32 filters][16 B] = taps (2kc, 2kc+1) x (R, G, B, 0); tap 3 is zero
    for (int i = tid; i < 6 * 32; i += THREADS) {
        const int f = i & 31, rk = i >> 5, r = rk >> 1, kc = rk & 1;
        float w[2][3];
#pragma unroll
        for (int t = 0; t < 2; ++t) {
            const int sx = 2 * kc + t;
#pragma unroll
            for (int ch = 0; ch < 3; ++ch) w[t][ch] = sx < 3 ? __ldg(p.w1 + ((r * 3 + sx) * 3 + ch) * C1 + f) : 0.f;
        }
        *reinterpret_cast<uint4*>(s_w1 + i * 16) = make_uint4(pack2(w[0][0], w[0][1]), pack2(w[0][2], 0.f), pack2(w[1][0], w[1][1]), pack2(w[1][2], 0.f));
    }
    // conv2 filters: global [64][9 * 32] -> [K chunk = tap * 4 + channel chunk][64 filters][16 B]
    for (int i = tid; i < 9 * NCH * C2; i += THREADS) {
        const int kc = i / C2, f = i - kc * C2;
        *reinterpret_cast<uint4*>(s_w2 + i * 16) = __ldg(reinterpret_cast<const uint4*>(p.w2 + static_cast<size_t>(f) * 9 * C1 + kc * 8));
    }
    for (int i = tid; i < (C1_SLOTS * C1_BYTES + IN_SLOTS * IN_SLOT_BYTES + IN_TAIL) / 16; i += THREADS)
        reinterpret_cast<uint4*>(s_c1)[i] = make_uint4(0u, 0u, 0u, 0u);
    if (tid == 0) {
        for (int i = 0; i < IN_SLOTS; ++i) { ptx::mbar_init(&in_full[i], BUILD_WARPS); ptx::mbar_init(&in_empty[i], 1); }
        for (int i = 0; i < A1_FULLS; ++i) ptx::mbar_init(&acc1_full[i], 1);
        ptx::mbar_init(acc1_empty, EPI1_WARPS);
        for (int i = 0; i < C1_SLOTS; ++i) { ptx::mbar_init(&c1_full[i], EPI1_WARPS); ptx::mbar_init(&c1_empty[i], 1); }
        for (int i = 0; i < ACC2S; ++i) { ptx::mbar_init(&acc2_full[i], 1); ptx::mbar_init(&acc2_empty[i], 4); }
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
        // ---------------------------------------------------------------- builders: u8 halo patch -> bf16, 8 B per pixel, three regions
        // The warps share every tile.  An item is 4 consecutive pixels of a patch row = 12 bytes, fetched as the 4 aligned
        // words around them: the row's first byte sits at (48 tx - 6) in a row of 3w bytes, i.e. always 2 bytes past a word
        // boundary when w % 4 == 0 (checked on the host), so the bytes of the 4 pixels are at fixed positions of the 4 words
        // (35 rows x 5 items = 175 items, 2 per lane: 8 word loads per lane and tile instead of 21 byte loads).  The words of
        // the next two tiles are in registers while the current one is converted (the loads come from DRAM / L2).
        const int ltid = (warp - MMA_WARP - 1) * 32 + lane;
        const uint32_t in_base = ptx::smem_u32(s_in);
        PROF_DECL
        constexpr int SEGS = (IW + 3) / 4, ITEMS = IH * SEGS;
        constexpr int IPL = (ITEMS + BUILD_WARPS * 32 - 1) / (BUILD_WARPS * 32);
        uint32_t irs[IPL];  // (patch row << 8) | segment, 0xFFFF: none
#pragma unroll
        for (int k = 0; k < IPL; ++k) {
            const int q = ltid + BUILD_WARPS * 32 * k;
            const int row = q / SEGS, seg = q - row * SEGS;
            irs[k] = q < ITEMS ? static_cast<uint32_t>((row << 8) | seg) : 0xFFFFu;
        }
        const uint8_t* const f_begin = p.frames;
        const uint8_t* const f_end = p.frames + static_cast<long long>(p.n) * p.h * p.w * 3;
        struct Set { uint32_t w[4 * IPL]; uint32_t rows; int x0; };  // rows: bit k = item k's row is inside the frame
        Set set_a, set_b;
#pragma unroll
        for (int i = 0; i < 4 * IPL; ++i) set_a.w[i] = set_b.w[i] = 0;
        set_a.rows = set_b.rows = 0; set_a.x0 = set_b.x0 = 0;
        auto fetch = [&](int it, Set& S) {  // no arithmetic on the words here: it would wait for the loads
            const int tile = blockIdx.x + it * gridDim.x;
            const int f = div_magic(tile, p.m_per_frame);
            const int rem = tile - f * per_frame;
            const int ty = div_magic(rem, p.m_tiles_x), tx = rem - ty * tiles_x;
            const int y0 = ty * (2 * TH) - 2, x0 = tx * (2 * TW) - 2;
            // word that holds the two bytes in front of patch pixel (0, 0) (may lie before the frame: every word is checked)
            const uint8_t* origin = p.frames + (static_cast<long long>(f) * p.h * p.w + static_cast<long long>(y0) * p.w + x0) * 3 - 2;
            S.rows = 0;
            S.x0 = x0;
#pragma unroll
            for (int k = 0; k < IPL; ++k) {
                const int row = static_cast<int>(irs[k] >> 8), seg = static_cast<int>(irs[k] & 255);
                const int gy = y0 + row;
                if (irs[k] != 0xFFFFu && gy >= 0 && gy < p.h && !STEM_DBG(1 | 64)) {  // rows outside: zero padding of the normalised input
                    const uint8_t* sp = origin + static_cast<long long>(row) * (p.w * 3) + 12 * seg;
                    S.rows |= 1u << k;
#pragma unroll
                    for (int j = 0; j < 4; ++j)
                        if (sp + 4 * j >= f_begin && sp + 4 * j + 4 <= f_end) S.w[4 * k + j] = __ldg(reinterpret_cast<const uint32_t*>(sp) + j);
                }
            }
        };
        // (2^23 + byte) as a float, straight from byte `n` of a word: PRMT picks {byte, 0, 0, 0x4B}
        auto norm_byte = [](uint32_t word, uint32_t sel) { return norm_bits(__byte_perm(word, 0x4B000000u, sel)); };
        auto publish = [&](int it, const Set& S) {
            const int slot = it % IN_SLOTS;
            PROF_WAIT(0, STEM_WAIT(ptx::smem_u32(&in_empty[slot]), ((it / IN_SLOTS) & 1) ^ 1));
            const uint32_t dst = in_base + slot * IN_SLOT_BYTES;
            PROF_MARK(1);
#pragma unroll
            for (int k = 0; k < IPL; ++k) {  // (branch-free: predicated shared-space stores)
                const uint32_t* w = &S.w[4 * k];
                const uint32_t seg = irs[k] & 255u;
                const bool item = irs[k] != 0xFFFFu && !STEM_DBG(1);
                const bool row_in = (S.rows >> k) & 1u;
                const int gx = S.x0 + 4 * static_cast<int>(seg);
                // pixel j = bytes 2 + 3j .. 4 + 3j of the 16 bytes: (R, G, B, 0) as two bf16 pairs, zero outside the frame
                uint32_t v[8];
                v[0] = pack2(norm_byte(w[0], 0x7442u), norm_byte(w[0], 0x7443u)); v[1] = pack2(norm_byte(w[1], 0x7440u), 0.f);
                v[2] = pack2(norm_byte(w[1], 0x7441u), norm_byte(w[1], 0x7442u)); v[3] = pack2(norm_byte(w[1], 0x7443u), 0.f);
                v[4] = pack2(norm_byte(w[2], 0x7440u), norm_byte(w[2], 0x7441u)); v[5] = pack2(norm_byte(w[2], 0x7442u), 0.f);
                v[6] = pack2(norm_byte(w[2], 0x7443u), norm_byte(w[3], 0x7440u)); v[7] = pack2(norm_byte(w[3], 0x7441u), 0.f);
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const uint32_t m = (row_in && gx + j >= 0 && gx + j < p.w) ? 0xFFFFFFFFu : 0u;
                    v[2 * j] &= m;
                    v[2 * j + 1] &= m;
                }
                const uint32_t d0 = dst + (irs[k] >> 8) * ROW_BYTES + seg * 32;
                // E0: pixel px at slot px
                ptx::st_shared_v4_if(d0, v[0], v[1], v[2], v[3], item);
                ptx::st_shared_v4_if(d0 + 16, v[4], v[5], v[6], v[7], item);
                // E1: pixels 16, 17, 18 at slots 0, 1, 2 (segment 4 only)
                ptx::st_shared_v4_if(d0 + (REGION - 128), v[0], v[1], v[2], v[3], item && seg == 4);
                ptx::st_shared_v2_if(d0 + (REGION - 128) + 16, v[4], v[5], item && seg == 4);
                // O: pixel px at slot px - 1
                ptx::st_shared_v2_if(d0 + (2 * REGION - 8), v[0], v[1], item && seg != 0);
                ptx::st_shared_v4_if(d0 + 2 * REGION, v[2], v[3], v[4], v[5], item);
                ptx::st_shared_v2_if(d0 + 2 * REGION + 16, v[6], v[7], item);
            }
            PROF_MARK_END(1);
        };
        // (after the next tile's loads have been issued: the fence waits for the stores above to drain)
        auto signal = [&](int it) {
            PROF_MARK(2);
            ptx::fence_proxy_async();  // generic-proxy writes of the patch -> visible to the tensor core
            __syncwarp();
            if (lane == 0) ptx::mbar_arrive(&in_full[it % IN_SLOTS]);
            PROF_MARK_END(2);
        };
        ptx::grid_dep_wait();
        if (0 < my_tiles) fetch(0, set_a);
        if (1 < my_tiles) fetch(1, set_b);
        for (int it = 0; it < my_tiles; it += 2) {
            publish(it, set_a);
            if (it + 2 < my_tiles) fetch(it + 2, set_a);
            signal(it);
            if (it + 1 >= my_tiles) break;
            publish(it + 1, set_b);
            if (it + 3 < my_tiles) fetch(it + 3, set_b);
            signal(it + 1);
        }
        PROF_STORE(0, ltid == 0);
    } else if (warp == MMA_WARP) {
        // ---------------------------------------------------------------- MMA issuer (all operands warp-uniform)
        const uint32_t idesc1 = ptx::make_idesc_bf16_f32(128, C1), idesc2 = ptx::make_idesc_bf16_f32(128, C2);
        const uint32_t bar0 = __shfl_sync(0xffffffffu, ptx::smem_u32(in_full), 0);  // all barriers: 8-byte steps from in_full
        const uint32_t tmem_u = __shfl_sync(0xffffffffu, tmem, 0);
        const uint64_t a1 = desc_kmajor(__shfl_sync(0xffffffffu, ptx::smem_u32(s_in), 0), 16, REGION);
        const uint64_t b1 = desc_kmajor(__shfl_sync(0xffffffffu, ptx::smem_u32(s_w1), 0), 512, 128);
        const uint64_t a2 = desc_kmajor(__shfl_sync(0xffffffffu, ptx::smem_u32(s_c1), 0), PLANE_BYTES, SPW * 16);
        const uint64_t b2 = desc_kmajor(__shfl_sync(0xffffffffu, ptx::smem_u32(s_w2), 0), C2 * 16, 128);
        constexpr uint32_t BAR_IN_EMPTY = IN_SLOTS, BAR_A1_FULL = 2 * IN_SLOTS, BAR_A1_EMPTY = BAR_A1_FULL + A1_FULLS,
                           BAR_C1_FULL = BAR_A1_EMPTY + 1, BAR_C1_EMPTY = BAR_C1_FULL + C1_SLOTS,
                           BAR_A2_FULL = BAR_C1_EMPTY + C1_SLOTS, BAR_A2_EMPTY = BAR_A2_FULL + ACC2S;
        const bool issuer = ptx::elect_one();
        PROF_DECL
        for (int step = 0; step <= my_tiles; ++step) {
            if (step < my_tiles) {
                // conv1 of tile `step`: 7 blocks x 3 MMAs (one per filter row: the next patch row is 3 regions further)
                const int it = step;
                const uint32_t slot = it % IN_SLOTS;
                PROF_WAIT(0, STEM_WAIT(bar0 + 8u * slot, (it / IN_SLOTS) & 1));  // in_full
                ptx::tc_fence_after();
                const uint64_t ad = a1 + slot * (IN_SLOT_BYTES / 16);
                PROF_WAIT(1, STEM_WAIT(bar0 + 8u * BAR_A1_EMPTY, (it & 1) ^ 1));  // the previous tile's accumulators have been drained
                ptx::tc_fence_after();
                if (issuer) {
#pragma unroll
                    for (int b = 0; b < BLOCKS1; ++b) {
#pragma unroll
                        for (int r = 0; r < 3; ++r)
                            if (!STEM_DBG(4)) ptx::umma_bf16(tmem_u + b * 32, ad + (16 * b + 3 * r) * (REGION / 16), b1 + r * (1024 / 16), idesc1, r ? 1u : 0u);
                        if ((b & 1) || b == BLOCKS1 - 1) ptx::umma_commit_addr(bar0 + 8u * (BAR_A1_FULL + (b >> 1)));
                    }
                    ptx::umma_commit_addr(bar0 + 8u * (BAR_IN_EMPTY + slot));
                }
                __syncwarp();
            }
            if (step >= 1) {
                // conv2 of tile `step - 1`: its conv1 patch has been finished by the epilogue-1 warps meanwhile
                const int it = step - 1;
                const uint32_t c = it & 1, as = it & 3;
                PROF_WAIT(2, STEM_WAIT(bar0 + 8u * (BAR_A2_EMPTY + as), ((it >> 2) & 1) ^ 1));
                PROF_WAIT(2, STEM_WAIT(bar0 + 8u * (BAR_C1_FULL + c), (it >> 1) & 1));  // (the writers fenced: generic -> async proxy)
                ptx::tc_fence_after();
                const uint64_t ad = a2 + c * (C1_BYTES / 16);
                const uint32_t d = tmem_u + TMEM_ACC2 + as * C2;
                if (issuer) {
#pragma unroll
                    for (int t = 0; t < 9; ++t) {
                        const int r = t / 3, s = t - 3 * r;
                        const int start = ((r & 1) * 2 + (s & 1)) * SUB + (r >> 1) * SPW + (s >> 1);
#pragma unroll
                        for (int j = 0; j < C1 / 16; ++j)
                            if (!STEM_DBG(8)) ptx::umma_bf16(d, ad + start + j * (2 * PLANE_BYTES / 16), b2 + (t * (C1 / 16) + j) * (2 * C2), idesc2, (t | j) ? 1u : 0u);
                    }
                    ptx::umma_commit_addr(bar0 + 8u * (BAR_C1_EMPTY + c));
                    ptx::umma_commit_addr(bar0 + 8u * (BAR_A2_FULL + as));
                }
                __syncwarp();
            }
        }
        PROF_STORE(4, lane == 0);
    } else if (warp >= EPI2_WARPS) {
        // ---------------------------------------------------------------- epilogue 1: conv1 accumulators -> conv2 patch
        const int group = (warp - EPI2_WARPS) >> 2, quarter = warp & 3;  // TMEM lane quarter = warp % 4
        const int gi = 4 * quarter + (lane >> 3), e = lane & 7;           // this lane's group within a block, pixel within the group
        const uint32_t c1_base = ptx::smem_u32(s_c1);
        PROF_DECL
        for (int it = 0; it < my_tiles; ++it) {
            const int tile = blockIdx.x + it * gridDim.x;
            const int f = div_magic(tile, p.m_per_frame);
            const int rem = tile - f * per_frame;
            const int ty = div_magic(rem, p.m_tiles_x), tx = rem - ty * tiles_x;
            const int cy0 = ty * (2 * TH) - 1, cx0 = tx * (2 * TW) - 1;   // conv1 pixel of patch position (0, 0)
            const bool border = cy0 < 0 || cx0 < 0 || cy0 + PH > p.h || cx0 + PW > p.w;  // (warp-uniform)
            const int c = it & 1;
            const uint32_t c1 = c1_base + c * C1_BYTES;
            PROF_WAIT(0, STEM_WAIT(ptx::smem_u32(&c1_empty[c]), ((it >> 1) & 1) ^ 1));  // conv2 of the tile two back has read this patch
            for (int b = group; b < BLOCKS1; b += EPI1_GROUPS) {
                const int G = 16 * b + gi;          // region index = 3 * patch row + {E0, E1, O}
                const int j = (G * 43) >> 7;        // G / 3 for G < 128
                const int k = G - 3 * j;
                const int i = k == 0 ? 2 * e : (k == 1 ? 16 + 2 * e : 2 * e + 1);
                const bool valid = j < PH && i < PW;
                PROF_WAIT(1, STEM_WAIT(ptx::smem_u32(&acc1_full[b >> 1]), it & 1));
                ptx::tc_fence_after();
                uint32_t acc[32];
                ptx::tmem_ld_32x32(tmem + b * 32 + (static_cast<uint32_t>(quarter * 32) << 16), acc);
                ptx::tmem_ld_wait();
                if (b + EPI1_GROUPS >= BLOCKS1) {  // this warp's last block of the tile: its share of the accumulators is drained
                    ptx::tc_fence_before();
                    __syncwarp();
                    if (lane == 0) ptx::mbar_arrive(acc1_empty);
                }
                if (STEM_DBG(2)) continue;
                uint32_t pk[16];
                finish32(acc, p.bias1, p.alpha1, pk);
                if (border) {
                    const int cy = cy0 + j, cx = cx0 + i;
                    if (cy < 0 || cy >= p.h || cx < 0 || cx >= p.w) {  // conv2's zero padding
#pragma unroll
                        for (int g = 0; g < 16; ++g) pk[g] = 0u;
                    }
                }
                {
                    const uint32_t dst = c1 + (((j & 1) * 2 + (i & 1)) * SUB + (j >> 1) * SPW + (i >> 1)) * 16;
#pragma unroll
                    for (int ch = 0; ch < NCH; ++ch)
                        ptx::st_shared_v4_if(dst + ch * PLANE_BYTES, pk[4 * ch], pk[4 * ch + 1], pk[4 * ch + 2], pk[4 * ch + 3], valid && !STEM_DBG(32));
                }
            }
            ptx::fence_proxy_async();  // generic-proxy writes of the patch -> visible to the tensor core
            __syncwarp();
            if (lane == 0) ptx::mbar_arrive(&c1_full[c]);
        }
        PROF_STORE(8, warp == EPI2_WARPS && lane == 0);
    } else {
        // ---------------------------------------------------------------- epilogue 2: conv2 accumulators -> global memory
        const int quarter = warp;
        uint8_t* stage = s_stage + warp * 8192;
        const uint32_t stage_u = ptx::smem_u32(stage);
        ptx::grid_dep_wait();
        PROF_DECL
        for (int it = 0; it < my_tiles; ++it) {
            const int as = it & 3;
            const int tile = blockIdx.x + it * gridDim.x;
            const int f = div_magic(tile, p.m_per_frame);
            const int rem = tile - f * per_frame;
            const int ty = div_magic(rem, p.m_tiles_x), tx = rem - ty * tiles_x;
            PROF_WAIT(0, STEM_WAIT(ptx::smem_u32(&acc2_full[as]), (it >> 2) & 1));
            ptx::tc_fence_after();
            const uint32_t taddr = tmem + TMEM_ACC2 + as * C2 + (static_cast<uint32_t>(quarter * 32) << 16);
            uint8_t* buf = stage + (it & 1) * 4096;
            if (lane == 0) PROF_WAIT(1, ptx::tma_store_wait_read<1>());  // the stores of two tiles ago have finished reading this buffer
            __syncwarp();
#pragma unroll
            for (int c0 = 0; c0 < C2; c0 += 32) {
                uint32_t acc[32];
                ptx::tmem_ld_32x32(taddr + c0, acc);
                ptx::tmem_ld_wait();
                if (c0 + 32 >= C2) {  // accumulator drained: hand the stage back to the MMA warp
                    ptx::tc_fence_before();
                    __syncwarp();
                    if (lane == 0) ptx::mbar_arrive(&acc2_empty[as]);
                }
                if (STEM_DBG(16)) continue;
                uint32_t pk[16];
                finish32(acc, p.bias2 + c0, p.alpha2, pk);
                // 32 pixels x 64 B with the 64-byte swizzle (chunk c of row r at slot c ^ ((r >> 1) & 3)): a SWIZZLE_64B box
                const uint32_t so = stage_u + (it & 1) * 4096 + (c0 >> 5) * 2048 + lane * 64;
#pragma unroll
                for (int ch = 0; ch < 4; ++ch)
                    ptx::st_shared_v4(so + ((ch ^ ((lane >> 1) & 3)) << 4), pk[4 * ch], pk[4 * ch + 1], pk[4 * ch + 2], pk[4 * ch + 3]);
            }
            ptx::fence_proxy_async();
            __syncwarp();
            if (lane == 0 && !STEM_DBG(16)) {
#pragma unroll
                for (int c0 = 0; c0 < C2; c0 += 32) ptx::tma_store_4d(&tm_out, buf + (c0 >> 5) * 2048, c0, tx * TW, ty * TH + 4 * quarter, f);  // clipped at the edges
                ptx::tma_store_commit();
            }
        }
        PROF_STORE(12, warp == 0 && lane == 0);
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

bool conv_stem_supported(const StemDesc& d) {
    if (d.c1 != C1 || d.c2 != C2 || d.pad_hi2 < 0 || d.pad_hi2 > 1) return false;
    if (d.act1 && !(d.alpha1 >= 0.f && d.alpha1 <= 1.f)) return false;
    if (d.act2 && !(d.alpha2 >= 0.f && d.alpha2 <= 1.f)) return false;
    if (d.out_pitch % 8 || (reinterpret_cast<uintptr_t>(d.out) & 15) || (reinterpret_cast<uintptr_t>(d.w2) & 15)) return false;
    if (d.w % 4 || (reinterpret_cast<uintptr_t>(d.frames) & 3)) return false;  // the builders read the frame rows as aligned words
    const int ho = (d.h + 1 + d.pad_hi2 - 3) / 2 + 1, wo = (d.w + 1 + d.pad_hi2 - 3) / 2 + 1;
    if (ho < 64 || wo < 64) return false;  // worth it on large maps only
    const long long per_frame = 1LL * ((wo + TW - 1) / TW) * ((ho + TH - 1) / TH);
    return per_frame < (1 << 16) && d.n * per_frame < (1LL << 24) && 1LL * d.h * d.w * 3 < (1LL << 30);
}

int conv_stem_prepare(const StemDesc& d, int num_sms, StemLaunch* L, char* err, size_t errlen) {
    memset(L, 0, sizeof(*L));
    if (!conv_stem_supported(d)) { if (err && errlen) snprintf(err, errlen, "conv_stem: unsupported layer pair"); return -1; }
    StemParams& p = L->p;
    p.frames = d.frames; p.n = d.n; p.h = d.h; p.w = d.w;
    p.ho = (d.h + 1 + d.pad_hi2 - 3) / 2 + 1;
    p.wo = (d.w + 1 + d.pad_hi2 - 3) / 2 + 1;
    p.w1 = d.w1; p.w2 = d.w2;
    p.alpha1 = d.act1 ? d.alpha1 : 1.f;
    p.alpha2 = d.act2 ? d.alpha2 : 1.f;
    p.tiles_x = (p.wo + TW - 1) / TW;
    p.per_frame = p.tiles_x * ((p.ho + TH - 1) / TH);
    p.total = d.n * p.per_frame;
    const unsigned long long one40 = 1ULL << 40;
    p.m_per_frame = (one40 + p.per_frame - 1) / p.per_frame;
    p.m_tiles_x = (one40 + p.tiles_x - 1) / p.tiles_x;
    memcpy(p.bias1, d.bias1_host, sizeof(float) * C1);
    memcpy(p.bias2, d.bias2_host, sizeof(float) * C2);
    const unsigned long long dims[4] = {static_cast<unsigned long long>(C2), static_cast<unsigned long long>(p.wo),
                                        static_cast<unsigned long long>(p.ho), static_cast<unsigned long long>(d.n)};
    const unsigned long long strides[3] = {2ULL * d.out_pitch, 2ULL * d.out_pitch * p.wo, 2ULL * d.out_pitch * p.wo * p.ho};
    const unsigned box[4] = {32, TW, 4, 1};
    if (encode_tiled_bf16(&L->tm_out, d.out, 4, dims, strides, box, 2)) { if (err && errlen) snprintf(err, errlen, "conv_stem: output tensor map encode failed"); return -1; }
    L->smem_bytes = SMEM_BYTES;
    L->grid = p.total < num_sms ? p.total : num_sms;
    L->flops = 2.0 * d.n * (1.0 * d.h * d.w * C1 * 27.0 + 1.0 * p.ho * p.wo * C2 * 9.0 * C1);
    return 0;
}

int conv_stem_init() {
    return cudaFuncSetAttribute(conv_stem_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES) == cudaSuccess ? 0 : -1;
}

int conv_stem_launch(const StemLaunch& L, cudaStream_t stream) {
    // launched without the programmatic-serialisation attribute (it is the first kernel of a pass: its input is a copy's
    // or another pass's output); the NEXT layer may still start its set-up early (griddepcontrol.launch_dependents above)
    conv_stem_kernel<<<L.grid, THREADS, L.smem_bytes, stream>>>(L.tm_out, L.p);
    return cudaPeekAtLastError() == cudaSuccess ? 0 : -1;
}

}  // namespace fd
