// conv_tc.h — host-side interface of the tcgen05 implicit-GEMM convolution.
//
// Replaces the Conv(+BatchNormalization)(+LeakyRelu)(+Add) node groups that the reference hands
// to ONNX Runtime in `self.model.run` (reference server/detector.py:135).  Activations are bf16
// NHWC ("pixel rows" of `pitch` channels), weights are bf16 [Cout][kh][kw][Cin] (K-major), the
// accumulator is fp32 in TMEM.
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace fd {

struct ConvDesc {
    // input feature map: NHWC view, `in` already points at the first channel of the slice
    int n, hi, wi, cin;
    int in_pitch;  // channels between consecutive pixels (>= cin; > cin when reading a concat slice)
    const __nv_bfloat16* in;
    // filter
    int cout, ksize, stride;
    int pad_lo, pad_hi;  // begin / end padding (same for h and w)
    const __nv_bfloat16* w;  // [cout][ksize*ksize*cin], tap-major then channel
    const float* bias;       // device, [>= round_up(cout, 256)] fp32 (BatchNorm folded in)
    const float* bias_host;  // the same values on the host (they travel in the kernel's parameter block)
    int act;                 // 0 = linear, 1 = LeakyReLU(alpha)
    float alpha;
    // optional residual (added after the activation, like ONNX Add after LeakyRelu)
    const __nv_bfloat16* residual;
    int res_pitch;
    // output: bf16 NHWC slice (pitch >= cout) or fp32 rows (heads; pitch = padded cout)
    void* out;
    int out_pitch;
    int out_fp32;
    int upsample2x;  // write every output pixel to its 2x2 nearest-neighbour block of a (2Ho,2Wo) map
    int ho, wo;      // filled by conv_tc_prepare
    // 1: the layer may be split along K when it has too few tiles to fill the GPU (small batches); the caller then
    // provides the workspace conv_tc_prepare asks for through conv_tc_bind_workspace before the first launch
    int allow_split_k;
};

struct ConvParams {
    int M, cout, num_k_blocks, cin_blocks, ksize, stride, pad_lo, ho, wo;
    int block_k;  // 64 (SWIZZLE_128B), 32 (SWIZZLE_64B) or 16 (SWIZZLE_32B)
    int a_im2col; // 0: A via 2D tiled map (1x1 s1), 1: via im2col map
    int num_m_tiles, num_n_tiles;
    int num_stages;  // depth of the shared-memory operand ring
    int swap;          // 1: channels on the MMA's M side (128 per tile), 256 output pixels on its N side
    int b_resident;    // 1: the N tile's whole filter bank stays in shared memory, the ring carries A only
    int kb_per_stage;  // K blocks per ring stage (one barrier round trip covers all of them)
    const float* bias;
    int act;
    float alpha;
    const __nv_bfloat16* residual;
    long long res_pitch;
    void* out;
    long long out_pitch;
    int out_fp32, upsample2x;
    int n_store_limit;
    long long* prof;  // developer: per-CTA cycle counters [grid][16] (null in production)
    int debug;  // developer switches (0 in production): 1 skip epilogue stores, 2 skip A loads, 4 skip MMA issue
    // split-K (small batches): a tile's K range is cut into split_k parts run by different CTAs; every epilogue warp
    // writes its fp32 partial region to `ws`, and the warp that arrives last on the region's counter sums the parts in
    // part order (deterministic) and finishes the tile.  Results do not depend on arrival order, but do depend on
    // split_k, i.e. on the batch size.
    int split_k;
    float* ws;
    int* counters;
    int swap_tma;  // swapped mode: plain bf16 outputs without residual leave through TMA stores (32 ch x 32 pixels, SWIZZLE_64B)
    int head_tma;  // fp32 head rows leave through TMA stores (32 columns x 32 rows, SWIZZLE_128B)
    // "strip" mode (3x3, stride 1, pad 1 on the CTA-pair kernel): the M side walks the zero-padded, flattened pixel
    // positions q = (n * (H+1) + y+1) * (W+1) + x+1 (one pad column in front of every image row, one pad row in front of
    // every image: a row's right neighbour is the next row's pad); ONE im2col load per 64-channel block (bounding box one
    // pixel larger than the image on its low sides, out-of-bounds = zeros) brings the strip of strip_rows = 128 + 2(W+1) + 2
    // positions a CTA's 128 rows need, and the nine taps are descriptor row offsets ky*(W+1)+kx into it: a third of the
    // operand bytes of nine separate tap tiles.  Pad positions are computed and never stored.
    int strip, strip_wp, strip_hp, strip_rows, strip_qfirst, strip_total_q;
    int store64;   // 1: the output map's box is 64 channels x 32 rows (SWIZZLE_128B), two chunks per TMA store
    int res_v8;    // 1: residual rows are 32-byte aligned -> 256-bit loads
    int epi_mode;  // 0 bf16 slice through a TMA store (+ residual), 1 fp32 head rows, 2 bf16 with x2 upsampling
    // the layer's bias, read by the epilogue from the constant bank with a warp-uniform index (shared-memory and
    // L1 loads queue behind the operand traffic in this kernel; the constant cache does not)
    float bias_c[1024];
};

struct ConvLaunch {
    CUtensorMap tmA, tmB, tmOut;  // tmOut: {channels, pixel rows} of the output slice, 32 x 32 boxes, SWIZZLE_64B
    ConvParams p;
    int block_n;
    int two_cta;  // 1: CTA-pair kernel (cta_group::2, 256 x 256 tiles)
    int grid;
    size_t smem_bytes;
    size_t ws_bytes;      // split-K workspace this launch needs (0: none)
    size_t counter_ints;  // zero-initialised ints it needs
    double flops;  // algorithmic: 2*M*cout*K
};

// Builds tensor maps + launch geometry.  block_n_hint: 0 = choose, else one of 32/64/128/256;
// 512 = force the CTA-pair kernel, 257 = force the single-CTA 256-wide kernel, 1024 = force the swapped mode.
// Returns 0 on success; on failure writes a message to err (if non-null).
int conv_tc_prepare(const ConvDesc& d, int num_sms, int block_n_hint, ConvLaunch* out, char* err, size_t errlen);
int conv_tc_launch(const ConvLaunch& L, cudaStream_t stream);
// Split-K launches (L.ws_bytes > 0) need `ws` (>= L.ws_bytes) and `counters` (>= L.counter_ints, zeroed once; the kernel
// leaves them zero).  Launches of one stream may share both.
void conv_tc_bind_workspace(ConvLaunch* L, float* ws, int* counters);
// Tiled bf16 tensor map (rank 2..5) through the driver entry point this library resolves at run time.
// swizzle: 0 none, 1 32 B, 2 64 B, 3 128 B.  Returns 0 on success.
int encode_tiled_bf16(CUtensorMap* out, void* base, int rank, const unsigned long long* dims,
                      const unsigned long long* strides_bytes, const unsigned* box, int swizzle);
// One-time per device: opt in to the large dynamic shared memory the kernels need.
int conv_tc_init(char* err, size_t errlen);

}  // namespace fd
