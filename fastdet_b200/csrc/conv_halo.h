// conv_halo.h — host interface of the halo-patch 3x3 convolution for narrow inputs (see conv_halo.cu).
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace fd {

struct HaloDesc {  // same meaning as ConvDesc (conv_tc.h)
    int n, hi, wi, cin, in_pitch;
    const __nv_bfloat16* in;
    int cout, ksize, stride, pad_lo, pad_hi;
    const __nv_bfloat16* w;  // [cout][3*3*cin]
    const float* bias_host;
    int act;
    float alpha;
    const __nv_bfloat16* residual;
    int res_pitch;
    void* out;
    int out_pitch, out_fp32, upsample2x;
    int pool2;  // 1: MaxPool(2, stride 2) of the activation in the epilogue; `out` is the (ho/2, wo/2) map
};

struct HaloParams {
    const __nv_bfloat16* in;
    int n, hi, wi;
    long long in_pitch;
    int ho, wo, stride;
    const __nv_bfloat16* w;
    int cin, cout, act;
    float alpha;
    const __nv_bfloat16* residual;
    long long res_pitch;
    int tiles_x, tiles_y, per_frame, total;
    int pool2;
    unsigned long long m_per_frame, m_tiles_x;  // ceil(2^40 / d): x / d == (x * m) >> 40 for the ranges checked on the host
    float bias_c[128];
};

struct HaloLaunch {
    CUtensorMap tm_out;  // {C, W, H, N} of the output slice, box 32 channels x 8 pixels x 4 rows, SWIZZLE_64B
    HaloParams p;
    int stride, cin, grid;
    size_t smem_bytes;
    double flops;
};

// One-time per device: opt in to the large dynamic shared memory the kernels need.
int conv_halo_init();
bool conv_halo_supported(const HaloDesc& d);
int conv_halo_prepare(const HaloDesc& d, int num_sms, HaloLaunch* out, char* err, size_t errlen);
int conv_halo_launch(const HaloLaunch& L, cudaStream_t stream);

}  // namespace fd
