// kernels.h — launch wrappers for the HBM-bound kernels around the conv stack (see the .cu files for the
// reference lines each one replaces).  All pointers are device pointers; every wrapper returns 0 or -1
// (cudaGetLastError() holds the reason).
#pragma once
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace fd {

// per-device one-time setup (opt-in shared memory sizes)
int kernels_init();

// ---- pre.cu -------------------------------------------------------------------------------------
// u8 HWC frames [n,h,w,3] -> f32 NCHW [n,3,h,w] = float32(k/255.0): reference server/detector.py:133-134.
int launch_normalise_f32_nchw(const uint8_t* frames, float* out, int n, int h, int w, cudaStream_t s);
// aspect-preserving bilinear letterbox (16.16 fixed point, grey fill) u8 [n,sh,sw,3] -> u8 [n,h,w,3]
// (extension: the reference server rejects non-net-sized frames, detector.py:131-132).
int launch_letterbox_u8(const uint8_t* src, uint8_t* dst, int n, int sh, int sw, int h, int w, int fill,
                        cudaStream_t s);
// first convolution fused with the normalisation: u8 [n,h,w,3] -> bf16 NHWC slice, 3x3 s1 p1, Cout <= 64,
// fp32 weights [3][3][3][cout] (BatchNorm folded), LeakyReLU(alpha) if act.
// pool2: MaxPool(2, stride 2) of the activation in the epilogue; `out` is then the (h/2, wd/2) map (Cout 16 / 32 only).
int launch_conv0_u8(const uint8_t* frames, const float* w, const float* bias, __nv_bfloat16* out, int n, int h,
                    int wd, int cout, int out_pitch, int act, float alpha, int pool2, cudaStream_t s);

// ---- pool.cu ------------------------------------------------------------------------------------
// max-pool over bf16 NHWC slices; cells outside the input take `pad_value` (-inf = ONNX MaxPool padding).
int launch_maxpool(const __nv_bfloat16* in, int in_pitch, __nv_bfloat16* out, int out_pitch, int n, int hi, int wi,
                   int c, int k, int stride, int pad_lo, int ho, int wo, float pad_value, cudaStream_t s);
// slice copy, optionally with x2 nearest upsampling (fallback when a Concat/Resize cannot be fused away).
int launch_copy_slice(const __nv_bfloat16* in, int in_pitch, __nv_bfloat16* out, int out_pitch, int n, int hi,
                      int wi, int c, int upsample2x, cudaStream_t s);
// bf16 NHWC slice / fp32 rows -> fp32 NCHW (parity hooks; not on the serving path)
int launch_nhwc_to_nchw_f32(const void* in, int in_pitch, int in_fp32, float* out, int n, int h, int w, int c,
                            cudaStream_t s);
// fp32 NCHW -> fp32 rows [n*h*w, pitch] (test hook: inject head tensors)
int launch_nchw_to_rows_f32(const float* in, float* out, int out_pitch, int n, int h, int w, int c, cudaStream_t s);

// ---- post.cu ------------------------------------------------------------------------------------
struct HeadDesc {
    const float* data;  // rows [n*h*w][pitch] fp32, channel = anchor*(5+nc)+{tx,ty,tw,th,obj,cls...}
    int pitch, h, w;
    int first_box;      // insertion-order index of this head's first box within a frame
    float anchor_w[3], anchor_h[3];
};
struct Candidate {     // one decoded box that passed both threshold tests (reference detector.py:152-165)
    double conf, x, y, w, h;  // normalised [0,1] top-left + size
    int box;                  // insertion-order index (head, row, column, anchor)
    int klass;                // 1-based
};
struct Detection {     // mirrors include/fastdet_b200.h: fd_det
    int32_t klass, box;
    double conf, x, y, w, h;
};
// Thresholds are per frame: thr[n] (the reference's `threshold`, a Python float) and obj_cut[n] = obj_cut_for(thr[f]),
// both device arrays, so frames of one batch may carry different thresholds.
// host: the objectness pre-test cut of decode for one threshold (-inf for thresholds outside (0, 1): no pre-test)
float obj_cut_for(double threshold);
// decode + two-stage threshold + compaction: fills cand[frame][*] (capacity boxes_per_frame) and counts.
int launch_decode(const HeadDesc* heads, int n_heads, int num_classes, int n, int net_w, int net_h,
                  const double* thr, const float* obj_cut, Candidate* cand, int* cand_count, int boxes_per_frame, cudaStream_t s);
// class-agnostic Gaussian Soft-NMS per frame (reference detector.py:45-59), frame f at threshold thr[f]; writes up to
// max_det detections per frame in selection order (pixels, top-left + size) and the per-frame count (untruncated count
// in total).
int launch_soft_nms(Candidate* cand, const int* cand_count, double* score_scratch, int boxes_per_frame, int n,
                    int net_w, int net_h, const double* thr, Detection* out, int* out_count, int* total_count,
                    int max_det, cudaStream_t s);

}  // namespace fd
