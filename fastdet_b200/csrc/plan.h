// plan.h — ONNX graph -> static layer plan.
//
// The optimisation half of `ort.InferenceSession(...)` (reference server/detector.py:118), rebuilt for this
// path: Conv -> [BatchNormalization] -> [LeakyRelu] -> [Add] -> [Resize x2] chains collapse into one fused
// convolution each (BatchNorm folded into fp32 weights/bias before the bf16 rounding; the activation is LeakyRelu / Relu or
// Mish, written as one Mish node or as Softplus -> Tanh -> Mul), Concat becomes a shared
// buffer its producers write channel slices of, a channel Slice / Split becomes a view (a location inside its source's
// buffer, no layer), Pad+MaxPool merge, the "same" stride-1 max-pools of one tensor that all go into one Concat (an SPP
// block) run as one launch, and every activation gets a bf16 NHWC location.  No device code here; capi.cu turns the plan into buffers, tensor maps and launches.
#pragma once
#include <stdint.h>

#include <string>
#include <vector>

#include "onnx_reader.h"

namespace fd {

struct TensorLoc {
    int buf = -1;  // index into ModelPlan::buffers; -2 = the u8 input frames
    int c = 0, h = 0, w = 0;
    int pitch = 0;   // channels between pixels in the buffer
    int ch_off = 0;  // first channel of this tensor inside the buffer
};

enum LayerKind { LAYER_CONV0 = 0, LAYER_CONV = 1, LAYER_MAXPOOL = 2, LAYER_COPY = 3 };

struct LayerPlan {
    int kind = LAYER_CONV;
    std::string name;      // ONNX node name (or output name) of the anchoring op
    std::string out_name;  // ONNX tensor name whose value `out` holds (after all fused ops)
    TensorLoc in, out, res;
    // convolution
    int cin = 0, cout = 0, ksize = 1, stride = 1, pad_lo = 0, pad_hi = 0;
    int act = 0;  // 0 linear, 1 leaky (alpha), 2 Mish
    float alpha = 0.f;  // leaky only
    int out_fp32 = 0, upsample2x = 0;
    int pool2 = 0;  // 1: a MaxPool(2, stride 2) that follows the convolution is applied in its epilogue; `out` is the pooled tensor
    size_t w_off = 0;  // LAYER_CONV: element offset into weights_bf16; LAYER_CONV0: into conv0_w
    size_t b_off = 0;  // float offset into bias_f32
    // max-pool (window k, stride s); padding cells hold pad_value (-inf for ONNX MaxPool pads)
    int pool_k = 0, pool_s = 0, pool_pad_lo = 0, pool_pad_hi = 0;
    float pad_value = 0.f;
    // SPP group (stride-1 max-pools, pad (k-1)/2 with -inf, of one tensor whose outputs all go into one Concat): computed by
    // one launch (pool.cu launch_spp) at the group's last layer.  1: a member that launches nothing; 2: the last member,
    // spp_members = every layer of the group in order (itself included).  The members still write their own outputs.
    int spp = 0;
    std::vector<int> spp_members;
    double flops = 0.0;  // algorithmic, per frame
};

struct BufferPlan {
    int pitch = 0, h = 0, w = 0;
    int fp32 = 0;
};

struct ModelPlan {
    int net_w = 0, net_h = 0, num_classes = 0;
    std::vector<LayerPlan> layers;
    std::vector<BufferPlan> buffers;
    std::vector<int> head_layers;        // graph-output order (coarsest first by the reference's contract)
    std::vector<uint16_t> weights_bf16;  // all LAYER_CONV filters, [cout][kh][kw][cin] each, 128-byte aligned
    std::vector<float> bias_f32;         // per conv, padded to a multiple of 256 floats
    std::vector<float> conv0_w;          // first layer in fp32: [kh][kw][3][cout]
    double conv_flops_per_frame = 0.0;
    size_t num_params = 0;
};

// fuse_pool: fold MaxPool(2, 2) into the producing convolution where a kernel that can do it will run the layer
// (the first convolution and the halo-patch layers: 3x3 stride 1, 16/32/64 input channels, maps >= 64x64)
bool build_plan(const OnnxGraph& g, int net_w, int net_h, int num_classes, bool fuse_pool, ModelPlan* plan, std::string* err);

uint16_t f32_to_bf16_rn(float f);

}  // namespace fd
