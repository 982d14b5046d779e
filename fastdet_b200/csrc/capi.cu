// capi.cu — the C ABI declared in include/fastdet_b200.h: model object, per-batch execution state
// (device buffers, tensor maps, captured CUDA graph) and the call sequence that stands in for
// ONNXDetector.__init__ / perform (reference server/detector.py:108-146).
#include <cuda_runtime.h>
#include <execinfo.h>
#include <math.h>
#include <signal.h>
#include <unistd.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <chrono>
#include <map>
#include <memory>
#include <mutex>
#include <string>
#include <vector>

#include "../../include/fastdet_b200.h"
#include "conv_block.h"
#include "conv_halo.h"
#include "conv_stem.h"
#include "conv_tc.h"
#include "jpeg.h"
#include "kernels.h"
#include "onnx_reader.h"
#include "options.h"
#include "plan.h"

using namespace fd;

static_assert(sizeof(Detection) == sizeof(fd_det), "Detection must mirror fd_det");

namespace {

thread_local char g_err[512] = "";

int fail(int code, const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return code;
}
#define CU(x)                                                                                          \
    do {                                                                                               \
        cudaError_t e_ = (x);                                                                          \
        if (e_ != cudaSuccess) return fail(FD_ERR_CUDA, "%s failed: %s", #x, cudaGetErrorString(e_)); \
    } while (0)

// reference server/detector.py:96-106
const float kAnchors3[3][3][2] = {{{116, 90}, {156, 198}, {373, 326}}, {{30, 61}, {62, 45}, {59, 119}}, {{10, 13}, {16, 30}, {33, 23}}};
const float kAnchors2[2][3][2] = {{{81, 82}, {135, 169}, {344, 319}}, {{10, 14}, {23, 27}, {37, 58}}};

// Launch descriptors of layers [0, layers) for pieces of `frames` frames each (piece k starts at frame k * frames, in the
// same buffers): the whole batch is one piece over every layer, fd_detect's copy-overlapped front four quarter-batch
// pieces over the leading layers.
struct LaunchSet {
    int layers = 0, frames = 0;
    std::vector<std::vector<ConvLaunch>> conv;  // [layer][piece]
    std::vector<std::vector<HaloLaunch>> halo;  // [layer][piece], used where use_halo[layer]
    std::vector<char> use_halo;                 // [layer]
    std::vector<StemLaunch> stem;               // [piece]; empty: no fused stem
    std::vector<BlockLaunch> block;             // [piece]; empty: no fused block
    size_t ws_bytes = 0, counter_ints = 0;      // split-K workspace the conv launches need (0: none)
};

struct Exec {  // everything that depends on the batch size
    int n = 0;
    std::vector<void*> bufs;
    LaunchSet whole;  // the forward pass
    // Fused stem (conv_stem.cu): layer 0 (u8 frames -> first convolution) runs inside layer 1's kernel; layer 0 has no launch
    // and its output tensor is never written (its buffer is only allocated when a parity hook asks for that tensor)
    bool use_stem = false;
    // Fused residual block (conv_block.cu): layer block_layer (1x1) runs inside layer block_layer + 1's kernel (3x3 + residual)
    int block_layer = -1;          // -1: none
    // per layer: 0 launches its own kernel, 1 computed inside the next layer's kernel (no launch, no output tensor), 2 launches a
    // fused kernel that also does the previous layer's work
    std::vector<char> fused_role;
    float* splitk_ws = nullptr;     // shared by the split-K launches of this batch size (they run one after another)
    int* splitk_counters = nullptr;
    uint8_t* frames = nullptr;     // [n, net_h, net_w, 3]
    uint8_t* src = nullptr;        // staging for frames that need the letterbox
    size_t src_cap = 0;
    Candidate* cand = nullptr;
    int* cand_count = nullptr;
    double* scores = nullptr;
    Detection* dets = nullptr;
    int* det_count = nullptr;  // [2n]: truncated counts then totals
    double* thr = nullptr;     // per-frame thresholds of the batch being post-processed: thr[b], then float obj_cut[b] (b frames)
    int max_det = 0;
    Detection* h_dets = nullptr;  // pinned
    int* h_count = nullptr;       // pinned [2n]
    float* scratch = nullptr;     // parity hooks
    size_t scratch_cap = 0;
    cudaGraphExec_t graph = nullptr;
    bool graph_tried = false;
    // fd_detect's copy-overlapped front (see forward_overlapping_copy): the layers in front of the second down-sampling
    // layer run from `front` quarter batch by quarter batch, the rest is graph_tail
    int ov_layers = 0;  // layers in the front; 0: not built yet, -1: not applicable
    LaunchSet front;
    cudaGraphExec_t graph_tail = nullptr;
    bool graph_tail_tried = false;
};

}  // namespace

struct Slot {  // one in-flight fd_submit: staged input + pinned results + the events that order them
    uint8_t* stage = nullptr;   // device staging for the H2D copy (copy stream)
    size_t stage_cap = 0;
    Detection* h_dets = nullptr;  // pinned
    size_t h_dets_cap = 0;
    int* h_count = nullptr;       // pinned [2n]
    size_t h_count_cap = 0;
    char* h_stage = nullptr;      // pinned: JPEG frame descriptors + quantised coefficients of one batch
    size_t h_stage_cap = 0;
    char* h_thr = nullptr;        // pinned: the batch's thresholds as the Exec's thr array takes them (stage_thresholds)
    size_t h_thr_cap = 0;
    int thr_n = 0;                // frames h_thr holds
    cudaEvent_t thr_copied = nullptr;  // the last copy out of h_thr has run
    cudaEvent_t staged = nullptr, stage_free = nullptr, done = nullptr;
    int n = 0, max_det = 0;
    bool busy = false;
};

struct fd_model {
    int device = 0;
    int num_sms = 148;
    cudaStream_t copy_stream = nullptr;
    Slot slots[FD_MAX_SLOTS + 1];  // the last one serves the synchronous JPEG calls and fd_postprocess
    std::unique_ptr<JpegPool> jpeg_pool;
    std::vector<JpegInfo> jpeg_info;
    uint8_t* jpeg_planes = nullptr;  // decoded component planes of the batch being converted (compute stream only)
    size_t jpeg_planes_cap = 0;
    ModelPlan plan;
    __nv_bfloat16* d_w = nullptr;
    float* d_bias = nullptr;
    float* d_conv0 = nullptr;
    cudaStream_t stream = nullptr;
    std::map<int, std::unique_ptr<Exec>> execs;
    cudaEvent_t h2d_ev[8] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};  // fd_detect: pieces of the frame copy
    cudaEvent_t idle_ev = nullptr;  // end of the last forward pass on the compute stream (its input tensor may be overwritten)
    fd_info info;
    int last_n = 0;
    int last_max_det = 0;
};

namespace {

// One process may drive several models on one device from different threads (fd_server: a lane per model).  CUDA calls
// that synchronise or reconfigure the whole device — cudaFree, cudaMallocHost, cudaDeviceSynchronize — conflict with a
// stream capture that another thread has open on the same device ("operation not permitted when stream is capturing",
// even in thread-local capture mode).  Everything rare that allocates, frees or captures therefore runs under the
// device's set-up lock; the steady-state enqueue / collect paths never take it.
std::recursive_mutex& device_setup_mutex(int device) {
    static std::recursive_mutex mu[64];
    return mu[device < 0 ? 63 : (device & 63)];
}
#define DEVICE_SETUP_LOCK(m) std::lock_guard<std::recursive_mutex> device_setup_lock_((device_setup_mutex((m)->device)))

// the two streams a model owns (never the whole device: another model's thread may be capturing on it)
int sync_model_streams(fd_model* m) {
    if (m->copy_stream) CU(cudaStreamSynchronize(m->copy_stream));
    if (m->stream) CU(cudaStreamSynchronize(m->stream));
    return FD_OK;
}

size_t buf_bytes(const BufferPlan& b, int n) { return size_t(n) * b.h * b.w * b.pitch * (b.fp32 ? 4 : 2); }

void free_exec(Exec* e) {
    for (void* p : e->bufs) cudaFree(p);
    cudaFree(e->splitk_ws); cudaFree(e->splitk_counters);
    cudaFree(e->frames); cudaFree(e->src); cudaFree(e->cand); cudaFree(e->cand_count); cudaFree(e->scores);
    cudaFree(e->dets); cudaFree(e->det_count); cudaFree(e->thr); cudaFree(e->scratch);
    if (e->h_dets) cudaFreeHost(e->h_dets);
    if (e->h_count) cudaFreeHost(e->h_count);
    if (e->graph) cudaGraphExecDestroy(e->graph);
    if (e->graph_tail) cudaGraphExecDestroy(e->graph_tail);
}

// first byte of tensor `t` for frames [k * frames, (k + 1) * frames) (k = 0: the whole batch)
void* loc_ptr(const Exec& e, const ModelPlan& P, const TensorLoc& t, bool fp32, int k = 0, int frames = 0) {
    char* base = static_cast<char*>(e.bufs[t.buf]) + static_cast<size_t>(k) * frames * buf_bytes(P.buffers[t.buf], 1);
    return base + size_t(t.ch_off) * (fp32 ? 4 : 2);
}

// Execution state is built per batch-size BUCKET, not per batch size: a serving front end submits whatever arrived
// (17 frames, then 43, ...), and a buffer set + captured graph for every distinct size would cost seconds of set-up
// and tens of GB.  n <= 64 rounds up to a power of two, larger batches to a multiple of 64; the conv stack runs on the
// bucket's frame count (frames past n hold stale pixels and are never decoded or copied out), everything else on n.
int bucket_of(int n) {
    if (n > 64) return (n + 63) / 64 * 64;
    int b = 1;
    while (b < n) b *= 2;
    return b;
}

// The fused stem applies when layer 0 is the u8 first convolution, layer 1 a 3x3 stride-2 convolution that is the ONLY
// reader of layer 0's output (no residual, no route), and conv_stem.cu takes the shapes (3 -> 32 -> 64: YOLOv3).
bool stem_candidate(const ModelPlan& P) {
    if (P.layers.size() < 2) return false;
    const LayerPlan& A = P.layers[0];
    const LayerPlan& B = P.layers[1];
    if (A.kind != LAYER_CONV0 || B.kind != LAYER_CONV || A.pool2 || B.pool2 || A.out_fp32 || B.out_fp32 || B.upsample2x || B.res.buf >= 0) return false;
    if (B.ksize != 3 || B.stride != 2 || B.pad_lo != 1 || A.ksize != 3 || A.stride != 1 || A.pad_lo != 1 || A.pad_hi != 1) return false;
    if (B.in.buf != A.out.buf || B.in.ch_off != A.out.ch_off || B.in.c != A.out.c || B.cin != A.cout) return false;
    for (size_t i = 2; i < P.layers.size(); ++i)
        if (P.layers[i].in.buf == A.out.buf || P.layers[i].res.buf == A.out.buf || P.layers[i].out.buf == A.out.buf) return false;
    for (int h : P.head_layers)
        if (h == 0) return false;
    return true;
}

// shapes and filters of the fused stem for `frames` frames; no frame / output pointers yet (null passes the kernel's alignment rules)
StemDesc stem_desc(const fd_model* m, int frames) {
    const ModelPlan& P = m->plan;
    const LayerPlan& A = P.layers[0];
    const LayerPlan& B = P.layers[1];
    StemDesc d;
    memset(&d, 0, sizeof(d));
    d.n = frames; d.h = A.in.h; d.w = A.in.w;
    d.c1 = A.cout; d.w1 = m->d_conv0 + A.w_off; d.bias1_host = P.bias_f32.data() + A.b_off; d.act1 = A.act; d.alpha1 = A.alpha;
    d.c2 = B.cout; d.pad_hi2 = B.pad_hi; d.w2 = m->d_w + B.w_off; d.bias2_host = P.bias_f32.data() + B.b_off; d.act2 = B.act; d.alpha2 = B.alpha;
    d.out_pitch = B.out.pitch;
    return d;
}

// the fused stem on frames [k * frames, (k + 1) * frames)
int prepare_stem(fd_model* m, Exec* e, int frames, int k, StemLaunch* sl) {
    const ModelPlan& P = m->plan;
    StemDesc d = stem_desc(m, frames);
    d.frames = e->frames + static_cast<size_t>(k) * frames * P.net_h * P.net_w * 3;
    d.out = static_cast<__nv_bfloat16*>(loc_ptr(*e, P, P.layers[1].out, false, k, frames));
    char err[256] = "";
    if (conv_stem_prepare(d, m->num_sms, sl, err, sizeof(err))) return fail(FD_ERR_CUDA, "stem (layers 0 + 1): %s", err);
    return FD_OK;
}

// A residual block conv_block.cu can fuse: layer i a 1x1 stride-1 convolution, layer i + 1 the 3x3 stride-1 convolution that
// is the ONLY reader of layer i's output and adds layer i's INPUT tensor as its residual.  Returns the first such i, or -1.
int block_candidate(const ModelPlan& P) {
    for (size_t i = 1; i + 1 < P.layers.size(); ++i) {
        const LayerPlan& A = P.layers[i];
        const LayerPlan& B = P.layers[i + 1];
        if (A.kind != LAYER_CONV || B.kind != LAYER_CONV || A.ksize != 1 || A.stride != 1 || A.res.buf >= 0 || A.pool2 || B.pool2 ||
            A.out_fp32 || B.out_fp32 || A.upsample2x || B.upsample2x)
            continue;
        if (B.ksize != 3 || B.stride != 1 || B.pad_lo != 1 || B.pad_hi != 1 || B.res.buf < 0) continue;
        if (B.in.buf != A.out.buf || B.in.ch_off != A.out.ch_off || B.in.c != A.out.c || B.cin != A.cout) continue;
        if (B.res.buf != A.in.buf || B.res.ch_off != A.in.ch_off || B.res.pitch != A.in.pitch || B.cout != A.cin) continue;
        bool sole = true;
        for (size_t j = 0; j < P.layers.size(); ++j)
            if (j != i && j != i + 1 && (P.layers[j].in.buf == A.out.buf || P.layers[j].res.buf == A.out.buf || P.layers[j].out.buf == A.out.buf)) sole = false;
        for (int h : P.head_layers)
            if (h == static_cast<int>(i)) sole = false;
        if (sole) return static_cast<int>(i);
    }
    return -1;
}

// shapes and filters of the fused block for `frames` frames; no tensor pointers yet (null passes the kernel's alignment rules)
BlockDesc block_desc(const fd_model* m, int layer, int frames) {
    const ModelPlan& P = m->plan;
    const LayerPlan& A = P.layers[layer];
    const LayerPlan& B = P.layers[layer + 1];
    BlockDesc d;
    memset(&d, 0, sizeof(d));
    d.n = frames; d.h = A.in.h; d.w = A.in.w; d.in_pitch = A.in.pitch;
    d.cin = A.cin; d.cmid = A.cout; d.cout = B.cout;
    d.wa = m->d_w + A.w_off; d.bias_a_host = P.bias_f32.data() + A.b_off; d.act_a = A.act; d.alpha_a = A.alpha;
    d.wb = m->d_w + B.w_off; d.bias_b_host = P.bias_f32.data() + B.b_off; d.act_b = B.act; d.alpha_b = B.alpha;
    d.out_pitch = B.out.pitch;
    return d;
}

// the fused block on frames [k * frames, (k + 1) * frames)
int prepare_block(fd_model* m, Exec* e, int layer, int frames, int k, BlockLaunch* bl) {
    const ModelPlan& P = m->plan;
    BlockDesc d = block_desc(m, layer, frames);
    d.in = static_cast<const __nv_bfloat16*>(loc_ptr(*e, P, P.layers[layer].in, false, k, frames));
    d.out = static_cast<__nv_bfloat16*>(loc_ptr(*e, P, P.layers[layer + 1].out, false, k, frames));
    char err[256] = "";
    if (conv_block_prepare(d, m->num_sms, bl, err, sizeof(err))) return fail(FD_ERR_CUDA, "residual block (layers %d + %d): %s", layer, layer + 1, err);
    return FD_OK;
}

// tensor maps + launch geometry of conv layer i on frames [k * frames, (k + 1) * frames)
int prepare_conv_layer(fd_model* m, Exec* e, size_t i, int frames, int k, ConvLaunch* cl, HaloLaunch* hl, char* use_halo) {
    const ModelPlan& P = m->plan;
    const LayerPlan& L = P.layers[i];
    const __nv_bfloat16* in = static_cast<const __nv_bfloat16*>(loc_ptr(*e, P, L.in, false, k, frames));
    const __nv_bfloat16* res = L.res.buf >= 0 ? static_cast<const __nv_bfloat16*>(loc_ptr(*e, P, L.res, false, k, frames)) : nullptr;
    void* out = loc_ptr(*e, P, L.out, L.out_fp32 != 0, k, frames);
    {   // narrow 3x3 layers on large maps: halo-patch kernel (conv_halo.cu)
        HaloDesc h;
        memset(&h, 0, sizeof(h));
        h.n = frames; h.hi = L.in.h; h.wi = L.in.w; h.cin = L.cin; h.in_pitch = L.in.pitch;
        h.in = in;
        h.cout = L.cout; h.ksize = L.ksize; h.stride = L.stride; h.pad_lo = L.pad_lo; h.pad_hi = L.pad_hi;
        h.w = m->d_w + L.w_off; h.bias_host = P.bias_f32.data() + L.b_off; h.act = L.act; h.alpha = L.alpha;
        if (res) { h.residual = res; h.res_pitch = L.res.pitch; }
        h.out = out; h.out_pitch = L.out.pitch; h.out_fp32 = L.out_fp32; h.upsample2x = L.upsample2x;
        h.pool2 = L.pool2;
        char herr[256] = "";
        if (conv_halo_supported(h) && conv_halo_prepare(h, m->num_sms, hl, herr, sizeof(herr)) == 0) { *use_halo = 1; return FD_OK; }
        if (L.pool2) return fail(FD_ERR_CUDA, "layer %zu (%s): its fused max-pool needs the halo-patch kernel (%s)", i, L.name.c_str(), herr);
    }
    *use_halo = 0;
    ConvDesc d;
    memset(&d, 0, sizeof(d));
    d.n = frames; d.hi = L.in.h; d.wi = L.in.w; d.cin = L.cin; d.in_pitch = L.in.pitch;
    d.in = in;
    d.cout = L.cout; d.ksize = L.ksize; d.stride = L.stride; d.pad_lo = L.pad_lo; d.pad_hi = L.pad_hi;
    d.w = m->d_w + L.w_off; d.bias = m->d_bias + L.b_off; d.bias_host = P.bias_f32.data() + L.b_off; d.act = L.act; d.alpha = L.alpha;
    if (res) { d.residual = res; d.res_pitch = L.res.pitch; }
    d.out = out; d.out_pitch = L.out.pitch; d.out_fp32 = L.out_fp32; d.upsample2x = L.upsample2x;
    d.allow_split_k = 1;
    char err[256] = "";
    if (conv_tc_prepare(d, m->num_sms, 0, cl, err, sizeof(err))) return fail(FD_ERR_CUDA, "layer %zu (%s): %s", i, L.name.c_str(), err);
    return FD_OK;
}

// the output buffer of a layer that is computed inside the next layer's kernel: not allocated up front (nothing writes it
// during a forward pass), only when a parity hook asks for that tensor
int ensure_fused_away_buffer(fd_model* m, Exec* e, int layer) {
    const ModelPlan& P = m->plan;
    const int b = P.layers[layer].out.buf;
    if (e->bufs[b]) return FD_OK;
    DEVICE_SETUP_LOCK(m);
    cudaError_t err = cudaMalloc(&e->bufs[b], buf_bytes(P.buffers[b], e->n));
    if (err != cudaSuccess) return fail(FD_ERR_CUDA, "cudaMalloc(output of layer %d, batch %d) failed: %s", layer, e->n, cudaGetErrorString(err));
    return FD_OK;
}

// Launch descriptors of layers [0, layers) for `pieces` pieces of `frames` frames, following the Exec's fusion plan.
int prepare_set(fd_model* m, Exec* e, int layers, int pieces, int frames, LaunchSet* ls) {
    const ModelPlan& P = m->plan;
    ls->layers = layers; ls->frames = frames;
    ls->conv.assign(layers, {});
    ls->halo.assign(layers, {});
    ls->use_halo.assign(layers, 0);
    for (int i = 0; i < layers; ++i) {
        if (P.layers[i].kind != LAYER_CONV) continue;
        ls->conv[i].resize(pieces);
        ls->halo[i].resize(pieces);
        if (e->fused_role[i]) continue;  // fused layers: a tensor of the pair does not exist, the pair has its own launch below
        for (int k = 0; k < pieces; ++k) {
            char uh = 0;
            if (int rc = prepare_conv_layer(m, e, i, frames, k, &ls->conv[i][k], &ls->halo[i][k], &uh)) return rc;
            ls->use_halo[i] = uh;
            ls->ws_bytes = std::max(ls->ws_bytes, ls->conv[i][k].ws_bytes);
            ls->counter_ints = std::max(ls->counter_ints, ls->conv[i][k].counter_ints);
        }
    }
    if (e->use_stem) {
        ls->stem.resize(pieces);
        for (int k = 0; k < pieces; ++k)
            if (int rc = prepare_stem(m, e, frames, k, &ls->stem[k])) return rc;
    }
    if (e->block_layer >= 0 && e->block_layer < layers) {
        ls->block.resize(pieces);
        for (int k = 0; k < pieces; ++k)
            if (int rc = prepare_block(m, e, e->block_layer, frames, k, &ls->block[k])) return rc;
    }
    return FD_OK;
}

int get_exec(fd_model* m, int n_frames, Exec** out) {
    if (n_frames <= 0) return fail(FD_ERR_ARG, "batch size must be positive (got %d)", n_frames);
    const int n = bucket_of(n_frames);
    auto it = m->execs.find(n);
    if (it != m->execs.end()) { *out = it->second.get(); return FD_OK; }
    DEVICE_SETUP_LOCK(m);
    std::unique_ptr<Exec> e(new Exec());
    e->n = n;
    const ModelPlan& P = m->plan;
    e->bufs.assign(P.buffers.size(), nullptr);
    // fused kernels: decided here, from the shapes, because the output buffer of a fused-away layer is then not allocated at all
    int32_t stem = 0, block = -1;
    if (int rc = fd_planned_fusions(m, n, &stem, &block)) return rc;
    e->use_stem = stem != 0;
    e->block_layer = block;
    e->fused_role.assign(P.layers.size(), 0);
    if (e->use_stem) { e->fused_role[0] = 1; e->fused_role[1] = 2; }
    if (e->block_layer >= 0) { e->fused_role[e->block_layer] = 1; e->fused_role[e->block_layer + 1] = 2; }
    for (size_t i = 0; i < P.buffers.size(); ++i) {
        bool skip = false;  // outputs of fused-away layers are never written: allocated on demand by the parity hook
        for (size_t li = 0; li < P.layers.size(); ++li)
            if (e->fused_role[li] == 1 && P.layers[li].out.buf == static_cast<int>(i)) skip = true;
        if (skip) continue;
        cudaError_t err = cudaMalloc(&e->bufs[i], buf_bytes(P.buffers[i], n));
        if (err != cudaSuccess) { free_exec(e.get()); return fail(FD_ERR_CUDA, "cudaMalloc(activation buffer %zu, batch %d) failed: %s", i, n, cudaGetErrorString(err)); }
    }
    const size_t frame_bytes = size_t(n) * P.net_h * P.net_w * 3;
    const int bpf = m->info.boxes_per_frame;
    if (cudaMalloc(&e->frames, frame_bytes) != cudaSuccess ||
        cudaMalloc(&e->cand, sizeof(Candidate) * size_t(n) * bpf) != cudaSuccess ||
        cudaMalloc(&e->cand_count, sizeof(int) * n) != cudaSuccess ||
        cudaMalloc(&e->scores, sizeof(double) * size_t(n) * bpf) != cudaSuccess ||
        cudaMalloc(&e->det_count, sizeof(int) * 2 * n) != cudaSuccess ||
        cudaMalloc(&e->thr, (sizeof(double) + sizeof(float)) * n) != cudaSuccess ||
        cudaMallocHost(&e->h_count, sizeof(int) * 2 * n) != cudaSuccess ||
        cudaMemset(e->frames, 0, frame_bytes) != cudaSuccess) {
        free_exec(e.get());
        return fail(FD_ERR_CUDA, "cudaMalloc(per-batch state, batch %d) failed: %s", n, cudaGetErrorString(cudaGetLastError()));
    }
    if (int rc = prepare_set(m, e.get(), static_cast<int>(P.layers.size()), 1, n, &e->whole)) { free_exec(e.get()); return rc; }
    if (e->whole.ws_bytes) {
        const size_t counter_ints = e->whole.counter_ints;
        if (cudaMalloc(&e->splitk_ws, e->whole.ws_bytes) != cudaSuccess || cudaMalloc(&e->splitk_counters, counter_ints * sizeof(int)) != cudaSuccess ||
            cudaMemset(e->splitk_counters, 0, counter_ints * sizeof(int)) != cudaSuccess) {
            free_exec(e.get());
            return fail(FD_ERR_CUDA, "cudaMalloc(split-K workspace, batch %d) failed: %s", n, cudaGetErrorString(cudaGetLastError()));
        }
        for (auto& v : e->whole.conv)
            for (ConvLaunch& c : v)
                if (c.ws_bytes) conv_tc_bind_workspace(&c, e->splitk_ws, e->splitk_counters);
    }
    *out = e.get();
    m->execs[n] = std::move(e);
    return FD_OK;
}

// layer i's own kernel on frames [k * frames, (k + 1) * frames), conv layers with the given launch descriptors
int launch_own(fd_model* m, Exec* e, int i, int k, int frames, bool halo, const ConvLaunch* cl, const HaloLaunch* hl, cudaStream_t s) {
    const ModelPlan& P = m->plan;
    const LayerPlan& L = P.layers[i];
    int rc = 0;
    switch (L.kind) {
        case LAYER_CONV0:
            rc = launch_conv0_u8(e->frames + static_cast<size_t>(k) * frames * P.net_h * P.net_w * 3, m->d_conv0 + L.w_off, m->d_bias + L.b_off,
                                 static_cast<__nv_bfloat16*>(loc_ptr(*e, P, L.out, false, k, frames)), frames, L.in.h, L.in.w, L.cout,
                                 L.out.pitch, L.act, L.alpha, L.pool2, s);
            break;
        case LAYER_CONV: rc = halo ? conv_halo_launch(*hl, s) : conv_tc_launch(*cl, s); break;
        case LAYER_MAXPOOL:
            rc = launch_maxpool(static_cast<const __nv_bfloat16*>(loc_ptr(*e, P, L.in, false, k, frames)), L.in.pitch,
                                static_cast<__nv_bfloat16*>(loc_ptr(*e, P, L.out, false, k, frames)), L.out.pitch, frames, L.in.h, L.in.w,
                                L.in.c, L.pool_k, L.pool_s, L.pool_pad_lo, L.out.h, L.out.w, L.pad_value, s);
            break;
        case LAYER_COPY:
            rc = launch_copy_slice(static_cast<const __nv_bfloat16*>(loc_ptr(*e, P, L.in, false, k, frames)), L.in.pitch,
                                   static_cast<__nv_bfloat16*>(loc_ptr(*e, P, L.out, false, k, frames)), L.out.pitch, frames, L.in.h, L.in.w,
                                   L.in.c, L.upsample2x, s);
            break;
        default: rc = -1;
    }
    if (rc) return fail(FD_ERR_CUDA, "launch of layer %d (%s) failed: %s", i, L.name.c_str(), cudaGetErrorString(cudaGetLastError()));
    return FD_OK;
}

// layer i, piece k of a launch set: a layer computed inside the next layer's kernel has no launch, the second layer of a
// fused pair launches the fused kernel (stem = layers 0 + 1, block = layers block_layer + block_layer + 1)
int launch_piece(fd_model* m, Exec* e, const LaunchSet& ls, int i, int k, cudaStream_t s) {
    if (e->fused_role[i] == 1) return FD_OK;
    if (e->fused_role[i] == 2 && e->use_stem && i == 1) {
        if (conv_stem_launch(ls.stem[k], s)) return fail(FD_ERR_CUDA, "launch of the fused stem (layers 0 + 1) failed: %s", cudaGetErrorString(cudaGetLastError()));
        return FD_OK;
    }
    if (e->fused_role[i] == 2) {
        if (conv_block_launch(ls.block[k], s)) return fail(FD_ERR_CUDA, "launch of the fused residual block (layers %d + %d) failed: %s", i - 1, i, cudaGetErrorString(cudaGetLastError()));
        return FD_OK;
    }
    const bool conv = m->plan.layers[i].kind == LAYER_CONV;
    return launch_own(m, e, i, k, ls.frames, ls.use_halo[i] != 0, conv ? &ls.conv[i][k] : nullptr, conv ? &ls.halo[i][k] : nullptr, s);
}

// The forward pass on the whole batch, from layer `from_layer` on.
int launch_layers(fd_model* m, Exec* e, cudaStream_t s, int from_layer = 0) {
    for (int i = from_layer; i < e->whole.layers; ++i)
        if (int rc = launch_piece(m, e, e->whole, i, 0, s)) return rc;
    return FD_OK;
}

#define NEED_DEVICE(m)                                                                                         \
    do {                                                                                                       \
        if ((m)->device < 0) return fail(FD_ERR_CUDA, "plan-only model (device -1): no CUDA device attached, no CPU fallback"); \
    } while (0)

cudaStream_t pick(fd_model* m, void* stream) { return stream ? static_cast<cudaStream_t>(stream) : m->stream; }

int ensure_scratch(Exec* e, size_t bytes) {
    if (e->scratch_cap >= bytes) return FD_OK;
    int dev = 0;
    cudaGetDevice(&dev);
    std::lock_guard<std::recursive_mutex> lk(device_setup_mutex(dev));
    cudaFree(e->scratch);
    e->scratch = nullptr; e->scratch_cap = 0;
    CU(cudaMalloc(&e->scratch, bytes));
    e->scratch_cap = bytes;
    return FD_OK;
}

}  // namespace

// library-internal (csrc/server.cc): pinned host memory under the device's set-up lock
void* fd_internal_pinned_alloc(int device, size_t bytes) {
    std::lock_guard<std::recursive_mutex> lk(device_setup_mutex(device));
    void* p = nullptr;
    if (cudaSetDevice(device) != cudaSuccess || cudaMallocHost(&p, bytes) != cudaSuccess) { cudaGetLastError(); return nullptr; }
    return p;
}
void fd_internal_pinned_free(int device, void* p) {
    std::lock_guard<std::recursive_mutex> lk(device_setup_mutex(device));
    cudaFreeHost(p);
}

extern "C" {

const char* fd_last_error(void) { return g_err; }
int fd_abi_version(void) { return FD_ABI_VERSION; }
int fd_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}

int fd_model_create(const void* onnx_bytes, size_t len, int num_classes, int net_w, int net_h, int device, fd_model** out) {
    if (!onnx_bytes || !len || !out) return fail(FD_ERR_ARG, "fd_model_create: null argument");
    if (num_classes < 1 || net_w < 32 || net_h < 32 || net_w % 32 || net_h % 32)
        return fail(FD_ERR_ARG, "fd_model_create: num_classes must be >= 1 and the network size a multiple of 32 (got %d, %dx%d)", num_classes, net_w, net_h);
    *out = nullptr;
    OnnxGraph g;
    std::string err;
    if (!onnx_parse(onnx_bytes, len, &g, &err)) return fail(FD_ERR_MODEL, "ONNX parse error: %s", err.c_str());
    struct Cleanup { void operator()(fd_model* p) const { fd_model_destroy(p); } };  // frees whatever a failed create had already allocated
    std::unique_ptr<fd_model, Cleanup> m(new fd_model());
    m->device = -1;  // until a device is attached: destroy then only frees host state
    if (!build_plan(g, net_w, net_h, num_classes, options().fuse_pool, &m->plan, &err)) return fail(FD_ERR_MODEL, "unsupported ONNX graph: %s", err.c_str());
    ModelPlan& P = m->plan;
    if (P.head_layers.size() > FD_MAX_HEADS) return fail(FD_ERR_MODEL, "graph has %zu outputs (max %d)", P.head_layers.size(), FD_MAX_HEADS);

    fd_info& I = m->info;
    memset(&I, 0, sizeof(I));
    I.abi_version = FD_ABI_VERSION; I.device = device; I.net_w = net_w; I.net_h = net_h; I.num_classes = num_classes;
    I.n_heads = static_cast<int>(P.head_layers.size());
    int boxes = 0;
    for (int h = 0; h < I.n_heads; ++h) {
        const LayerPlan& L = P.layers[P.head_layers[h]];
        I.head_h[h] = L.out.h; I.head_w[h] = L.out.w; I.head_c[h] = L.out.c;
        if (L.out.c != 3 * (5 + num_classes))
            return fail(FD_ERR_MODEL, "head %d has %d channels but num_classes=%d needs %d", h, L.out.c, num_classes, 3 * (5 + num_classes));
        boxes += 3 * L.out.h * L.out.w;
        for (int k = 0; k < 3; ++k)
            for (int j = 0; j < 2; ++j)
                I.anchors[h][k][j] = I.n_heads == 3 ? kAnchors3[h][k][j] : (I.n_heads == 2 ? kAnchors2[h][k][j] : 0.f);
    }
    I.boxes_per_frame = boxes;
    I.n_layers = static_cast<int>(P.layers.size());
    for (const auto& L : P.layers) I.n_conv += (L.kind == LAYER_CONV || L.kind == LAYER_CONV0);
    I.launches_per_detect = I.n_layers + 2;
    I.conv_flops_per_frame = P.conv_flops_per_frame;
    I.num_params = P.num_params;
    I.weight_bytes = P.weights_bf16.size() * 2 + P.bias_f32.size() * 4 + P.conv0_w.size() * 4;

    if (device == -1) {  // plan-only model: host logic (parse, fuse, fold, pack) without touching CUDA
        m->device = -1;
        *out = m.release();
        return FD_OK;
    }
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
        cudaGetLastError();
        return fail(FD_ERR_CUDA, "no CUDA device available: fastdet_b200 has no CPU fallback");
    }
    if (device < 0 || device >= ndev) return fail(FD_ERR_ARG, "device %d out of range (have %d)", device, ndev);
    CU(cudaSetDevice(device));
    m->device = device;
    DEVICE_SETUP_LOCK(m);
    cudaDeviceProp prop;
    CU(cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10) return fail(FD_ERR_CUDA, "device %d is sm_%d%d; this library is built for sm_100a (B200) only", device, prop.major, prop.minor);
    m->num_sms = prop.multiProcessorCount;
    char cerr[256] = "";
    if (conv_tc_init(cerr, sizeof(cerr))) return fail(FD_ERR_CUDA, "conv_tc_init: %s", cerr);
    if (kernels_init()) return fail(FD_ERR_CUDA, "kernels_init failed: %s", cudaGetErrorString(cudaGetLastError()));
    if (conv_halo_init()) return fail(FD_ERR_CUDA, "conv_halo_init failed: %s", cudaGetErrorString(cudaGetLastError()));
    if (conv_stem_init()) return fail(FD_ERR_CUDA, "conv_stem_init failed: %s", cudaGetErrorString(cudaGetLastError()));
    if (conv_block_init()) return fail(FD_ERR_CUDA, "conv_block_init failed: %s", cudaGetErrorString(cudaGetLastError()));
    CU(cudaStreamCreateWithFlags(&m->stream, cudaStreamNonBlocking));
    CU(cudaMalloc(&m->d_w, std::max<size_t>(P.weights_bf16.size(), 64) * 2));
    CU(cudaMalloc(&m->d_bias, std::max<size_t>(P.bias_f32.size(), 64) * 4));
    CU(cudaMalloc(&m->d_conv0, std::max<size_t>(P.conv0_w.size(), 64) * 4));
    CU(cudaMemcpy(m->d_w, P.weights_bf16.data(), P.weights_bf16.size() * 2, cudaMemcpyHostToDevice));
    CU(cudaMemcpy(m->d_bias, P.bias_f32.data(), P.bias_f32.size() * 4, cudaMemcpyHostToDevice));
    CU(cudaMemcpy(m->d_conv0, P.conv0_w.data(), P.conv0_w.size() * 4, cudaMemcpyHostToDevice));
    // host copies are no longer needed
    std::vector<uint16_t>().swap(P.weights_bf16);
    *out = m.release();
    return FD_OK;
}

void fd_model_destroy(fd_model* m) {
    if (!m) return;
    if (m->device < 0) { delete m; return; }
    cudaSetDevice(m->device);
    DEVICE_SETUP_LOCK(m);
    sync_model_streams(m);
    for (auto& kv : m->execs) free_exec(kv.second.get());
    cudaFree(m->d_w); cudaFree(m->d_bias); cudaFree(m->d_conv0);
    for (Slot& S : m->slots) {
        cudaFree(S.stage);
        if (S.h_stage) cudaFreeHost(S.h_stage);
        if (S.h_dets) cudaFreeHost(S.h_dets);
        if (S.h_count) cudaFreeHost(S.h_count);
        if (S.h_thr) cudaFreeHost(S.h_thr);
        if (S.thr_copied) cudaEventDestroy(S.thr_copied);
        if (S.staged) { cudaEventDestroy(S.staged); cudaEventDestroy(S.stage_free); cudaEventDestroy(S.done); }
    }
    cudaFree(m->jpeg_planes);
    if (m->idle_ev) { cudaEventDestroy(m->idle_ev); for (cudaEvent_t ev : m->h2d_ev) cudaEventDestroy(ev); }
    if (m->copy_stream) cudaStreamDestroy(m->copy_stream);
    if (m->stream) cudaStreamDestroy(m->stream);
    delete m;
}

int fd_model_info(const fd_model* m, fd_info* out) {
    if (!m || !out) return fail(FD_ERR_ARG, "fd_model_info: null argument");
    *out = m->info;
    return FD_OK;
}

int fd_layer_info(const fd_model* m, int layer, fd_layer_desc* out) {
    if (!m || !out || layer < 0 || layer >= static_cast<int>(m->plan.layers.size())) return fail(FD_ERR_ARG, "fd_layer_info: bad layer %d", layer);
    const LayerPlan& L = m->plan.layers[layer];
    memset(out, 0, sizeof(*out));
    out->kind = L.kind; out->c = L.out.c; out->h = L.out.h; out->w = L.out.w;
    out->cin = L.cin; out->ksize = L.ksize; out->stride = L.stride; out->act = L.act;
    out->has_residual = L.res.buf >= 0; out->upsample2x = L.upsample2x; out->out_fp32 = L.out_fp32;
    out->flops = L.flops;
    if (L.kind == LAYER_CONV && !m->execs.empty()) {
        const Exec& e0 = *m->execs.begin()->second;
        out->block_n = e0.whole.use_halo[layer] ? -1 : e0.whole.conv[layer][0].block_n;  // -1: halo-patch kernel
    }
    snprintf(out->name, sizeof(out->name), "%s", L.name.c_str());
    snprintf(out->out_name, sizeof(out->out_name), "%s", L.out_name.c_str());
    return FD_OK;
}

// Host logic only (works on a plan-only model): which layers the planner would hand to the fused kernels at batch n under the
// current options — *stem = 1 when layers 0 + 1 run as conv_stem_kernel, *block_layer = the 1x1 layer of the pair that runs
// as conv_block_kernel (or -1).  The execution state of batch n is built from this answer.
int fd_planned_fusions(const fd_model* m, int n, int32_t* stem, int32_t* block_layer) {
    if (!m || !stem || !block_layer || n < 1) return fail(FD_ERR_ARG, "fd_planned_fusions: bad argument");
    const ModelPlan& P = m->plan;
    *stem = (options().stem && stem_candidate(P) && conv_stem_supported(stem_desc(m, n))) ? 1 : 0;
    *block_layer = -1;
    if (options().block) {
        const int bc = block_candidate(P);
        if (bc >= 0 && conv_block_supported(block_desc(m, bc, n))) *block_layer = bc;
    }
    return FD_OK;
}

int fd_layer_exec_info(fd_model* m, int layer, int n, fd_layer_exec* out) {
    if (!m || !out || layer < 0 || layer >= static_cast<int>(m->plan.layers.size())) return fail(FD_ERR_ARG, "fd_layer_exec_info: bad layer %d", layer);
    NEED_DEVICE(m);
    CU(cudaSetDevice(m->device));
    Exec* e;
    if (int rc = get_exec(m, n, &e)) return rc;
    const LayerPlan& L = m->plan.layers[layer];
    memset(out, 0, sizeof(*out));
    out->bucket = e->n;
    out->chunk_frames = e->n;
    out->launches = e->fused_role[layer] == 1 ? 0 : 1;
    const LaunchSet& W = e->whole;
    if (e->use_stem && layer < 2) {
        out->kernel = layer == 0 ? FD_KERNEL_FUSED_NEXT : FD_KERNEL_STEM;
        if (layer == 1) { out->grid = W.stem[0].grid; out->smem_bytes = static_cast<int32_t>(W.stem[0].smem_bytes); }
        return FD_OK;
    }
    if (e->block_layer >= 0 && (layer == e->block_layer || layer == e->block_layer + 1)) {
        out->kernel = layer == e->block_layer ? FD_KERNEL_FUSED_NEXT : FD_KERNEL_BLOCK;
        if (layer != e->block_layer) { out->grid = W.block[0].grid; out->smem_bytes = static_cast<int32_t>(W.block[0].smem_bytes); }
        return FD_OK;
    }
    switch (L.kind) {
        case LAYER_CONV0: out->kernel = FD_KERNEL_CONV0; break;
        case LAYER_MAXPOOL: out->kernel = FD_KERNEL_MAXPOOL; break;
        case LAYER_COPY: out->kernel = FD_KERNEL_COPY; break;
        default:
            if (W.use_halo[layer]) {
                out->kernel = FD_KERNEL_HALO;
                out->grid = W.halo[layer][0].grid;
                out->smem_bytes = static_cast<int32_t>(W.halo[layer][0].smem_bytes);
            } else {
                const ConvLaunch& c = W.conv[layer][0];
                out->kernel = c.p.strip ? FD_KERNEL_TC_PAIR_STRIP : c.two_cta ? FD_KERNEL_TC_PAIR : c.p.swap ? FD_KERNEL_TC_SWAPPED : FD_KERNEL_TC_SINGLE;
                out->block_n = c.block_n; out->split_k = c.p.split_k; out->grid = c.grid; out->num_stages = c.p.num_stages;
                out->kb_per_stage = c.p.kb_per_stage; out->b_resident = c.p.b_resident;
                out->smem_bytes = static_cast<int32_t>(c.smem_bytes);
            }
    }
    return FD_OK;
}

// developer aid (fd_set_option("segv_backtrace", 1)): a crash inside the library's host threads prints its call stack
// (module + offset, resolvable with addr2line against the same .so) instead of dying silently under a test runner
static void segv_backtrace_handler(int sig) {
    void* frames[64];
    const int n = backtrace(frames, 64);
    const char msg[] = "fastdet_b200: fatal signal, call stack:\n";
    if (write(2, msg, sizeof(msg) - 1) < 0) {}
    backtrace_symbols_fd(frames, n, 2);
    _exit(128 + sig);
}

int fd_set_option(const char* name, int value) {
    if (name && !strcmp(name, "segv_backtrace")) {
        signal(SIGSEGV, value ? segv_backtrace_handler : SIG_DFL);
        signal(SIGBUS, value ? segv_backtrace_handler : SIG_DFL);
        return FD_OK;
    }
    int* slot = option_slot(name);
    if (!slot) return fail(FD_ERR_ARG, "fd_set_option: unknown option '%s'", name ? name : "(null)");
    *slot = value;
    return FD_OK;
}

int fd_get_option(const char* name, int* value) {
    const int* slot = option_slot(name);
    if (!slot || !value) return fail(FD_ERR_ARG, "fd_get_option: unknown option '%s'", name ? name : "(null)");
    *value = *slot;
    return FD_OK;
}

int fd_preprocess(fd_model* m, const uint8_t* frames, int n, int src_w, int src_h, int on_device, int allow_resize, void* stream) {
    if (!m || !frames) return fail(FD_ERR_ARG, "fd_preprocess: null argument");
    const ModelPlan& P = m->plan;
    const bool same = src_w == P.net_w && src_h == P.net_h;
    if (!same && !allow_resize) return fail(FD_ERR_SIZE, "invalid image size");  // reference detector.py:132
    if (src_w < 1 || src_h < 1) return fail(FD_ERR_SIZE, "invalid image size");
    NEED_DEVICE(m);
    CU(cudaSetDevice(m->device));
    Exec* e;
    if (int rc = get_exec(m, n, &e)) return rc;
    cudaStream_t s = pick(m, stream);
    const size_t bytes = size_t(n) * src_w * src_h * 3;
    const cudaMemcpyKind kind = on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice;
    if (same) {
        CU(cudaMemcpyAsync(e->frames, frames, bytes, kind, s));
    } else {
        const uint8_t* src = frames;
        if (!on_device) {
            if (e->src_cap < bytes) {
                DEVICE_SETUP_LOCK(m);
                if (int rc = sync_model_streams(m)) return rc;
                cudaFree(e->src); e->src = nullptr; e->src_cap = 0;
                CU(cudaMalloc(&e->src, bytes));
                e->src_cap = bytes;
            }
            CU(cudaMemcpyAsync(e->src, frames, bytes, cudaMemcpyHostToDevice, s));
            src = e->src;
        }
        if (launch_letterbox_u8(src, e->frames, n, src_h, src_w, P.net_h, P.net_w, 128, s))
            return fail(FD_ERR_CUDA, "letterbox launch failed: %s", cudaGetErrorString(cudaGetLastError()));
    }
    return FD_OK;
}

// the layers from `from_layer` on as an instantiated CUDA graph (nullptr if capture is not possible: callers then launch directly)
static cudaGraphExec_t capture_layers(fd_model* m, Exec* e, int from_layer) {
    DEVICE_SETUP_LOCK(m);
    cudaGraph_t graph = nullptr;
    cudaGraphExec_t exec = nullptr;
    if (cudaStreamBeginCapture(m->stream, cudaStreamCaptureModeThreadLocal) == cudaSuccess) {
        const int rc = launch_layers(m, e, m->stream, from_layer);
        const cudaError_t ce = cudaStreamEndCapture(m->stream, &graph);
        if (rc == FD_OK && ce == cudaSuccess && graph) {
            if (cudaGraphInstantiate(&exec, graph, 0) != cudaSuccess) exec = nullptr;
        }
        if (graph) cudaGraphDestroy(graph);
    }
    cudaGetLastError();
    return exec;
}

int fd_forward(fd_model* m, int n, void* stream) {
    if (!m) return fail(FD_ERR_ARG, "fd_forward: null model");
    NEED_DEVICE(m);
    CU(cudaSetDevice(m->device));
    Exec* e;
    if (int rc = get_exec(m, n, &e)) return rc;
    cudaStream_t s = pick(m, stream);
    m->last_n = n;
    if (!e->graph_tried) {
        e->graph_tried = true;
        e->graph = capture_layers(m, e, 0);
    }
    if (e->graph) {
        CU(cudaGraphLaunch(e->graph, s));
        return FD_OK;
    }
    return launch_layers(m, e, s);
}

// The batch's thresholds thr[n] (host) and their objectness cuts, through slot T's pinned area into the Exec's thr array on
// stream s (ahead of decode).  Pinned contents an earlier copy may still be reading are rewritten only after that copy has run;
// a repeat at the same thresholds (fd_postprocess in a loop) rewrites nothing and never waits.
static int stage_thresholds(fd_model* m, Exec* e, Slot& T, int n, const double* thr, cudaStream_t s) {
    const size_t bytes = (sizeof(double) + sizeof(float)) * size_t(n);
    if (!T.thr_copied) {
        DEVICE_SETUP_LOCK(m);
        CU(cudaEventCreateWithFlags(&T.thr_copied, cudaEventDisableTiming));
    }
    if (T.thr_n != n || memcmp(T.h_thr, thr, sizeof(double) * size_t(n)) != 0) {
        CU(cudaEventSynchronize(T.thr_copied));
        if (T.h_thr_cap < bytes) {
            DEVICE_SETUP_LOCK(m);
            if (T.h_thr) cudaFreeHost(T.h_thr);
            T.h_thr = nullptr; T.h_thr_cap = 0; T.thr_n = 0;
            CU(cudaMallocHost(&T.h_thr, bytes));
            T.h_thr_cap = bytes;
        }
        double* h = reinterpret_cast<double*>(T.h_thr);
        float* cut = reinterpret_cast<float*>(h + n);
        for (int f = 0; f < n; ++f) { h[f] = thr[f]; cut[f] = obj_cut_for(thr[f]); }
        T.thr_n = n;
    }
    CU(cudaMemcpyAsync(e->thr, T.h_thr, bytes, cudaMemcpyHostToDevice, s));
    CU(cudaEventRecord(T.thr_copied, s));
    return FD_OK;
}

// decode + Soft-NMS on the head tensors, frame f at threshold thr[f] (host array, staged through slot T), then the records to
// pinned host memory (h_dets / h_count) on stream s
static int postprocess_on(fd_model* m, Exec* e, Slot& T, int n, const double* thr, int max_det, cudaStream_t s, Detection* h_dets,
                          int* h_count) {
    const fd_info& I = m->info;
    if (int rc = stage_thresholds(m, e, T, n, thr, s)) return rc;
    const double* d_thr = e->thr;
    const float* d_cut = reinterpret_cast<const float*>(e->thr + n);
    HeadDesc heads[FD_MAX_HEADS];
    int first = 0;
    for (int h = 0; h < I.n_heads; ++h) {
        const LayerPlan& L = m->plan.layers[m->plan.head_layers[h]];
        heads[h].data = static_cast<const float*>(loc_ptr(*e, m->plan, L.out, true));
        heads[h].pitch = L.out.pitch; heads[h].h = L.out.h; heads[h].w = L.out.w;
        heads[h].first_box = first;
        first += 3 * L.out.h * L.out.w;
        for (int k = 0; k < 3; ++k) { heads[h].anchor_w[k] = I.anchors[h][k][0]; heads[h].anchor_h[k] = I.anchors[h][k][1]; }
    }
    if (launch_decode(heads, I.n_heads, I.num_classes, n, I.net_w, I.net_h, d_thr, d_cut, e->cand, e->cand_count, I.boxes_per_frame, s))
        return fail(FD_ERR_CUDA, "decode launch failed: %s", cudaGetErrorString(cudaGetLastError()));
    if (launch_soft_nms(e->cand, e->cand_count, e->scores, I.boxes_per_frame, n, I.net_w, I.net_h, d_thr, e->dets,
                        e->det_count, e->det_count + n, max_det, s))
        return fail(FD_ERR_CUDA, "soft-nms launch failed: %s", cudaGetErrorString(cudaGetLastError()));
    CU(cudaMemcpyAsync(h_count, e->det_count, sizeof(int) * 2 * n, cudaMemcpyDeviceToHost, s));
    CU(cudaMemcpyAsync(h_dets, e->dets, sizeof(Detection) * size_t(n) * max_det, cudaMemcpyDeviceToHost, s));
    return FD_OK;
}

int fd_postprocess(fd_model* m, int n, double threshold, int max_det, void* stream) {
    if (!m) return fail(FD_ERR_ARG, "fd_postprocess: null model");
    if (n < 1) return fail(FD_ERR_ARG, "batch size must be positive (got %d)", n);
    const std::vector<double> thr(n, threshold);
    return fd_postprocess_thresholds(m, n, thr.data(), max_det, stream);
}

int fd_postprocess_thresholds(fd_model* m, int n, const double* thresholds, int max_det, void* stream) {
    if (!m || !thresholds) return fail(FD_ERR_ARG, "fd_postprocess: null argument");
    const fd_info& I = m->info;
    if (I.n_heads != 2 && I.n_heads != 3) return fail(FD_ERR_HEADS, "%d", I.n_heads);  // KeyError(len(outputs)) in the reference
    if (max_det < 1) return fail(FD_ERR_ARG, "max_det must be >= 1");
    NEED_DEVICE(m);
    CU(cudaSetDevice(m->device));
    Exec* e;
    if (int rc = get_exec(m, n, &e)) return rc;
    cudaStream_t s = pick(m, stream);
    if (e->max_det != max_det || !e->h_dets) {
        DEVICE_SETUP_LOCK(m);
        if (int rc = sync_model_streams(m)) return rc;  // (rare) the record buffers may be in use on the compute or the copy stream
        cudaFree(e->dets); e->dets = nullptr;
        if (e->h_dets) { cudaFreeHost(e->h_dets); e->h_dets = nullptr; }
        CU(cudaMalloc(&e->dets, sizeof(Detection) * size_t(e->n) * max_det));
        CU(cudaMallocHost(&e->h_dets, sizeof(Detection) * size_t(e->n) * max_det));
        e->max_det = max_det;
    }
    // results to pinned host memory on the same stream; fd_fetch synchronises
    if (int rc = postprocess_on(m, e, m->slots[FD_MAX_SLOTS], n, thresholds, max_det, s, e->h_dets, e->h_count)) return rc;
    m->last_n = n;
    m->last_max_det = max_det;
    return FD_OK;
}

int fd_fetch(fd_model* m, int n, fd_det* out, int32_t* counts, int32_t* total, void* stream) {
    if (!m || !out || !counts) return fail(FD_ERR_ARG, "fd_fetch: null argument");
    auto it = m->execs.find(bucket_of(n));
    if (n < 1 || it == m->execs.end() || !it->second->h_dets)
        return fail(FD_ERR_ARG, "fd_fetch: no postprocess results for batch %d", n);
    Exec* e = it->second.get();
    NEED_DEVICE(m);
    CU(cudaSetDevice(m->device));
    CU(cudaStreamSynchronize(pick(m, stream)));
    const int md = m->last_max_det;
    for (int f = 0; f < n; ++f) {
        counts[f] = e->h_count[f];
        if (total) total[f] = e->h_count[n + f];
        memcpy(out + size_t(f) * md, e->h_dets + size_t(f) * md, sizeof(fd_det) * size_t(e->h_count[f]));
    }
    return FD_OK;
}

// fd_detect with host frames of the network's own size: the synchronous call used to pay the whole PCIe copy (33 MB,
// 0.66 ms at batch 64) in front of every batch.  Here the copy is cut into four pieces on the copy stream, and the layers
// in front of the second down-sampling layer (YOLOv3: conv1..conv4, the 416 / 208 stages: 0.8 ms) run quarter by quarter,
// each quarter behind the piece that carries its frames, so all but the first piece hides behind them.  The rest of the
// network follows as one captured graph.  Same kernels on the same frames: results are those of the plain path bit for bit.
static int build_overlap_plan(fd_model* m, Exec* e) {
    const ModelPlan& P = m->plan;
    e->ov_layers = -1;
    if (e->n < 16 || e->n % 4) return FD_OK;
    int downs = 0, depth = 0;
    for (size_t i = 0; i < P.layers.size(); ++i) {
        const LayerPlan& L = P.layers[i];
        const bool down = (L.kind == LAYER_CONV && L.stride == 2) || (L.kind == LAYER_MAXPOOL && L.pool_s == 2) || L.pool2;
        if (down && ++downs == 2) break;
        if (L.out_fp32 || L.upsample2x || L.kind == LAYER_COPY) return FD_OK;
        // every tensor these layers touch must be written inside the front (or be the input frames): nothing may reach back
        depth = static_cast<int>(i) + 1;
    }
    if (downs < 2 || depth < 1 || P.layers[0].kind != LAYER_CONV0) return FD_OK;
    const int quarter = e->n / 4;
    // a fused pair must lie inside the front or behind it, and take quarter batches (as it does for every shape the
    // whole-batch plan fused); otherwise leave the plain path
    if (e->use_stem && (depth < 2 || !conv_stem_supported(stem_desc(m, quarter)))) return FD_OK;
    const int bl = e->block_layer;
    if (bl >= 0 && bl < depth && (bl + 1 >= depth || !conv_block_supported(block_desc(m, bl, quarter)))) return FD_OK;
    if (int rc = prepare_set(m, e, depth, 4, quarter, &e->front)) return rc;
    if (e->front.ws_bytes) return FD_OK;  // (a split-K layer this early would need its own workspace: leave the plain path)
    e->ov_layers = depth;
    return FD_OK;
}

static int forward_overlapping_copy(fd_model* m, Exec* e, const uint8_t* frames, int n) {
    const ModelPlan& P = m->plan;
    cudaStream_t s = m->stream;
    if (!m->copy_stream) CU(cudaStreamCreateWithFlags(&m->copy_stream, cudaStreamNonBlocking));
    if (!m->idle_ev) {
        CU(cudaEventCreateWithFlags(&m->idle_ev, cudaEventDisableTiming));
        for (cudaEvent_t& ev : m->h2d_ev) CU(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
    }
    const size_t frame_bytes = size_t(P.net_h) * P.net_w * 3;
    const int quarter = e->front.frames;
    // everything queued on the compute stream so far (a previous pass that reads this input tensor) comes first
    CU(cudaEventRecord(m->idle_ev, s));
    CU(cudaStreamWaitEvent(m->copy_stream, m->idle_ev, 0));
    for (int p = 0; p < 4; ++p) {
        const int f0 = p * quarter, f1 = std::min(n, f0 + quarter);
        if (f1 > f0) CU(cudaMemcpyAsync(e->frames + f0 * frame_bytes, frames + f0 * frame_bytes, (f1 - f0) * frame_bytes, cudaMemcpyHostToDevice, m->copy_stream));
        CU(cudaEventRecord(m->h2d_ev[p], m->copy_stream));
    }
    for (int k = 0; k < 4; ++k) {
        CU(cudaStreamWaitEvent(s, m->h2d_ev[k], 0));
        for (int i = 0; i < e->ov_layers; ++i)
            if (int rc = launch_piece(m, e, e->front, i, k, s)) return rc;
    }
    if (!e->graph_tail_tried) {
        e->graph_tail_tried = true;
        e->graph_tail = capture_layers(m, e, e->ov_layers);
    }
    m->last_n = n;
    if (e->graph_tail) {
        CU(cudaGraphLaunch(e->graph_tail, s));
        return FD_OK;
    }
    return launch_layers(m, e, s, e->ov_layers);
}

int fd_detect(fd_model* m, const uint8_t* frames, int n, int src_w, int src_h, int on_device, int allow_resize,
              double threshold, int max_det, fd_det* out, int32_t* counts) {
    if (m && frames && m->device >= 0 && !on_device && src_w == m->plan.net_w && src_h == m->plan.net_h) {
        CU(cudaSetDevice(m->device));
        Exec* e;
        if (int rc = get_exec(m, n, &e)) return rc;
        if (e->ov_layers == 0)
            if (int rc = build_overlap_plan(m, e)) return rc;
        if (e->ov_layers > 0) {
            if (int rc = forward_overlapping_copy(m, e, frames, n)) return rc;
            if (int rc = fd_postprocess(m, n, threshold, max_det, nullptr)) return rc;
            return fd_fetch(m, n, out, counts, nullptr, nullptr);
        }
    }
    if (int rc = fd_preprocess(m, frames, n, src_w, src_h, on_device, allow_resize, nullptr)) return rc;
    if (int rc = fd_forward(m, n, nullptr)) return rc;
    if (int rc = fd_postprocess(m, n, threshold, max_det, nullptr)) return rc;
    return fd_fetch(m, n, out, counts, nullptr, nullptr);
}

namespace {

// A submit that fails after it has queued work (a copy from the slot's pinned staging buffer, kernels on its tensors)
// leaves the slot free (busy stays false): the queued work must have drained before the caller can reuse the slot's
// buffers.  The error text of the failing call is kept.
int quiesce_after_failure(fd_model* m, int rc) {
    char keep[sizeof(g_err)];
    memcpy(keep, g_err, sizeof(keep));
    if (m->copy_stream) cudaStreamSynchronize(m->copy_stream);
    if (m->stream) cudaStreamSynchronize(m->stream);
    cudaGetLastError();
    memcpy(g_err, keep, sizeof(keep));
    return rc;
}

int slot_begin_resize(fd_model* m, Exec* e, Slot& S, int n, int max_det, Exec** e_out, Slot** s_out);

// common front of fd_submit / fd_submit_jpeg: argument checks, the Exec of this batch size, the slot's events and
// pinned result buffers
int slot_begin(fd_model* m, int slot, int n, int max_det, Exec** e_out, Slot** s_out) {
    const fd_info& I = m->info;
    if (I.n_heads != 2 && I.n_heads != 3) return fail(FD_ERR_HEADS, "%d", I.n_heads);
    if (max_det < 1) return fail(FD_ERR_ARG, "max_det must be >= 1");
    NEED_DEVICE(m);
    CU(cudaSetDevice(m->device));
    Slot& S = m->slots[slot];
    if (S.busy) return fail(FD_ERR_ARG, "slot %d still holds uncollected results", slot);
    Exec* e;
    if (int rc = get_exec(m, n, &e)) return rc;
    if (!m->copy_stream || !S.staged) {
        DEVICE_SETUP_LOCK(m);
        if (!m->copy_stream) CU(cudaStreamCreateWithFlags(&m->copy_stream, cudaStreamNonBlocking));
        if (!S.staged) {
            CU(cudaEventCreateWithFlags(&S.staged, cudaEventDisableTiming));
            CU(cudaEventCreateWithFlags(&S.stage_free, cudaEventDisableTiming));
            CU(cudaEventCreateWithFlags(&S.done, cudaEventDisableTiming));
        }
    }
    if (S.h_dets_cap < sizeof(Detection) * size_t(n) * max_det || S.h_count_cap < sizeof(int) * 2 * size_t(n) || e->max_det != max_det) {
        DEVICE_SETUP_LOCK(m);
        return slot_begin_resize(m, e, S, n, max_det, e_out, s_out);
    }
    *e_out = e;
    *s_out = &S;
    return FD_OK;
}

// (rare) the slot's pinned result buffers or the Exec's record buffer have to grow: under the device's set-up lock
int slot_begin_resize(fd_model* m, Exec* e, Slot& S, int n, int max_det, Exec** e_out, Slot** s_out) {
    const size_t det_bytes = sizeof(Detection) * size_t(n) * max_det, cnt_bytes = sizeof(int) * 2 * size_t(n);
    if (S.h_dets_cap < det_bytes) {
        if (S.h_dets) cudaFreeHost(S.h_dets);
        S.h_dets = nullptr; S.h_dets_cap = 0;
        CU(cudaMallocHost(&S.h_dets, det_bytes));
        S.h_dets_cap = det_bytes;
    }
    if (S.h_count_cap < cnt_bytes) {
        if (S.h_count) cudaFreeHost(S.h_count);
        S.h_count = nullptr; S.h_count_cap = 0;
        CU(cudaMallocHost(&S.h_count, cnt_bytes));
        S.h_count_cap = cnt_bytes;
    }
    if (e->max_det != max_det) {
        if (int rc = sync_model_streams(m)) return rc;  // the record buffers may be in use on the compute or the copy stream
        cudaFree(e->dets); e->dets = nullptr;
        if (e->h_dets) { cudaFreeHost(e->h_dets); e->h_dets = nullptr; }
        CU(cudaMalloc(&e->dets, sizeof(Detection) * size_t(e->n) * max_det));
        e->max_det = max_det;
    }
    *e_out = e;
    *s_out = &S;
    return FD_OK;
}

int slot_stage_reserve(fd_model* m, Slot& S, size_t bytes) {
    if (S.stage_cap >= bytes) return FD_OK;
    DEVICE_SETUP_LOCK(m);
    if (int rc = sync_model_streams(m)) return rc;
    cudaFree(S.stage); S.stage = nullptr; S.stage_cap = 0;
    CU(cudaMalloc(&S.stage, bytes));
    S.stage_cap = bytes;
    return FD_OK;
}

// common tail: the conv stack, decode + Soft-NMS (frame f at threshold thr[f]), results into the slot's pinned buffers, the
// `done` event
int slot_finish(fd_model* m, Exec* e, Slot& S, int n, const double* thr, int max_det) {
    cudaStream_t s = m->stream;
    if (int rc = fd_forward(m, n, nullptr)) return rc;
    if (int rc = postprocess_on(m, e, S, n, thr, max_det, s, S.h_dets, S.h_count)) return rc;
    CU(cudaEventRecord(S.done, s));
    S.n = n; S.max_det = max_det; S.busy = true;
    return FD_OK;
}

int slot_collect(fd_model* m, Slot& S, fd_det* out, int32_t* counts, int32_t* total) {
    CU(cudaSetDevice(m->device));
    S.busy = false;
    CU(cudaEventSynchronize(S.done));
    for (int f = 0; f < S.n; ++f) {
        counts[f] = S.h_count[f];
        if (total) total[f] = S.h_count[S.n + f];
        memcpy(out + size_t(f) * S.max_det, S.h_dets + size_t(f) * S.max_det, sizeof(fd_det) * size_t(S.h_count[f]));
    }
    return FD_OK;
}

// ------------------------------------------------------------------ JPEG front end (jpeg.h)
// Host half of a JPEG batch: parse + entropy-decode every frame (one frame per pool thread) into the slot's pinned
// buffer, laid out as [JpegFrameDev x n][coefficients of frame 0][frame 1]...  Fills status[] (FD_JPEG_*).
int jpeg_host_stage(fd_model* m, Slot& S, const uint8_t* const* data, const size_t* lens, int n, int allow_resize, int32_t* status,
                    size_t* bytes_out, int* max_blocks_out, int* src_w, int* src_h) {
    const ModelPlan& P = m->plan;
    if (!m->jpeg_pool) {
        int t = options().jpeg_threads > 0 ? options().jpeg_threads : static_cast<int>(std::thread::hardware_concurrency());
        m->jpeg_pool.reset(new JpegPool(std::max(1, std::min(t, 64))));
    }
    std::vector<JpegInfo>& info = m->jpeg_info;
    if (info.size() < size_t(n)) info.resize(n);
    std::vector<int32_t> local(n, 0);
    int32_t* st = status ? status : local.data();
    std::vector<std::string> why(n);
    m->jpeg_pool->run(n, [&](int i) {
        char buf[160] = "";
        st[i] = jpeg_parse(data[i], lens[i], &info[i], buf, sizeof(buf));
        why[i] = buf;
    });
    // frame size: the network's (reference detector.py:131-132) or, with allow_resize, any one size for the whole batch
    int want_w = P.net_w, want_h = P.net_h;
    if (allow_resize)
        for (int i = 0; i < n; ++i)
            if (st[i] == JPEG_OK) { want_w = info[i].width; want_h = info[i].height; break; }
    if (want_w > 8192 || want_h > 8192) { want_w = P.net_w; want_h = P.net_h; }  // bounds the staging memory
    for (int i = 0; i < n; ++i)
        if (st[i] == JPEG_OK && (info[i].width != want_w || info[i].height != want_h)) {
            st[i] = FD_JPEG_SIZE;
            char buf[64];
            snprintf(buf, sizeof(buf), "%dx%d", info[i].width, info[i].height);
            why[i] = buf;
        }
    *src_w = want_w;
    *src_h = want_h;
    bool only_size = true;
    int bad = -1;
    for (int i = n - 1; i >= 0; --i)
        if (st[i] != JPEG_OK) { bad = i; only_size = only_size && st[i] == FD_JPEG_SIZE; }
    if (bad >= 0) {
        if (only_size) return fail(FD_ERR_SIZE, "invalid image size");  // reference detector.py:132
        return fail(FD_ERR_JPEG, "frame %d: %s (status %d)", bad, why[bad].c_str(), st[bad]);
    }
    const size_t head = jpeg_head_bytes(n);
    std::vector<size_t> off(n + 1);
    off[0] = head;
    int max_blocks = 0;
    for (int i = 0; i < n; ++i) {
        const size_t count = jpeg_coef_count(info[i]);
        off[i + 1] = off[i] + count * sizeof(int16_t);
        max_blocks = std::max(max_blocks, static_cast<int>(count / 64));
    }
    if (off[n] > 0xffffffffull * 2) return fail(FD_ERR_ARG, "JPEG batch too large");
    if (S.h_stage_cap < off[n]) {
        DEVICE_SETUP_LOCK(m);
        if (S.h_stage) {
            CU(cudaStreamSynchronize(m->copy_stream));
            cudaFreeHost(S.h_stage);
        }
        S.h_stage = nullptr; S.h_stage_cap = 0;
        CU(cudaMallocHost(&S.h_stage, off[n] + off[n] / 4));
        S.h_stage_cap = off[n] + off[n] / 4;
    }
    char* base = S.h_stage;
    m->jpeg_pool->run(n, [&](int i) {
        char buf[160] = "";
        st[i] = jpeg_decode_coefficients(data[i], lens[i], info[i], reinterpret_cast<int16_t*>(base + off[i]), buf, sizeof(buf));
        why[i] = buf;
    });
    for (int i = 0; i < n; ++i)
        if (st[i] != JPEG_OK) return fail(FD_ERR_JPEG, "frame %d: %s (status %d)", i, why[i].c_str(), st[i]);
    JpegFrameDev* fr = reinterpret_cast<JpegFrameDev*>(base);
    for (int i = 0; i < n; ++i) jpeg_frame_desc(info[i], (off[i] - head) / sizeof(int16_t), &fr[i]);
    *bytes_out = off[n];
    *max_blocks_out = max_blocks;
    return FD_OK;
}

// byte ranges [first, second) of a pinned JPEG batch that hold descriptors or coefficients
using ByteRuns = std::vector<std::pair<size_t, size_t>>;

// Device half: the byte ranges `runs` of the pinned batch `src` -> the same offsets of the slot's device staging on the copy
// stream, then IDCT and colour conversion on the compute stream, ending with RGB u8 frames in the Exec's input tensor (where
// fd_preprocess would have put them).  The batch is [JpegFrameDev x n] from offset 0, coefficients from offset `head`.
int jpeg_device_stage(fd_model* m, Exec* e, Slot& S, const char* src, size_t head, const ByteRuns& runs, int n, int max_blocks,
                      int src_w, int src_h) {
    const ModelPlan& P = m->plan;
    if (int rc = slot_stage_reserve(m, S, runs.back().second)) return rc;
    const bool same = src_w == P.net_w && src_h == P.net_h;
    const size_t plane_stride = size_t(3) * ((src_w + 15) / 16 * 16) * ((src_h + 15) / 16 * 16);
    uint8_t* rgb = e->frames;
    if (!same) {  // decode at the source size, then the letterbox of fd_preprocess
        const size_t src_bytes = size_t(n) * src_w * src_h * 3;
        if (e->src_cap < src_bytes) {
            DEVICE_SETUP_LOCK(m);
            if (int rc = sync_model_streams(m)) return rc;
            cudaFree(e->src); e->src = nullptr; e->src_cap = 0;
            CU(cudaMalloc(&e->src, src_bytes));
            e->src_cap = src_bytes;
        }
        rgb = e->src;
    }
    if (m->jpeg_planes_cap < plane_stride * n) {
        DEVICE_SETUP_LOCK(m);
        if (int rc = sync_model_streams(m)) return rc;
        cudaFree(m->jpeg_planes); m->jpeg_planes = nullptr; m->jpeg_planes_cap = 0;
        CU(cudaMalloc(&m->jpeg_planes, plane_stride * n));
        m->jpeg_planes_cap = plane_stride * n;
    }
    cudaStream_t cs = m->copy_stream, s = m->stream;
    CU(cudaStreamWaitEvent(cs, S.stage_free, 0));
    for (const auto& r : runs) CU(cudaMemcpyAsync(S.stage + r.first, src + r.first, r.second - r.first, cudaMemcpyHostToDevice, cs));
    CU(cudaEventRecord(S.staged, cs));
    CU(cudaStreamWaitEvent(s, S.staged, 0));
    const JpegFrameDev* fr = reinterpret_cast<const JpegFrameDev*>(S.stage);
    const int16_t* coefs = reinterpret_cast<const int16_t*>(S.stage + head);
    if (launch_jpeg_idct(coefs, fr, m->jpeg_planes, plane_stride, n, max_blocks, s))
        return fail(FD_ERR_CUDA, "JPEG kernel launch failed: %s", cudaGetErrorString(cudaGetLastError()));
    if (launch_jpeg_rgb(m->jpeg_planes, plane_stride, fr, rgb, n, src_h, src_w, s))
        return fail(FD_ERR_CUDA, "JPEG kernel launch failed: %s", cudaGetErrorString(cudaGetLastError()));
    if (!same && launch_letterbox_u8(rgb, e->frames, n, src_h, src_w, P.net_h, P.net_w, 128, s))
        return fail(FD_ERR_CUDA, "letterbox launch failed: %s", cudaGetErrorString(cudaGetLastError()));
    CU(cudaEventRecord(S.stage_free, s));
    return FD_OK;
}

}  // namespace

// ------------------------------------------------------------------ pipelined serving: fd_submit / fd_collect
// Two (FD_MAX_SLOTS) batches can be in flight: the host->device copy of a slot runs on the model's copy stream while
// the compute stream works on the other slot, so a caller that alternates slots keeps the conv stack busy
// back to back (the synchronous fd_detect pays the PCIe copy in front of every batch).
int fd_submit(fd_model* m, int slot, const uint8_t* frames, int n, int src_w, int src_h, int on_device, int allow_resize,
              double threshold, int max_det) {
    if (!m || !frames) return fail(FD_ERR_ARG, "fd_submit: null argument");
    if (slot < 0 || slot >= FD_MAX_SLOTS) return fail(FD_ERR_ARG, "fd_submit: slot %d out of range [0, %d)", slot, FD_MAX_SLOTS);
    const ModelPlan& P = m->plan;
    const bool same = src_w == P.net_w && src_h == P.net_h;
    if (!same && !allow_resize) return fail(FD_ERR_SIZE, "invalid image size");  // reference detector.py:132
    if (src_w < 1 || src_h < 1) return fail(FD_ERR_SIZE, "invalid image size");
    Exec* e;
    Slot* sp;
    if (int rc = slot_begin(m, slot, n, max_det, &e, &sp)) return rc;
    Slot& S = *sp;
    const size_t bytes = size_t(n) * src_w * src_h * 3;
    if (int rc = slot_stage_reserve(m, S, bytes)) return rc;
    cudaStream_t cs = m->copy_stream, s = m->stream;
    // copy stream: wait until the compute stream has consumed this slot's previous contents, then stage the frames
    CU(cudaStreamWaitEvent(cs, S.stage_free, 0));
    CU(cudaMemcpyAsync(S.stage, frames, bytes, on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice, cs));
    CU(cudaEventRecord(S.staged, cs));
    // compute stream: staged frames -> the Exec's input tensor (33 MB device copy at bs64, ~10 us), then the batch
    CU(cudaStreamWaitEvent(s, S.staged, 0));
    if (same) {
        CU(cudaMemcpyAsync(e->frames, S.stage, bytes, cudaMemcpyDeviceToDevice, s));
    } else if (launch_letterbox_u8(S.stage, e->frames, n, src_h, src_w, P.net_h, P.net_w, 128, s)) {
        return fail(FD_ERR_CUDA, "letterbox launch failed: %s", cudaGetErrorString(cudaGetLastError()));
    }
    CU(cudaEventRecord(S.stage_free, s));
    const std::vector<double> thr(n, threshold);
    if (int rc = slot_finish(m, e, S, n, thr.data(), max_det)) return quiesce_after_failure(m, rc);
    return FD_OK;
}

int fd_collect(fd_model* m, int slot, fd_det* out, int32_t* counts, int32_t* total) {
    if (!m || !out || !counts) return fail(FD_ERR_ARG, "fd_collect: null argument");
    if (slot < 0 || slot >= FD_MAX_SLOTS) return fail(FD_ERR_ARG, "fd_collect: slot %d out of range [0, %d)", slot, FD_MAX_SLOTS);
    NEED_DEVICE(m);
    Slot& S = m->slots[slot];
    if (!S.busy) return fail(FD_ERR_ARG, "fd_collect: nothing was submitted to slot %d", slot);
    return slot_collect(m, S, out, counts, total);
}

}  // extern "C"

// library-internal (csrc/server.cc): submit a JPEG batch that the callers of fd_server_perform_jpeg have entropy-decoded
// into pinned memory, with frame f at threshold thresholds[f].  Layout: [JpegFrameDev x cap] from offset 0, frame i's
// coefficients from byte jpeg_head_bytes(cap) + i * stride.  Only the bytes the n frames use are copied.
int fd_internal_submit_jpeg(fd_model* m, int slot, const uint8_t* pinned, int n, int cap, size_t stride, const double* thresholds,
                            int max_det) {
    if (!m || !pinned || !thresholds || n < 1 || n > cap) return fail(FD_ERR_ARG, "fd_internal_submit_jpeg: bad argument");
    if (slot < 0 || slot >= FD_MAX_SLOTS) return fail(FD_ERR_ARG, "fd_internal_submit_jpeg: slot %d out of range [0, %d)", slot, FD_MAX_SLOTS);
    const size_t head = jpeg_head_bytes(cap);
    const JpegFrameDev* fr = reinterpret_cast<const JpegFrameDev*>(pinned);
    ByteRuns runs{{0, sizeof(JpegFrameDev) * size_t(n)}};
    int max_blocks = 0;
    for (int i = 0; i < n; ++i) {
        int blocks = 0;
        for (int c = 0; c < 3; ++c) blocks += fr[i].bw[c] * fr[i].bh[c];
        max_blocks = std::max(max_blocks, blocks);
        const size_t o = head + stride * i, end = o + size_t(blocks) * 64 * sizeof(int16_t);
        if (runs.back().second == o) runs.back().second = end;
        else runs.push_back({o, end});
    }
    Exec* e;
    Slot* sp;
    if (int rc = slot_begin(m, slot, n, max_det, &e, &sp)) return rc;
    if (int rc = jpeg_device_stage(m, e, *sp, reinterpret_cast<const char*>(pinned), head, runs, n, max_blocks, m->plan.net_w, m->plan.net_h))
        return quiesce_after_failure(m, rc);
    if (int rc = slot_finish(m, e, *sp, n, thresholds, max_det)) return quiesce_after_failure(m, rc);
    return FD_OK;
}

extern "C" {

// ------------------------------------------------------------------ JPEG in: reference detector.py:128-133
int fd_jpeg_probe(const uint8_t* data, size_t len, fd_jpeg_info* out) {
    if (!data || !out) return fail(FD_ERR_ARG, "fd_jpeg_probe: null argument");
    std::unique_ptr<JpegInfo> J(new JpegInfo());
    char why[160] = "";
    memset(out, 0, sizeof(*out));
    out->status = jpeg_parse(data, len, J.get(), why, sizeof(why));
    snprintf(out->reason, sizeof(out->reason), "%s", why);
    out->width = J->width; out->height = J->height; out->components = J->ncomp;
    if (out->status != JPEG_OK) return FD_OK;
    out->h_samp = J->hs; out->v_samp = J->vs; out->restart_interval = J->restart_interval;
    for (int c = 0; c < 3; ++c) {
        out->blocks_w[c] = J->bw[c];
        out->blocks_h[c] = J->bh[c];
        memcpy(out->quant[c], J->q[c], sizeof(out->quant[c]));
    }
    out->coef_count = static_cast<int64_t>(jpeg_coef_count(*J));
    return FD_OK;
}

int fd_jpeg_coefficients(const uint8_t* data, size_t len, int16_t* coefs, size_t cap, fd_jpeg_info* out) {
    if (!coefs) return fail(FD_ERR_ARG, "fd_jpeg_coefficients: null argument");
    if (int rc = fd_jpeg_probe(data, len, out)) return rc;
    if (out->status != JPEG_OK) return fail(FD_ERR_JPEG, "%s (status %d)", out->reason, out->status);
    if (cap < size_t(out->coef_count)) return fail(FD_ERR_ARG, "fd_jpeg_coefficients: buffer holds %zu coefficients, %lld needed", cap, static_cast<long long>(out->coef_count));
    std::unique_ptr<JpegInfo> J(new JpegInfo());
    char why[160] = "";
    jpeg_parse(data, len, J.get(), why, sizeof(why));
    out->status = jpeg_decode_coefficients(data, len, *J, coefs, why, sizeof(why));
    snprintf(out->reason, sizeof(out->reason), "%s", why);
    if (out->status != JPEG_OK) return fail(FD_ERR_JPEG, "%s (status %d)", why, out->status);
    return FD_OK;
}

int fd_decode_jpeg(fd_model* m, const uint8_t* const* data, const size_t* lens, int n, int allow_resize, int32_t* status,
                   uint8_t* rgb_out) {
    if (!m || !data || !lens) return fail(FD_ERR_ARG, "fd_decode_jpeg: null argument");
    NEED_DEVICE(m);
    CU(cudaSetDevice(m->device));
    Slot& S = m->slots[FD_MAX_SLOTS];
    Exec* e;
    if (int rc = get_exec(m, n, &e)) return rc;
    if (!m->copy_stream) CU(cudaStreamCreateWithFlags(&m->copy_stream, cudaStreamNonBlocking));
    if (!S.staged) {
        CU(cudaEventCreateWithFlags(&S.staged, cudaEventDisableTiming));
        CU(cudaEventCreateWithFlags(&S.stage_free, cudaEventDisableTiming));
        CU(cudaEventCreateWithFlags(&S.done, cudaEventDisableTiming));
    }
    size_t bytes = 0;
    int max_blocks = 0, sw = 0, sh = 0;
    if (int rc = jpeg_host_stage(m, S, data, lens, n, allow_resize, status, &bytes, &max_blocks, &sw, &sh)) return rc;
    if (int rc = jpeg_device_stage(m, e, S, S.h_stage, jpeg_head_bytes(n), ByteRuns{{0, bytes}}, n, max_blocks, sw, sh)) return rc;
    if (rgb_out) CU(cudaMemcpyAsync(rgb_out, e->frames, size_t(n) * m->plan.net_w * m->plan.net_h * 3, cudaMemcpyDeviceToHost, m->stream));
    CU(cudaStreamSynchronize(m->stream));
    return FD_OK;
}

int fd_submit_jpeg(fd_model* m, int slot, const uint8_t* const* data, const size_t* lens, int n, int allow_resize, double threshold,
                   int max_det, int32_t* status) {
    if (!m || !data || !lens) return fail(FD_ERR_ARG, "fd_submit_jpeg: null argument");
    if (slot < 0 || slot >= FD_MAX_SLOTS) return fail(FD_ERR_ARG, "fd_submit_jpeg: slot %d out of range [0, %d)", slot, FD_MAX_SLOTS);
    Exec* e;
    Slot* sp;
    if (int rc = slot_begin(m, slot, n, max_det, &e, &sp)) return rc;
    size_t bytes = 0;
    int max_blocks = 0, sw = 0, sh = 0;
    if (int rc = jpeg_host_stage(m, *sp, data, lens, n, allow_resize, status, &bytes, &max_blocks, &sw, &sh)) return rc;  // nothing queued yet
    if (int rc = jpeg_device_stage(m, e, *sp, sp->h_stage, jpeg_head_bytes(n), ByteRuns{{0, bytes}}, n, max_blocks, sw, sh)) return quiesce_after_failure(m, rc);
    const std::vector<double> thr(n, threshold);
    if (int rc = slot_finish(m, e, *sp, n, thr.data(), max_det)) return quiesce_after_failure(m, rc);
    return FD_OK;
}

int fd_detect_jpeg(fd_model* m, const uint8_t* const* data, const size_t* lens, int n, int allow_resize, double threshold, int max_det,
                   fd_det* out, int32_t* counts, int32_t* status) {
    if (!m || !data || !lens || !out || !counts) return fail(FD_ERR_ARG, "fd_detect_jpeg: null argument");
    Exec* e;
    Slot* sp;
    if (int rc = slot_begin(m, FD_MAX_SLOTS, n, max_det, &e, &sp)) return rc;
    size_t bytes = 0;
    int max_blocks = 0, sw = 0, sh = 0;
    if (int rc = jpeg_host_stage(m, *sp, data, lens, n, allow_resize, status, &bytes, &max_blocks, &sw, &sh)) return rc;  // nothing queued yet
    if (int rc = jpeg_device_stage(m, e, *sp, sp->h_stage, jpeg_head_bytes(n), ByteRuns{{0, bytes}}, n, max_blocks, sw, sh)) return quiesce_after_failure(m, rc);
    const std::vector<double> thr(n, threshold);
    if (int rc = slot_finish(m, e, *sp, n, thr.data(), max_det)) return quiesce_after_failure(m, rc);
    return slot_collect(m, *sp, out, counts, nullptr);
}

// ------------------------------------------------------------------ letterbox geometry (extension, SURVEY 8f rank 4)
int fd_letterbox_geometry(int src_w, int src_h, int net_w, int net_h, int32_t* new_w, int32_t* new_h, int32_t* off_x, int32_t* off_y) {
    if (src_w < 1 || src_h < 1 || net_w < 1 || net_h < 1 || !new_w || !new_h || !off_x || !off_y)
        return fail(FD_ERR_ARG, "fd_letterbox_geometry: bad argument");
    int nw, nh;  // the same integers launch_letterbox_u8 derives (pre.cu)
    if (1LL * src_w * net_h >= 1LL * src_h * net_w) {
        nw = net_w;
        nh = static_cast<int>((1LL * src_h * net_w + src_w / 2) / src_w);
        if (nh < 1) nh = 1;
    } else {
        nh = net_h;
        nw = static_cast<int>((1LL * src_w * net_h + src_h / 2) / src_h);
        if (nw < 1) nw = 1;
    }
    *new_w = nw; *new_h = nh; *off_x = (net_w - nw) / 2; *off_y = (net_h - nh) / 2;
    return FD_OK;
}

int fd_unmap_letterbox(fd_det* dets, int count, int src_w, int src_h, int net_w, int net_h) {
    if ((!dets && count > 0) || count < 0) return fail(FD_ERR_ARG, "fd_unmap_letterbox: bad argument");
    int32_t nw, nh, ox, oy;
    if (int rc = fd_letterbox_geometry(src_w, src_h, net_w, net_h, &nw, &nh, &ox, &oy)) return rc;
    const double sx = static_cast<double>(src_w) / nw, sy = static_cast<double>(src_h) / nh;
    for (int i = 0; i < count; ++i) {
        dets[i].x = (dets[i].x - ox) * sx;
        dets[i].y = (dets[i].y - oy) * sy;
        dets[i].w *= sx;
        dets[i].h *= sy;
    }
    return FD_OK;
}

// ------------------------------------------------------------------ wire format (reference server/server.py:234-239)
int fd_pack_wire(const fd_det* dets, int count, uint32_t reqid, uint32_t msec, int saturate, uint8_t* out, size_t cap, size_t* len) {
    if ((!dets && count > 0) || !out || !len || count < 0) return fail(FD_ERR_ARG, "fd_pack_wire: bad argument");
    const size_t need = 16 + 10 * static_cast<size_t>(count);
    if (cap < need) return fail(FD_ERR_ARG, "fd_pack_wire: buffer of %zu bytes, %zu needed", cap, need);
    auto be32 = [](uint8_t* p, uint32_t v) { p[0] = v >> 24; p[1] = (v >> 16) & 255; p[2] = (v >> 8) & 255; p[3] = v & 255; };
    memcpy(out, "YOLO", 4);
    be32(out + 4, reqid);
    be32(out + 8, msec);
    be32(out + 12, static_cast<uint32_t>(10 * count));
    uint8_t* r = out + 16;
    for (int i = 0; i < count; ++i, r += 10) {
        const fd_det& d = dets[i];
        long long v[6] = {d.klass, static_cast<long long>(d.conf * 255.0), static_cast<long long>(d.x), static_cast<long long>(d.y),
                          static_cast<long long>(d.w), static_cast<long long>(d.h)};  // (long long)double truncates toward zero like int()
        for (int k = 0; k < 6; ++k) {
            const long long lo = k < 2 ? 0 : -32768, hi = k < 2 ? 255 : 32767;
            if (v[k] < lo || v[k] > hi) {
                if (!saturate) return fail(FD_ERR_ARG, "fd_pack_wire: detection %d field %d = %lld does not fit the wire format", i, k, v[k]);
                v[k] = v[k] < lo ? lo : hi;
            }
        }
        r[0] = static_cast<uint8_t>(v[0]);
        r[1] = static_cast<uint8_t>(v[1]);
        for (int k = 0; k < 4; ++k) {
            const uint16_t u = static_cast<uint16_t>(static_cast<int16_t>(v[2 + k]));
            r[2 + 2 * k] = u >> 8;
            r[3 + 2 * k] = u & 255;
        }
    }
    *len = need;
    return FD_OK;
}

// ------------------------------------------------------------------ parity / profiling hooks
// `layer`: the layer that produces `t`.
// The output of a layer that is computed inside the next layer's kernel never exists during a forward pass; the hook for
// that tensor runs the layer's own kernel (the two-kernel path's, which the fused kernel is checked against) into a buffer
// allocated on demand.
static int launch_unfused(fd_model* m, Exec* e, int layer) {
    const LayerPlan& L = m->plan.layers[layer];
    if (L.kind == LAYER_CONV0) return launch_own(m, e, layer, 0, e->n, false, nullptr, nullptr, m->stream);
    ConvLaunch cl;
    HaloLaunch hl;
    char uh = 0;
    if (int rc = prepare_conv_layer(m, e, layer, e->n, 0, &cl, &hl, &uh)) return rc;
    if (!uh && cl.ws_bytes) return fail(FD_ERR_ARG, "layer %d: its unfused form would need a split-K workspace", layer);
    return launch_own(m, e, layer, 0, e->n, uh != 0, &cl, &hl, m->stream);
}

static int tensor_to_host_nchw(fd_model* m, Exec* e, int layer, const TensorLoc& t, bool fp32, float* dst, int n) {
    const size_t elems = size_t(n) * t.c * t.h * t.w;
    if (int rc = ensure_scratch(e, elems * 4)) return rc;
    if (e->fused_role[layer] == 1) {
        if (int rc = ensure_fused_away_buffer(m, e, layer)) return rc;
        if (int rc = launch_unfused(m, e, layer)) return rc;
    }
    if (launch_nhwc_to_nchw_f32(loc_ptr(*e, m->plan, t, fp32), t.pitch, fp32, e->scratch, n, t.h, t.w, t.c, m->stream))
        return fail(FD_ERR_CUDA, "layout kernel launch failed");
    CU(cudaMemcpyAsync(dst, e->scratch, elems * 4, cudaMemcpyDeviceToHost, m->stream));
    CU(cudaStreamSynchronize(m->stream));
    return FD_OK;
}

int fd_heads_fp32(fd_model* m, int head, float* dst, int n) {
    if (!m || !dst || head < 0 || head >= m->info.n_heads) return fail(FD_ERR_ARG, "fd_heads_fp32: bad argument");
    NEED_DEVICE(m);
    CU(cudaSetDevice(m->device));
    Exec* e;
    if (int rc = get_exec(m, n, &e)) return rc;
    CU(cudaDeviceSynchronize());
    return tensor_to_host_nchw(m, e, m->plan.head_layers[head], m->plan.layers[m->plan.head_layers[head]].out, true, dst, n);
}

int fd_set_heads_fp32(fd_model* m, int head, const float* src, int n) {
    if (!m || !src || head < 0 || head >= m->info.n_heads) return fail(FD_ERR_ARG, "fd_set_heads_fp32: bad argument");
    NEED_DEVICE(m);
    CU(cudaSetDevice(m->device));
    Exec* e;
    if (int rc = get_exec(m, n, &e)) return rc;
    const TensorLoc& t = m->plan.layers[m->plan.head_layers[head]].out;
    const size_t elems = size_t(n) * t.c * t.h * t.w;
    if (int rc = ensure_scratch(e, elems * 4)) return rc;
    CU(cudaDeviceSynchronize());
    // same stream as the layout kernel: a plain cudaMemcpy from pageable memory may return before its DMA lands
    CU(cudaMemcpyAsync(e->scratch, src, elems * 4, cudaMemcpyHostToDevice, m->stream));
    if (launch_nchw_to_rows_f32(e->scratch, static_cast<float*>(loc_ptr(*e, m->plan, t, true)), t.pitch, n, t.h, t.w, t.c, m->stream))
        return fail(FD_ERR_CUDA, "layout kernel launch failed");
    CU(cudaStreamSynchronize(m->stream));
    return FD_OK;
}

int fd_layer_output_fp32(fd_model* m, int layer, float* dst, int n) {
    if (!m || !dst || layer < 0 || layer >= static_cast<int>(m->plan.layers.size())) return fail(FD_ERR_ARG, "fd_layer_output_fp32: bad argument");
    NEED_DEVICE(m);
    CU(cudaSetDevice(m->device));
    Exec* e;
    if (int rc = get_exec(m, n, &e)) return rc;
    CU(cudaDeviceSynchronize());
    const LayerPlan& L = m->plan.layers[layer];
    return tensor_to_host_nchw(m, e, layer, L.out, L.out_fp32 != 0, dst, n);
}

int fd_normalise_f32(fd_model* m, const uint8_t* frames, int n, float* dst) {
    if (!m || !frames || !dst || n < 1) return fail(FD_ERR_ARG, "fd_normalise_f32: bad argument");
    NEED_DEVICE(m);
    CU(cudaSetDevice(m->device));
    const size_t px = size_t(n) * m->plan.net_h * m->plan.net_w;
    uint8_t* d_in = nullptr;
    float* d_out = nullptr;
    CU(cudaMalloc(&d_in, px * 3));
    if (cudaMalloc(&d_out, px * 3 * 4) != cudaSuccess) { cudaFree(d_in); return fail(FD_ERR_CUDA, "cudaMalloc failed"); }
    int rc = FD_OK;
    if (cudaMemcpyAsync(d_in, frames, px * 3, cudaMemcpyHostToDevice, m->stream) != cudaSuccess ||
        launch_normalise_f32_nchw(d_in, d_out, n, m->plan.net_h, m->plan.net_w, m->stream) ||
        cudaMemcpyAsync(dst, d_out, px * 3 * 4, cudaMemcpyDeviceToHost, m->stream) != cudaSuccess ||
        cudaStreamSynchronize(m->stream) != cudaSuccess)
        rc = fail(FD_ERR_CUDA, "fd_normalise_f32 failed: %s", cudaGetErrorString(cudaGetLastError()));
    cudaFree(d_in); cudaFree(d_out);
    return rc;
}

int fd_letterbox_u8(fd_model* m, const uint8_t* frames, int n, int src_w, int src_h, uint8_t* dst) {
    if (!m || !frames || !dst || n < 1 || src_w < 1 || src_h < 1) return fail(FD_ERR_ARG, "fd_letterbox_u8: bad argument");
    NEED_DEVICE(m);
    CU(cudaSetDevice(m->device));
    const size_t in_b = size_t(n) * src_w * src_h * 3, out_b = size_t(n) * m->plan.net_w * m->plan.net_h * 3;
    uint8_t *d_in = nullptr, *d_out = nullptr;
    CU(cudaMalloc(&d_in, in_b));
    if (cudaMalloc(&d_out, out_b) != cudaSuccess) { cudaFree(d_in); return fail(FD_ERR_CUDA, "cudaMalloc failed"); }
    int rc = FD_OK;
    if (cudaMemcpyAsync(d_in, frames, in_b, cudaMemcpyHostToDevice, m->stream) != cudaSuccess ||
        launch_letterbox_u8(d_in, d_out, n, src_h, src_w, m->plan.net_h, m->plan.net_w, 128, m->stream) ||
        cudaMemcpyAsync(dst, d_out, out_b, cudaMemcpyDeviceToHost, m->stream) != cudaSuccess ||
        cudaStreamSynchronize(m->stream) != cudaSuccess)
        rc = fail(FD_ERR_CUDA, "fd_letterbox_u8 failed: %s", cudaGetErrorString(cudaGetLastError()));
    cudaFree(d_in); cudaFree(d_out);
    return rc;
}

int fd_time_layers(fd_model* m, int n, int reps, float* ms) {
    if (!m || !ms || reps < 1) return fail(FD_ERR_ARG, "fd_time_layers: bad argument");
    NEED_DEVICE(m);
    CU(cudaSetDevice(m->device));
    Exec* e;
    if (int rc = get_exec(m, n, &e)) return rc;
    const int nl = static_cast<int>(m->plan.layers.size());
    cudaEvent_t e0, e1;
    CU(cudaEventCreate(&e0));
    CU(cudaEventCreate(&e1));
    if (int rc = launch_layers(m, e, m->stream)) return rc;  // warm-up, also fills every buffer
    CU(cudaStreamSynchronize(m->stream));
    for (int i = 0; i < nl; ++i) {  // each layer timed alone: reps back-to-back launches
        if (int rc = launch_piece(m, e, e->whole, i, 0, m->stream)) return rc;
        CU(cudaEventRecord(e0, m->stream));
        for (int r = 0; r < reps; ++r)
            if (int rc = launch_piece(m, e, e->whole, i, 0, m->stream)) return rc;
        CU(cudaEventRecord(e1, m->stream));
        CU(cudaStreamSynchronize(m->stream));
        float t = 0.f;
        CU(cudaEventElapsedTime(&t, e0, e1));
        ms[i] = t / reps;
    }
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    return FD_OK;
}

int fd_time_forward(fd_model* m, int n, int reps, float* ms) {
    if (!m || !ms || reps < 1) return fail(FD_ERR_ARG, "fd_time_forward: bad argument");
    NEED_DEVICE(m);
    CU(cudaSetDevice(m->device));
    cudaEvent_t e0, e1;
    CU(cudaEventCreate(&e0));
    CU(cudaEventCreate(&e1));
    for (int r = 0; r < 2; ++r)
        if (int rc = fd_forward(m, n, nullptr)) return rc;  // graph capture + warm-up
    CU(cudaEventRecord(e0, m->stream));
    for (int r = 0; r < reps; ++r)
        if (int rc = fd_forward(m, n, nullptr)) return rc;
    CU(cudaEventRecord(e1, m->stream));
    CU(cudaStreamSynchronize(m->stream));
    float t = 0.f;
    CU(cudaEventElapsedTime(&t, e0, e1));
    *ms = t / reps;
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    return FD_OK;
}

}  // extern "C"
