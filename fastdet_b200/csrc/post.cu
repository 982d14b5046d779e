// post.cu — YOLO head decode + threshold + compaction, and per-frame Gaussian Soft-NMS.
//
// Replaces the two pure-Python hot loops of the reference:
//   decode_kernel    : ONNXDetector.process_yolo, server/detector.py:148-166 (+ sigmoid :12-13)
//   soft_nms_kernel  : soft_nms :45-59 with YOLOObject.get_iou :38-42 / rect_intersect :15-22, and the
//                      pixel scaling of the result tuples :142-144
// All arithmetic is float64 in the reference (Python floats); it is float64 here too, in the same
// operation order, so decisions at the threshold agree except where exp() differs in its last bit.
//
// decode: one thread per box tests the objectness; only for a box that passes does its warp read the class logits
// (coalesced) for a first-maximum arg-max.
// Candidates are appended with an atomic per-frame counter and carry their insertion-order index `box`
// (head, row, column, anchor) — the order the reference's list/dict iteration has — so later tie-breaks
// do not depend on the append order.
#include <limits.h>
#include <math.h>
#include <stdlib.h>

#include "kernels.h"
#include "options.h"

namespace fd {

struct DecodeParams {
    HeadDesc heads[4];
    int cell_start[5];  // prefix sum of h*w per head
    int n_heads, num_classes, n, net_w, net_h, boxes_per_frame;
    const double* thr;     // [n] the frame's threshold
    const float* obj_cut;  // [n] objectness logits below this cannot reach the frame's threshold (obj_cut_for)
};

float obj_cut_for(double threshold) {  // logit(threshold) minus a safety margin; -inf: no pre-test
    return (threshold > 0.0 && threshold < 1.0) ? static_cast<float>(log(threshold / (1.0 - threshold)) - 1e-3) : -INFINITY;
}

__device__ __forceinline__ double logistic(float v) { return 1.0 / (1.0 + exp(-static_cast<double>(v))); }

// One thread per box for the objectness test (a warp's 32 loads are in flight together; with a warp per cell only three
// were, and the kernel crawled at 1 TB/s of sector traffic); boxes that pass are then finished by the whole warp, one
// after another: coalesced class logits, first-maximum arg-max by shuffles, the float64 box math on the owning lane.
__global__ void __launch_bounds__(256)
decode_kernel(const DecodeParams p, Candidate* __restrict__ cand, int* __restrict__ cand_count) {
    const int lane = threadIdx.x & 31;
    const long long gid = blockIdx.x * 256LL + threadIdx.x;
    const int bpf = p.boxes_per_frame;  // 3 boxes per cell, heads in order: also the insertion order of the reference
    const int span = 5 + p.num_classes;
    const bool live = gid < 1LL * p.n * bpf;
    const int f = live ? static_cast<int>(gid / bpf) : 0;
    const int b = live ? static_cast<int>(gid - 1LL * f * bpf) : 0;

    auto locate = [&](int frame, int box, int& hi, int& cell, int& k) -> const float* {
        const int cell_all = box / 3;
        k = box - 3 * cell_all;
        hi = 0;
        while (hi + 1 < p.n_heads && cell_all >= p.cell_start[hi + 1]) ++hi;
        cell = cell_all - p.cell_start[hi];
        const HeadDesc& H = p.heads[hi];
        return H.data + (1LL * frame * H.h * H.w + cell) * H.pitch + k * span;
    };

    double obj = 0.0, threshold = 0.0;
    bool pass = false;
    if (live) {
        int hi, cell, k;
        const float t4 = __ldg(locate(f, b, hi, cell, k) + 4);
        threshold = __ldg(p.thr + f);
        // float pre-test (sigmoid is monotonic, the margin dwarfs any rounding): ~99 % of the boxes end here; the decision
        // itself is taken in float64 exactly as the reference does
        if (!(t4 < __ldg(p.obj_cut + f))) {
            obj = logistic(t4);
            pass = !(obj < threshold);  // reference: `if conf < threshold: continue`
        }
    }
    unsigned mask = __ballot_sync(0xffffffffu, pass);
    while (mask) {
        const int src = __ffs(mask) - 1;
        mask &= mask - 1;
        const int bf = __shfl_sync(0xffffffffu, f, src), bb = __shfl_sync(0xffffffffu, b, src);
        int hi, cell, k;
        const float* box = locate(bf, bb, hi, cell, k);
        const float* cls = box + 5;
        // first-maximum arg-max over the raw logits (np.argmax)
        float best = -INFINITY;
        int best_i = INT_MAX;
        for (int c = lane; c < p.num_classes; c += 32) {
            const float v = __ldg(cls + c);
            if (v > best || best_i == INT_MAX) { best = v; best_i = c; }
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const float ov = __shfl_xor_sync(0xffffffffu, best, o);
            const int oi = __shfl_xor_sync(0xffffffffu, best_i, o);
            if (oi != INT_MAX && (best_i == INT_MAX || ov > best || (ov == best && oi < best_i))) { best = ov; best_i = oi; }
        }
        if (lane == src) {  // (the owning lane: its f is bf, its threshold the frame's)
            const double conf = obj * logistic(best);
            if (!(conf < threshold)) {
                const HeadDesc& H = p.heads[hi];
                const int gy = cell / H.w, gx = cell - gy * H.w;
                const double x = (gx + logistic(__ldg(box + 0))) / H.w;
                const double y = (gy + logistic(__ldg(box + 1))) / H.h;
                const double w = static_cast<double>(H.anchor_w[k]) * exp(static_cast<double>(__ldg(box + 2))) / p.net_w;
                const double h = static_cast<double>(H.anchor_h[k]) * exp(static_cast<double>(__ldg(box + 3))) / p.net_h;
                const int slot = atomicAdd(cand_count + bf, 1);
                Candidate c;
                c.conf = conf;
                c.x = x - w / 2;
                c.y = y - h / 2;
                c.w = w;
                c.h = h;
                c.box = H.first_box + cell * 3 + k;
                c.klass = best_i + 1;
                cand[1LL * bf * p.boxes_per_frame + slot] = c;
            }
        }
    }
}

int launch_decode(const HeadDesc* heads, int n_heads, int num_classes, int n, int net_w, int net_h,
                  const double* thr, const float* obj_cut, Candidate* cand, int* cand_count, int boxes_per_frame, cudaStream_t s) {
    if (n_heads < 1 || n_heads > 4) return -1;
    DecodeParams p;
    p.cell_start[0] = 0;
    for (int i = 0; i < n_heads; ++i) {
        p.heads[i] = heads[i];
        p.cell_start[i + 1] = p.cell_start[i] + heads[i].h * heads[i].w;
    }
    p.n_heads = n_heads; p.num_classes = num_classes; p.n = n; p.net_w = net_w; p.net_h = net_h;
    p.boxes_per_frame = boxes_per_frame; p.thr = thr; p.obj_cut = obj_cut;
    if (cudaMemsetAsync(cand_count, 0, sizeof(int) * n, s) != cudaSuccess) return -1;
    if (boxes_per_frame != 3 * p.cell_start[n_heads]) return -1;
    const long long boxes = 1LL * n * boxes_per_frame;
    const int blocks = static_cast<int>((boxes + 255) / 256);
    decode_kernel<<<blocks, 256, 0, s>>>(p, cand, cand_count);
    return cudaPeekAtLastError() == cudaSuccess ? 0 : -1;  // (peek: the caller reports the reason)
}

// ------------------------------------------------------------------------------------ Soft-NMS
static constexpr int NMS_THREADS = 512, NMS_WARPS = NMS_THREADS / 32;

// Frames with at most one candidate per thread (the usual case at serving thresholds): every candidate lives in its
// thread's registers, one __syncthreads per selected box.  Same selection rule, same decay arithmetic and the same
// emission order as the general loop below.
// Warp-wide arg-max of (score, lowest box index on ties) with three redux.sync steps instead of five rounds of double
// shuffles.  Scores are non-negative doubles, so their bit patterns order like unsigned integers: max of the high word
// (+1, so that 0 can mean "no candidate"), then max of the low word among the lanes still tied, then min box index.
// Returns the winning lane, or -1 if no lane holds a candidate.
__device__ __forceinline__ int warp_best(bool live, double score, int box) {
    const unsigned long long bits = static_cast<unsigned long long>(__double_as_longlong(score));
    const unsigned hi = live ? static_cast<unsigned>(bits >> 32) + 1u : 0u;
    const unsigned top = __reduce_max_sync(0xffffffffu, hi);
    if (top == 0u) return -1;
    const bool in1 = hi == top;
    const unsigned lo = in1 ? static_cast<unsigned>(bits) : 0u;
    const unsigned top_lo = __reduce_max_sync(0xffffffffu, lo);
    const bool in2 = in1 && lo == top_lo;
    const unsigned b = in2 ? static_cast<unsigned>(box) : 0xffffffffu;  // box indices are non-negative
    const unsigned first = __reduce_min_sync(0xffffffffu, b);
    return __ffs(__ballot_sync(0xffffffffu, in2 && b == first)) - 1;
}

// Frames with at most one candidate per thread (the usual case at serving thresholds): every candidate lives in its
// thread's registers, one __syncthreads per selected box.  Same selection rule, same decay arithmetic and the same
// emission order as the general loop below.
__device__ __forceinline__ void soft_nms_in_registers(const Candidate* __restrict__ cand, int C, int net_w, int net_h,
                                                      double threshold, Detection* __restrict__ out, int max_det, int* kept_out) {
    __shared__ double w_score[2][NMS_WARPS], w_geo[2][NMS_WARPS][4];
    __shared__ int w_box[2][NMS_WARPS];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    Candidate c;
    c.conf = 0; c.x = c.y = c.w = c.h = 0; c.box = INT_MAX; c.klass = 0;
    double sc = -2.0;  // < 0: not a live candidate
    if (tid < C) { c = cand[tid]; sc = c.conf; }
    int kept = 0;
    for (int it = 0;; ++it) {
        const int buf = it & 1;
        // arg-max of the live scores; ties go to the lowest insertion index (strict '<' at detector.py:51)
        const int wl = warp_best(sc >= 0.0, sc, c.box);
        if (lane == (wl < 0 ? 0 : wl)) {
            w_score[buf][warp] = wl < 0 ? -1.0 : sc;
            w_box[buf][warp] = c.box;
            w_geo[buf][warp][0] = c.x; w_geo[buf][warp][1] = c.y; w_geo[buf][warp][2] = c.w; w_geo[buf][warp][3] = c.h;
        }
        __syncthreads();
        // every warp repeats the same reduction over the per-warp winners (lane j looks at warp j)
        const double ws = lane < NMS_WARPS ? w_score[buf][lane] : -1.0;
        const int wb = lane < NMS_WARPS ? w_box[buf][lane] : INT_MAX;
        const int win = warp_best(ws >= 0.0, ws, wb);
        if (win < 0) break;
        const double best = __shfl_sync(0xffffffffu, ws, win);
        if (best < threshold) break;  // `if mconf < threshold: break`
        const int best_box = __shfl_sync(0xffffffffu, wb, win);
        if (sc >= 0.0 && c.box == best_box) {  // box indices are unique within a frame: this thread owns the selected box
            if (kept < max_det) {
                Detection d;
                d.klass = c.klass;
                d.box = c.box;
                d.conf = c.conf;  // the reference reports the original, undecayed score (detector.py:142)
                d.x = c.x * net_w; d.y = c.y * net_h; d.w = c.w * net_w; d.h = c.h * net_h;
                out[kept] = d;
            }
            sc = -2.0;
        } else if (sc >= 0.0) {
            const double x0 = w_geo[buf][win][0], y0 = w_geo[buf][win][1], w0 = w_geo[buf][win][2], h0 = w_geo[buf][win][3];
            const double iw = fmin(x0 + w0, c.x + c.w) - fmax(x0, c.x);
            const double ih = fmin(y0 + h0, c.y + c.h) - fmax(y0, c.y);
            if (iw > 0.0 && ih > 0.0) {  // overlap 0 -> factor exp(0) = 1
                const double ov = (iw * ih) / (w0 * h0);  // area(sel ∩ other) / area(sel): asymmetric, as the reference
                sc = sc * exp(-3.0 * (ov * ov));
            }
        }
        ++kept;
    }
    *kept_out = kept;
}

__global__ void __launch_bounds__(NMS_THREADS)
soft_nms_kernel(const Candidate* __restrict__ cand_all, const int* __restrict__ cand_count, double* __restrict__ score_all,
                int cap, int net_w, int net_h, const double* __restrict__ thr, Detection* __restrict__ out, int* __restrict__ out_count,
                int* __restrict__ total_count, int max_det, int allow_fast) {
    const int f = blockIdx.x;
    const double threshold = thr[f];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int C = min(cand_count[f], cap);
    const Candidate* cand = cand_all + 1LL * f * cap;
    if (C <= NMS_THREADS && allow_fast) {
        int kept = 0;
        soft_nms_in_registers(cand, C, net_w, net_h, threshold, out + 1LL * f * max_det, max_det, &kept);
        if (tid == 0) {
            out_count[f] = kept < max_det ? kept : max_det;
            total_count[f] = kept;
        }
        return;
    }
    double* sc = score_all + 1LL * f * cap;
    __shared__ double s_score[NMS_WARPS];
    __shared__ int s_box[NMS_WARPS], s_pos[NMS_WARPS];
    __shared__ double sel_box[4];
    __shared__ int sel_pos;

    for (int i = tid; i < C; i += NMS_THREADS) sc[i] = cand[i].conf;
    __syncthreads();
    int kept = 0;
    while (true) {
        // arg-max of the live scores; ties go to the lowest insertion index (strict '<' at detector.py:51)
        double best = -1.0;
        int best_box = INT_MAX, best_pos = -1;
        for (int i = tid; i < C; i += NMS_THREADS) {
            const double s = sc[i];
            if (s < 0.0) continue;  // already selected
            const int b = cand[i].box;
            if (s > best || (s == best && b < best_box)) { best = s; best_box = b; best_pos = i; }
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const double os = __shfl_xor_sync(0xffffffffu, best, o);
            const int ob = __shfl_xor_sync(0xffffffffu, best_box, o);
            const int op = __shfl_xor_sync(0xffffffffu, best_pos, o);
            if (os > best || (os == best && ob < best_box)) { best = os; best_box = ob; best_pos = op; }
        }
        if (lane == 0) { s_score[warp] = best; s_box[warp] = best_box; s_pos[warp] = best_pos; }
        __syncthreads();
        if (tid == 0) {
            for (int w2 = 1; w2 < NMS_WARPS; ++w2)
                if (s_score[w2] > best || (s_score[w2] == best && s_box[w2] < best_box)) {
                    best = s_score[w2]; best_box = s_box[w2]; best_pos = s_pos[w2];
                }
            if (best_pos < 0 || best < threshold) {  // `if mconf < threshold: break`
                sel_pos = -1;
            } else {
                sel_pos = best_pos;
                const Candidate c = cand[best_pos];
                sel_box[0] = c.x; sel_box[1] = c.y; sel_box[2] = c.w; sel_box[3] = c.h;
                if (kept < max_det) {
                    Detection d;
                    d.klass = c.klass;
                    d.box = c.box;
                    d.conf = c.conf;  // the reference reports the original, undecayed score (detector.py:142)
                    d.x = c.x * net_w; d.y = c.y * net_h; d.w = c.w * net_w; d.h = c.h * net_h;
                    out[1LL * f * max_det + kept] = d;
                }
                sc[best_pos] = -2.0;
            }
        }
        __syncthreads();
        if (sel_pos < 0) break;
        ++kept;
        const double x0 = sel_box[0], y0 = sel_box[1], w0 = sel_box[2], h0 = sel_box[3];
        for (int i = tid; i < C; i += NMS_THREADS) {
            const double s = sc[i];
            if (s < 0.0) continue;
            const Candidate c = cand[i];
            const double iw = fmin(x0 + w0, c.x + c.w) - fmax(x0, c.x);
            const double ih = fmin(y0 + h0, c.y + c.h) - fmax(y0, c.y);
            if (iw <= 0.0 || ih <= 0.0) continue;  // overlap 0 -> factor exp(0) = 1
            const double ov = (iw * ih) / (w0 * h0);  // area(sel ∩ other) / area(sel): asymmetric, as the reference
            sc[i] = s * exp(-3.0 * (ov * ov));
        }
        __syncthreads();
    }
    if (tid == 0) {
        out_count[f] = kept < max_det ? kept : max_det;
        total_count[f] = kept;
    }
}

int launch_soft_nms(Candidate* cand, const int* cand_count, double* score_scratch, int boxes_per_frame, int n,
                    int net_w, int net_h, const double* thr, Detection* out, int* out_count, int* total_count,
                    int max_det, cudaStream_t s) {
    const int allow_fast = options().nms_general ? 0 : 1;  // option nms_general: force the general loop (tests run both)
    soft_nms_kernel<<<n, NMS_THREADS, 0, s>>>(cand, cand_count, score_scratch, boxes_per_frame, net_w, net_h, thr,
                                              out, out_count, total_count, max_det, allow_fast);
    return cudaPeekAtLastError() == cudaSuccess ? 0 : -1;  // (peek: the caller reports the reason)
}

}  // namespace fd
