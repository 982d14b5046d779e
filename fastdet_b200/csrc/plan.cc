// plan.cc — see plan.h.
#include "plan.h"

#include <math.h>
#include <string.h>

#include <algorithm>
#include <map>

#include "kernels.h"

namespace fd {

uint16_t f32_to_bf16_rn(float f) {
    uint32_t u;
    memcpy(&u, &f, 4);
    if ((u & 0x7F800000u) == 0x7F800000u && (u & 0x007FFFFFu)) return static_cast<uint16_t>((u >> 16) | 0x40);  // NaN
    u += 0x7FFFu + ((u >> 16) & 1u);
    return static_cast<uint16_t>(u >> 16);
}

namespace {

enum AKind { A_INPUT, A_CONV, A_BN, A_LEAKY, A_ADD, A_MAXPOOL, A_PAD, A_RESIZE, A_CONCAT, A_VIEW, A_MISH };

struct ANode {
    AKind kind;
    int node = -1;  // index into graph.nodes
    std::vector<int> in;
    int c = 0, h = 0, w = 0;
    std::string out_name;
    std::vector<int> consumers;
    bool is_output = false;
    // per-kind payload
    int ksize = 1, stride = 1, pad_lo = 0, pad_hi = 0;  // conv / pool
    float alpha = 0.f;                                   // leaky
    float pad_value = 0.f;                               // pad
    int pads[4] = {0, 0, 0, 0};                          // pad node: t,l,b,r
    int view_start = 0;                                  // view: first channel inside the source (Slice / Split on axis 1)
    int value = -1;                                      // Value id this anode's result lives in
};

struct Value {
    TensorLoc loc;
    int view_of = -1;  // a channel view: the Value it reads, view_start channels in (resolved after buffer assignment)
    int view_start = 0;
    bool placed = false;
    bool is_input = false;
    bool fp32 = false;
};

struct Fused {
    LayerKind kind;
    int anchor = 0;  // execution position (anode id)
    int conv = -1, bn = -1, leaky = -1, add = -1, residual = -1, resize = -1, pool = -1, pad = -1;
    int in_anode = -1, final_anode = -1;
    int copy_src_value = -1, copy_dst_buf = -1, copy_dst_off = 0, copy_dst_pitch = 0, copy_up = 0;
};

struct Builder {
    const OnnxGraph& g;
    std::string* err;
    std::map<std::string, OnnxTensor> consts;
    std::map<std::string, int> acts;
    std::vector<ANode> an;

    Builder(const OnnxGraph& gg, std::string* e) : g(gg), err(e) {}

    bool fail(const std::string& m) {
        *err = m;
        return false;
    }
    const OnnxTensor* cst(const std::string& name) const {
        auto it = consts.find(name);
        return it == consts.end() ? nullptr : &it->second;
    }
    int act(const std::string& name) const {
        auto it = acts.find(name);
        return it == acts.end() ? -1 : it->second;
    }
    int add_anode(AKind k, int node, std::vector<int> in, int c, int h, int w, const std::string& out) {
        ANode a;
        a.kind = k;
        a.node = node;
        a.in = std::move(in);
        a.c = c; a.h = h; a.w = w;
        a.out_name = out;
        an.push_back(a);
        const int id = static_cast<int>(an.size()) - 1;
        for (int i : an[id].in) an[i].consumers.push_back(id);
        acts[out] = id;
        return id;
    }

    // ---- constant folding of the integer/float shape arithmetic exporters wrap around Resize / Pad ----
    // Small N-d tensors (row-major); values are carried as doubles and stored back as f32 or i64.
    struct CT {
        std::vector<int64_t> dims;
        std::vector<double> v;
        bool fl = false;
    };
    static CT to_ct(const OnnxTensor& t) {
        CT c;
        c.dims = t.dims;
        c.fl = t.is_float();
        if (c.fl) c.v.assign(t.f.begin(), t.f.end());
        else c.v.assign(t.i.begin(), t.i.end());
        return c;
    }
    static OnnxTensor from_ct(const CT& c) {
        OnnxTensor t;
        t.dims = c.dims;
        if (c.fl) { t.dtype = 1; t.f.assign(c.v.begin(), c.v.end()); }
        else { t.dtype = 7; t.i.resize(c.v.size()); for (size_t k = 0; k < c.v.size(); ++k) t.i[k] = static_cast<int64_t>(c.v[k]); }
        return t;
    }
    static std::vector<int64_t> strides_of(const std::vector<int64_t>& dims) {
        std::vector<int64_t> st(dims.size(), 1);
        for (int k = static_cast<int>(dims.size()) - 2; k >= 0; --k) st[k] = st[k + 1] * dims[k + 1];
        return st;
    }
    static int64_t numel_of(const std::vector<int64_t>& dims) {
        int64_t n = 1;
        for (int64_t d : dims) n *= d;
        return n;
    }
    // out[idx] = in[map(idx)] where map gives, per output axis, (input axis, start, step)
    static CT gather_nd(const CT& in, const std::vector<int64_t>& out_dims, const std::vector<int>& in_axis,
                        const std::vector<int64_t>& start, const std::vector<int64_t>& step) {
        CT out;
        out.dims = out_dims;
        out.fl = in.fl;
        const int64_t n = numel_of(out_dims);
        out.v.resize(static_cast<size_t>(n));
        const std::vector<int64_t> ist = strides_of(in.dims);
        std::vector<int64_t> idx(out_dims.size(), 0);
        for (int64_t k = 0; k < n; ++k) {
            int64_t off = 0;
            for (size_t a = 0; a < out_dims.size(); ++a) off += (start[a] + idx[a] * step[a]) * ist[in_axis[a]];
            out.v[static_cast<size_t>(k)] = in.v[static_cast<size_t>(off)];
            for (int a = static_cast<int>(out_dims.size()) - 1; a >= 0; --a) {
                if (++idx[a] < out_dims[a]) break;
                idx[a] = 0;
            }
        }
        return out;
    }
    bool try_fold(const OnnxNode& n) {
        const std::string& op = n.op;
        if (op == "Shape") {
            const int a = act(n.inputs[0]);
            OnnxTensor t;
            t.dtype = 7;
            if (a >= 0) t.i = {1, an[a].c, an[a].h, an[a].w};
            else if (const OnnxTensor* c = cst(n.inputs[0])) t.i = c->dims;
            else return false;
            t.dims = {static_cast<int64_t>(t.i.size())};
            consts[n.outputs[0]] = t;
            return true;
        }
        std::vector<CT> in;
        std::vector<bool> have;
        for (const auto& nm : n.inputs) {
            if (nm.empty()) { in.emplace_back(); have.push_back(false); continue; }
            const OnnxTensor* c = cst(nm);
            if (!c) return false;
            in.push_back(to_ct(*c));
            have.push_back(true);
        }
        if (in.empty() || !have[0]) return false;
        if (numel_of(in[0].dims) > (1 << 20)) return false;  // shape arithmetic only, never weights
        auto ints_of = [](const CT& c) { std::vector<int64_t> r; for (double d : c.v) r.push_back(static_cast<int64_t>(d)); return r; };
        CT out;
        if (op == "Identity") {
            out = in[0];
        } else if (op == "Cast") {
            const int64_t to = n.attr_i("to", 1);
            out = in[0];
            out.fl = (to == 1 || to == 10 || to == 11);
            if (!out.fl) for (auto& x : out.v) x = trunc(x);
        } else if (op == "Floor") {
            out = in[0];
            for (auto& x : out.v) x = floor(x);
        } else if (op == "Mul" || op == "Div" || op == "Add" || op == "Sub") {
            if (in.size() < 2 || !have[1] || in[0].v.empty() || in[1].v.empty()) return false;
            const CT &a = in[0], &b = in[1];
            if (a.v.size() != b.v.size() && a.v.size() != 1 && b.v.size() != 1) return false;
            out.fl = a.fl || b.fl;
            out.dims = a.v.size() >= b.v.size() ? a.dims : b.dims;
            const size_t nn = std::max(a.v.size(), b.v.size());
            out.v.resize(nn);
            for (size_t k = 0; k < nn; ++k) {
                const double x = a.v[a.v.size() == 1 ? 0 : k], y = b.v[b.v.size() == 1 ? 0 : k];
                double r = op == "Mul" ? x * y : op == "Add" ? x + y : op == "Sub" ? x - y : (y != 0 ? x / y : 0);
                if (op == "Div" && !out.fl) r = trunc(r);
                out.v[k] = r;
            }
        } else if (op == "Gather") {
            if (in.size() < 2 || !have[1] || n.attr_i("axis", 0) != 0 || in[0].dims.empty()) return false;
            const int64_t d0 = in[0].dims[0];
            const int64_t inner = d0 ? numel_of(in[0].dims) / d0 : 0;
            out.fl = in[0].fl;
            out.dims = in[1].dims;
            out.dims.insert(out.dims.end(), in[0].dims.begin() + 1, in[0].dims.end());
            for (double di : in[1].v) {
                int64_t idx = static_cast<int64_t>(di);
                if (idx < 0) idx += d0;
                if (idx < 0 || idx >= d0) return false;
                out.v.insert(out.v.end(), in[0].v.begin() + idx * inner, in[0].v.begin() + (idx + 1) * inner);
            }
        } else if (op == "ConstantOfShape") {
            out.dims = ints_of(in[0]);
            double fill = 0.0;
            out.fl = true;
            auto it = n.attrs.find("value");
            if (it != n.attrs.end()) {
                const OnnxTensor& t = it->second.t;
                out.fl = t.is_float();
                if (out.fl && !t.f.empty()) fill = t.f[0];
                if (!out.fl && !t.i.empty()) fill = static_cast<double>(t.i[0]);
            }
            const int64_t cnt = numel_of(out.dims);
            if (cnt < 0 || cnt > (1 << 20)) return false;
            out.v.assign(static_cast<size_t>(cnt), fill);
        } else if (op == "Concat") {
            int64_t axis = n.attr_i("axis", 0);
            const size_t rank = in[0].dims.size();
            if (axis < 0) axis += static_cast<int64_t>(rank);
            if (rank == 0 || axis < 0 || axis >= static_cast<int64_t>(rank)) return false;
            out.dims = in[0].dims;
            out.dims[axis] = 0;
            int64_t outer = 1;
            for (int64_t a = 0; a < axis; ++a) outer *= in[0].dims[a];
            for (size_t k = 0; k < in.size(); ++k) {
                if (!have[k] || in[k].dims.size() != rank) return false;
                out.dims[axis] += in[k].dims[axis];
                out.fl = out.fl || in[k].fl;
            }
            for (int64_t o = 0; o < outer; ++o)
                for (const CT& t : in) {
                    const int64_t chunk = outer ? numel_of(t.dims) / outer : 0;
                    out.v.insert(out.v.end(), t.v.begin() + o * chunk, t.v.begin() + (o + 1) * chunk);
                }
        } else if (op == "Reshape") {
            if (in.size() < 2 || !have[1]) return false;
            std::vector<int64_t> shape = ints_of(in[1]);
            const int64_t total = numel_of(in[0].dims);
            int64_t known = 1;
            int infer = -1;
            for (size_t k = 0; k < shape.size(); ++k) {
                if (shape[k] == 0 && k < in[0].dims.size()) shape[k] = in[0].dims[k];
                if (shape[k] == -1) infer = static_cast<int>(k);
                else known *= shape[k];
            }
            if (infer >= 0) { if (known == 0) return false; shape[infer] = total / known; }
            if (numel_of(shape) != total) return false;
            out = in[0];
            out.dims = shape;
        } else if (op == "Unsqueeze" || op == "Squeeze") {
            std::vector<int64_t> axes;
            if (const auto* ax = n.attr_ints("axes")) axes = *ax;
            else if (in.size() > 1 && have[1]) axes = ints_of(in[1]);
            out = in[0];
            if (op == "Unsqueeze") {
                const int64_t rank = static_cast<int64_t>(in[0].dims.size() + axes.size());
                for (auto& a : axes) if (a < 0) a += rank;
                std::sort(axes.begin(), axes.end());
                for (int64_t a : axes) { if (a < 0 || a > static_cast<int64_t>(out.dims.size())) return false; out.dims.insert(out.dims.begin() + a, 1); }
            } else {
                const int64_t rank = static_cast<int64_t>(in[0].dims.size());
                std::vector<int64_t> keep;
                for (int64_t a = 0; a < rank; ++a) {
                    bool drop = axes.empty() ? in[0].dims[a] == 1 : false;
                    for (int64_t x : axes) if ((x < 0 ? x + rank : x) == a) drop = true;
                    if (!drop) keep.push_back(in[0].dims[a]);
                }
                out.dims = keep;
            }
        } else if (op == "Transpose") {
            const size_t rank = in[0].dims.size();
            std::vector<int64_t> perm;
            if (const auto* pp = n.attr_ints("perm")) perm = *pp;
            else for (size_t k = 0; k < rank; ++k) perm.push_back(static_cast<int64_t>(rank - 1 - k));
            if (perm.size() != rank) return false;
            std::vector<int64_t> od(rank), start(rank, 0), step(rank, 1);
            std::vector<int> axis(rank);
            for (size_t k = 0; k < rank; ++k) {
                if (perm[k] < 0 || perm[k] >= static_cast<int64_t>(rank)) return false;
                od[k] = in[0].dims[perm[k]];
                axis[k] = static_cast<int>(perm[k]);
            }
            out = gather_nd(in[0], od, axis, start, step);
        } else if (op == "Slice") {
            const size_t rank = in[0].dims.size();
            std::vector<int64_t> starts, ends, axes, steps;
            if (in.size() >= 3 && have[1] && have[2]) {
                starts = ints_of(in[1]); ends = ints_of(in[2]);
                if (in.size() >= 4 && have[3]) axes = ints_of(in[3]);
                if (in.size() >= 5 && have[4]) steps = ints_of(in[4]);
            } else {
                const auto* ss = n.attr_ints("starts"); const auto* ee = n.attr_ints("ends");
                if (!ss || !ee) return false;
                starts = *ss; ends = *ee;
                if (const auto* ax = n.attr_ints("axes")) axes = *ax;
            }
            if (axes.empty()) for (size_t k = 0; k < starts.size(); ++k) axes.push_back(static_cast<int64_t>(k));
            if (steps.empty()) steps.assign(starts.size(), 1);
            if (ends.size() != starts.size() || axes.size() != starts.size() || steps.size() != starts.size()) return false;
            std::vector<int64_t> od = in[0].dims, start(rank, 0), step(rank, 1);
            std::vector<int> axis(rank);
            for (size_t k = 0; k < rank; ++k) axis[k] = static_cast<int>(k);
            for (size_t k = 0; k < starts.size(); ++k) {
                int64_t a = axes[k];
                if (a < 0) a += static_cast<int64_t>(rank);
                if (a < 0 || a >= static_cast<int64_t>(rank) || steps[k] == 0) return false;
                const int64_t dim = in[0].dims[a], st = steps[k];
                int64_t s0 = starts[k], e0 = ends[k];
                // ONNX Slice clamping rules (INT64 extremes mean "to the end")
                if (s0 < 0) s0 = std::max<int64_t>(s0 + dim, st > 0 ? 0 : -1);
                if (e0 < 0) e0 = std::max<int64_t>(e0 + dim, -1);
                if (st > 0) { s0 = std::min(s0, dim); e0 = std::min(e0, dim); }
                else { s0 = std::min(s0, dim - 1); e0 = std::min(e0, dim - 1); if (ends[k] < -dim) e0 = -1; }
                int64_t cnt = st > 0 ? (e0 - s0 + st - 1) / st : (s0 - e0 + (-st) - 1) / (-st);
                if (cnt < 0) cnt = 0;
                od[a] = cnt; start[a] = s0; step[a] = st;
            }
            out = gather_nd(in[0], od, axis, start, step);
        } else {
            return false;
        }
        consts[n.outputs[0]] = from_ct(out);
        return true;
    }

    // ---- per-op shape/semantics checks while walking the graph ----
    bool conv_geometry(const OnnxNode& n, int k, int hin, int win, int* stride, int* pad_lo, int* pad_hi) {
        const auto* st = n.attr_ints("strides");
        const int sh = st && st->size() >= 2 ? static_cast<int>((*st)[0]) : 1;
        const int sw = st && st->size() >= 2 ? static_cast<int>((*st)[1]) : 1;
        if (sh != sw) return fail(n.name + ": anisotropic strides are not supported");
        if (const auto* d = n.attr_ints("dilations"))
            for (int64_t v : *d) if (v != 1) return fail(n.name + ": dilation != 1 is not supported");
        const std::string auto_pad = n.attr_s("auto_pad", "NOTSET");
        int t = 0, l = 0, b = 0, r = 0;
        if (auto_pad == "NOTSET" || auto_pad.empty()) {
            if (const auto* p = n.attr_ints("pads")) {
                if (p->size() != 4) return fail(n.name + ": pads must have 4 entries");
                t = static_cast<int>((*p)[0]); l = static_cast<int>((*p)[1]);
                b = static_cast<int>((*p)[2]); r = static_cast<int>((*p)[3]);
            }
        } else if (auto_pad == "SAME_UPPER" || auto_pad == "SAME_LOWER") {
            const int dims[2] = {hin, win};
            int lo[2], hi[2];
            for (int i = 0; i < 2; ++i) {
                const int out = (dims[i] + sh - 1) / sh;
                const int total = std::max((out - 1) * sh + k - dims[i], 0);
                lo[i] = auto_pad == "SAME_UPPER" ? total / 2 : total - total / 2;
                hi[i] = total - lo[i];
            }
            t = lo[0]; l = lo[1]; b = hi[0]; r = hi[1];
        } else if (auto_pad != "VALID") {
            return fail(n.name + ": unknown auto_pad " + auto_pad);
        }
        if (t != l || b != r) return fail(n.name + ": padding must be the same for height and width");
        *stride = sh; *pad_lo = t; *pad_hi = b;
        return true;
    }

    // Slice / Split of an activation on the channel axis: a view of the source's channels [start, start + len), no layer.
    // Views of views compose; the alignment rule is checked where the view is read (an unread Split output may be anything).
    bool add_view(const OnnxNode& n, int x, int64_t start, int64_t len, const std::string& out) {
        if (an[x].kind == A_INPUT) return fail(n.name + ": channel slice of the network input is not supported");
        if (len <= 0 || start < 0 || start + len > an[x].c) return fail(n.name + ": empty or out-of-range channel slice");
        int src = x;
        int64_t off = start;
        if (an[x].kind == A_VIEW) { off += an[x].view_start; src = an[x].in[0]; }
        const int id = add_anode(A_VIEW, static_cast<int>(&n - g.nodes.data()), {src}, static_cast<int>(len), an[x].h, an[x].w, out);
        an[id].view_start = static_cast<int>(off);
        return true;
    }
    bool channel_axis(const OnnxNode& n, int64_t axis) {
        if (axis != 1 && axis != -3) return fail(n.name + ": " + n.op + " on axis " + std::to_string(axis) + " (only channel slices, axis 1, are supported)");
        return true;
    }
    bool slice_view(const OnnxNode& n, int x) {
        std::vector<int64_t> starts, ends, axes, steps;
        if (n.inputs.size() >= 3) {  // opset >= 10: inputs, constant or folded from the shape chain
            const OnnxTensor* s = cst(n.inputs[1]);
            const OnnxTensor* e = cst(n.inputs[2]);
            const OnnxTensor* a = n.inputs.size() > 3 && !n.inputs[3].empty() ? cst(n.inputs[3]) : nullptr;
            const OnnxTensor* st = n.inputs.size() > 4 && !n.inputs[4].empty() ? cst(n.inputs[4]) : nullptr;
            if (!s || !e || (n.inputs.size() > 3 && !n.inputs[3].empty() && !a) || (n.inputs.size() > 4 && !n.inputs[4].empty() && !st))
                return fail(n.name + ": Slice starts / ends / axes / steps must be constant");
            starts = s->i; ends = e->i;
            if (a) axes = a->i;
            if (st) steps = st->i;
        } else {
            const auto* ss = n.attr_ints("starts");
            const auto* ee = n.attr_ints("ends");
            if (!ss || !ee) return fail(n.name + ": Slice without starts / ends");
            starts = *ss; ends = *ee;
            if (const auto* ax = n.attr_ints("axes")) axes = *ax;
        }
        if (axes.empty()) for (size_t k = 0; k < starts.size(); ++k) axes.push_back(static_cast<int64_t>(k));
        if (steps.empty()) steps.assign(starts.size(), 1);
        if (starts.size() != 1 || ends.size() != 1 || axes.size() != 1 || steps.size() != 1)
            return fail(n.name + ": Slice must touch the channel axis only (it slices N, H or W)");
        if (!channel_axis(n, axes[0])) return false;
        if (steps[0] != 1) return fail(n.name + ": Slice step " + std::to_string(steps[0]) + " (only step 1 is supported)");
        // ONNX clamping: negative values count from the end, anything past the ends (INT64_MAX) clamps to them
        const int64_t c = an[x].c;
        int64_t s0 = starts[0], e0 = ends[0];
        if (s0 < 0) s0 += c;
        if (e0 < 0) e0 += c;
        s0 = std::min(std::max<int64_t>(s0, 0), c);
        e0 = std::min(std::max<int64_t>(e0, 0), c);
        return add_view(n, x, s0, e0 - s0, n.outputs[0]);
    }
    bool split_views(const OnnxNode& n, int x) {
        if (!channel_axis(n, n.attr_i("axis", 0))) return false;
        std::vector<int64_t> sizes;
        if (const auto* sp = n.attr_ints("split")) sizes = *sp;
        else if (n.inputs.size() > 1 && !n.inputs[1].empty()) {
            const OnnxTensor* t = cst(n.inputs[1]);
            if (!t) return fail(n.name + ": Split sizes must be constant");
            sizes = t->i;
        } else {
            const int64_t parts = static_cast<int64_t>(n.outputs.size());
            if (an[x].c % parts) return fail(n.name + ": Split into equal parts of a channel count they do not divide");
            sizes.assign(static_cast<size_t>(parts), an[x].c / parts);
        }
        if (sizes.size() != n.outputs.size()) return fail(n.name + ": Split has " + std::to_string(sizes.size()) + " sizes for " + std::to_string(n.outputs.size()) + " outputs");
        int64_t off = 0;
        for (size_t k = 0; k < sizes.size(); ++k) {
            if (!n.outputs[k].empty() && !add_view(n, x, off, sizes[k], n.outputs[k])) return false;
            off += sizes[k];
        }
        if (off != an[x].c) return fail(n.name + ": Split sizes do not add up to the channel count");
        return true;
    }

    // Mish written out as Softplus(x) -> Tanh -> Mul(x, tanh) (torch's exporter, symbolic_opset9.mish): the Softplus and
    // the Tanh become pending chain links, the Mul that closes the chain becomes one A_MISH anode.  Anything else with
    // Softplus or Tanh in it is refused, naming the node.
    struct MishLink { int x = -1; std::string node; bool used = false; std::string src; };  // src: a Tanh's Softplus output
    std::map<std::string, MishLink> softplus, tanh_of;  // by output name
    std::map<std::string, int> readers;                 // nodes (and graph outputs) that read a tensor
    // returns true when the node belongs to a Mish chain (then *ok says whether it was accepted)
    bool mish_link(const OnnxNode& n, int ni, bool* ok) {
        *ok = true;
        const std::string& out = n.outputs[0];
        if (n.op == "Softplus") {
            const int x = n.inputs.empty() ? -1 : act(n.inputs[0]);
            if (x < 0) { *ok = fail(n.name + ": Softplus of a tensor that is not an activation"); return true; }
            softplus[out] = {x, n.name, false};
            return true;
        }
        if (n.op == "Tanh") {
            auto it = n.inputs.empty() ? softplus.end() : softplus.find(n.inputs[0]);
            if (it == softplus.end()) { *ok = fail(n.name + ": Tanh is only supported as the tanh(softplus(x)) of Mish"); return true; }
            it->second.used = true;
            tanh_of[out] = {it->second.x, n.name, false, n.inputs[0]};
            return true;
        }
        if (n.op != "Mul" || n.inputs.size() != 2) return false;
        const int t = tanh_of.count(n.inputs[0]) ? 0 : tanh_of.count(n.inputs[1]) ? 1 : -1;
        if (t < 0) return false;
        MishLink& tl = tanh_of[n.inputs[t]];
        tl.used = true;
        const int x = tl.x;
        if (act(n.inputs[1 - t]) != x) { *ok = fail(n.name + ": Mul of tanh(softplus(x)) with a tensor other than x is not Mish"); return true; }
        if (readers[tl.src] != 1) { *ok = fail(softplus[tl.src].node + ": Softplus output of Mish '" + n.name + "' has other readers"); return true; }
        if (readers[n.inputs[t]] != 1) { *ok = fail(tl.node + ": Tanh output of Mish '" + n.name + "' has other readers"); return true; }
        add_anode(A_MISH, ni, {x}, an[x].c, an[x].h, an[x].w, out);
        return true;
    }

    bool walk() {
        for (const auto& kv : g.initializers) consts[kv.first] = kv.second;
        // graph input: the reference feeds {'input': a} (server/detector.py:135)
        const OnnxValueInfo* in = nullptr;
        for (const auto& vi : g.inputs) if (vi.name == "input") in = &vi;
        if (!in) return fail("graph has no input named 'input' (reference server/detector.py:135 feeds that name)");
        return true;
    }
};

}  // namespace

bool build_plan(const OnnxGraph& g, int net_w, int net_h, int num_classes, bool fuse_pool, ModelPlan* plan, std::string* err) {
    Builder B(g, err);
    if (!B.walk()) return false;
    plan->net_w = net_w; plan->net_h = net_h; plan->num_classes = num_classes;
    const int input_id = B.add_anode(A_INPUT, -1, {}, 3, net_h, net_w, "input");
    for (const auto& n : g.nodes)
        for (const auto& nm : n.inputs) ++B.readers[nm];
    for (const auto& o : g.outputs) ++B.readers[o.name];

    // ------------------------------------------------------------------ pass 1: activation graph
    for (size_t ni = 0; ni < g.nodes.size(); ++ni) {
        const OnnxNode& n = g.nodes[ni];
        if (n.outputs.empty()) continue;
        const std::string& out = n.outputs[0];
        if (n.op == "Constant") {
            auto it = n.attrs.find("value");
            if (it == n.attrs.end()) return B.fail("Constant node '" + n.name + "' without a tensor value");
            B.consts[out] = it->second.t;
            continue;
        }
        {
            bool ok = true;
            if (B.mish_link(n, static_cast<int>(ni), &ok)) {
                if (!ok) return false;
                continue;
            }
            for (const auto& nm : n.inputs) {  // any other reader of a Softplus / Tanh output
                auto sp = B.softplus.find(nm);
                if (sp != B.softplus.end()) return B.fail(sp->second.node + ": Softplus is only supported as the softplus of Mish, x * tanh(softplus(x)) (read by '" + n.name + "')");
                auto th = B.tanh_of.find(nm);
                if (th != B.tanh_of.end()) return B.fail(th->second.node + ": Tanh is only supported as the tanh(softplus(x)) of Mish, multiplied by x (read by '" + n.name + "')");
            }
        }
        const int x = n.inputs.empty() ? -1 : B.act(n.inputs[0]);
        if (n.op == "Shape" || x < 0) {
            // integer/float shape arithmetic (or an op on constants only)
            bool any_act = false;
            for (const auto& nm : n.inputs) any_act |= B.act(nm) >= 0;
            if (n.op == "Shape" || !any_act) {
                if (B.try_fold(n)) continue;
                if (!any_act) return B.fail("cannot constant-fold node '" + n.name + "' (" + n.op + ")");
            }
        }
        if (n.op == "Identity" || n.op == "Dropout") {
            if (x < 0) return B.fail(n.name + ": Identity of an unknown tensor");
            B.acts[out] = x;
            continue;
        }
        if (n.op == "Conv") {
            if (x < 0) return B.fail(n.name + ": Conv input is not an activation");
            const OnnxTensor* W = n.inputs.size() > 1 ? B.cst(n.inputs[1]) : nullptr;
            if (!W || W->dims.size() != 4 || !W->is_float()) return B.fail(n.name + ": Conv weight must be a constant 4-D float tensor");
            if (n.attr_i("group", 1) != 1) return B.fail(n.name + ": grouped convolution is not supported");
            const int cout = static_cast<int>(W->dims[0]), cin = static_cast<int>(W->dims[1]);
            const int kh = static_cast<int>(W->dims[2]), kw = static_cast<int>(W->dims[3]);
            if (kh != kw || !(kh == 1 || kh == 3)) return B.fail(n.name + ": only 1x1 and 3x3 filters are supported");
            if (cin != B.an[x].c) return B.fail(n.name + ": weight Cin does not match the input channels");
            int stride, pl, ph;
            if (!B.conv_geometry(n, kh, B.an[x].h, B.an[x].w, &stride, &pl, &ph)) return false;
            const int ho = (B.an[x].h + pl + ph - kh) / stride + 1, wo = (B.an[x].w + pl + ph - kh) / stride + 1;
            const int id = B.add_anode(A_CONV, static_cast<int>(ni), {x}, cout, ho, wo, out);
            B.an[id].ksize = kh; B.an[id].stride = stride; B.an[id].pad_lo = pl; B.an[id].pad_hi = ph;
        } else if (n.op == "BatchNormalization") {
            if (x < 0 || n.inputs.size() < 5) return B.fail(n.name + ": malformed BatchNormalization");
            for (int k = 1; k < 5; ++k) {
                const OnnxTensor* t = B.cst(n.inputs[k]);
                if (!t || static_cast<int>(t->numel()) != B.an[x].c) return B.fail(n.name + ": BatchNormalization parameters must be constants of size C");
            }
            B.add_anode(A_BN, static_cast<int>(ni), {x}, B.an[x].c, B.an[x].h, B.an[x].w, out);
        } else if (n.op == "LeakyRelu" || n.op == "Relu") {
            if (x < 0) return B.fail(n.name + ": activation input is not an activation tensor");
            const int id = B.add_anode(A_LEAKY, static_cast<int>(ni), {x}, B.an[x].c, B.an[x].h, B.an[x].w, out);
            B.an[id].alpha = n.op == "Relu" ? 0.f : n.attr_f("alpha", 0.01f);
        } else if (n.op == "Mish") {
            if (x < 0) return B.fail(n.name + ": activation input is not an activation tensor");
            B.add_anode(A_MISH, static_cast<int>(ni), {x}, B.an[x].c, B.an[x].h, B.an[x].w, out);
        } else if (n.op == "Add") {
            const int y = n.inputs.size() > 1 ? B.act(n.inputs[1]) : -1;
            if (x < 0 || y < 0) return B.fail(n.name + ": Add needs two activation inputs");
            if (B.an[x].c != B.an[y].c || B.an[x].h != B.an[y].h || B.an[x].w != B.an[y].w) return B.fail(n.name + ": Add operands differ in shape");
            B.add_anode(A_ADD, static_cast<int>(ni), {x, y}, B.an[x].c, B.an[x].h, B.an[x].w, out);
        } else if (n.op == "MaxPool") {
            if (x < 0) return B.fail(n.name + ": MaxPool input is not an activation");
            const auto* ks = n.attr_ints("kernel_shape");
            if (!ks || ks->size() != 2 || (*ks)[0] != (*ks)[1]) return B.fail(n.name + ": MaxPool needs a square kernel_shape");
            if (n.attr_i("ceil_mode", 0) != 0) return B.fail(n.name + ": ceil_mode is not supported");
            const int k = static_cast<int>((*ks)[0]);
            int stride, pl, ph;
            if (!B.conv_geometry(n, k, B.an[x].h, B.an[x].w, &stride, &pl, &ph)) return false;
            const int ho = (B.an[x].h + pl + ph - k) / stride + 1, wo = (B.an[x].w + pl + ph - k) / stride + 1;
            const int id = B.add_anode(A_MAXPOOL, static_cast<int>(ni), {x}, B.an[x].c, ho, wo, out);
            B.an[id].ksize = k; B.an[id].stride = stride; B.an[id].pad_lo = pl; B.an[id].pad_hi = ph;
        } else if (n.op == "Pad") {
            if (x < 0) return B.fail(n.name + ": Pad input is not an activation");
            std::vector<int64_t> pads;
            float value = 0.f;
            if (n.inputs.size() > 1 && !n.inputs[1].empty()) {
                const OnnxTensor* p = B.cst(n.inputs[1]);
                if (!p) return B.fail(n.name + ": Pad amounts must be constant");
                pads = p->i;
                if (n.inputs.size() > 2 && !n.inputs[2].empty()) {
                    const OnnxTensor* v = B.cst(n.inputs[2]);
                    if (!v) return B.fail(n.name + ": Pad value must be constant");
                    if (!v->f.empty()) value = v->f[0];
                }
            } else if (const auto* p = n.attr_ints("pads")) {
                pads = *p;
                value = n.attr_f("value", 0.f);
            }
            if (n.attr_s("mode", "constant") != "constant") return B.fail(n.name + ": only constant Pad is supported");
            if (pads.size() != 8 || pads[0] || pads[1] || pads[4] || pads[5]) return B.fail(n.name + ": Pad must touch H and W only");
            const int id = B.add_anode(A_PAD, static_cast<int>(ni), {x}, B.an[x].c, B.an[x].h + static_cast<int>(pads[2] + pads[6]),
                                       B.an[x].w + static_cast<int>(pads[3] + pads[7]), out);
            B.an[id].pads[0] = static_cast<int>(pads[2]); B.an[id].pads[1] = static_cast<int>(pads[3]);
            B.an[id].pads[2] = static_cast<int>(pads[6]); B.an[id].pads[3] = static_cast<int>(pads[7]);
            B.an[id].pad_value = value;
        } else if (n.op == "Resize" || n.op == "Upsample") {
            if (x < 0) return B.fail(n.name + ": Resize input is not an activation");
            if (n.attr_s("mode", "nearest") != "nearest") return B.fail(n.name + ": only nearest-neighbour Resize is supported");
            double sy = 0, sx = 0;
            const OnnxTensor* scales = nullptr;
            const OnnxTensor* sizes = nullptr;
            if (n.op == "Upsample" || n.inputs.size() == 2) {
                if (n.inputs.size() > 1) scales = B.cst(n.inputs[1]);
            } else {
                if (n.inputs.size() > 2 && !n.inputs[2].empty()) scales = B.cst(n.inputs[2]);
                if (n.inputs.size() > 3 && !n.inputs[3].empty()) sizes = B.cst(n.inputs[3]);
            }
            if (scales && scales->numel() == 4 && !scales->f.empty()) { sy = scales->f[2]; sx = scales->f[3]; }
            else if (sizes && sizes->i.size() == 4) { sy = double(sizes->i[2]) / B.an[x].h; sx = double(sizes->i[3]) / B.an[x].w; }
            else {
                auto it = n.attrs.find("scales");
                if (it != n.attrs.end() && it->second.floats.size() == 4) { sy = it->second.floats[2]; sx = it->second.floats[3]; }
                else return B.fail(n.name + ": Resize scales/sizes must be constant");
            }
            if (sy != 2.0 || sx != 2.0) return B.fail(n.name + ": only x2 nearest upsampling is supported");
            B.add_anode(A_RESIZE, static_cast<int>(ni), {x}, B.an[x].c, 2 * B.an[x].h, 2 * B.an[x].w, out);
        } else if (n.op == "Concat") {
            if (n.attr_i("axis", 1) != 1) return B.fail(n.name + ": only channel Concat (axis=1) is supported");
            std::vector<int> ins;
            int c = 0;
            for (const auto& nm : n.inputs) {
                const int a = B.act(nm);
                if (a < 0) return B.fail(n.name + ": Concat input '" + nm + "' is not an activation");
                if (!ins.empty() && (B.an[a].h != B.an[ins[0]].h || B.an[a].w != B.an[ins[0]].w)) return B.fail(n.name + ": Concat inputs differ in spatial size");
                ins.push_back(a);
                c += B.an[a].c;
            }
            if (ins.empty()) return B.fail(n.name + ": empty Concat");
            const int h = B.an[ins[0]].h, w = B.an[ins[0]].w;
            B.add_anode(A_CONCAT, static_cast<int>(ni), ins, c, h, w, out);
        } else if (n.op == "Slice") {
            if (!B.slice_view(n, x)) return false;
        } else if (n.op == "Split") {
            if (!B.split_views(n, x)) return false;
        } else {
            return B.fail("unsupported ONNX operator '" + n.op + "' (node '" + n.name + "')");
        }
    }
    for (const auto& kv : B.softplus)
        if (!kv.second.used) return B.fail(kv.second.node + ": Softplus is only supported as the softplus of Mish, x * tanh(softplus(x))");
    for (const auto& kv : B.tanh_of)
        if (!kv.second.used) return B.fail(kv.second.node + ": Tanh is only supported as the tanh(softplus(x)) of Mish, multiplied by x");
    std::vector<int> out_anodes;
    for (const auto& o : g.outputs) {
        const int a = B.act(o.name);
        if (a < 0) return B.fail("graph output '" + o.name + "' is not produced by a supported operator");
        if (B.an[a].kind == A_VIEW) return B.fail("graph output '" + o.name + "' is a channel slice (node '" + g.nodes[B.an[a].node].name + "'): a head must be a convolution's own output");
        B.an[a].is_output = true;
        out_anodes.push_back(a);
    }
    if (out_anodes.empty()) return B.fail("graph has no outputs");

    // ------------------------------------------------------------------ pass 2: fusion
    std::vector<ANode>& an = B.an;
    std::vector<int> owner(an.size(), -1);  // fused op each anode belongs to
    std::vector<Fused> ops;
    auto sole_consumer = [&](int a) -> int {
        return (!an[a].is_output && an[a].consumers.size() == 1) ? an[a].consumers[0] : -1;
    };
    for (int a = 0; a < static_cast<int>(an.size()); ++a) {
        if (owner[a] >= 0 || an[a].kind == A_INPUT || an[a].kind == A_CONCAT || an[a].kind == A_VIEW) continue;
        Fused f;
        const int id = static_cast<int>(ops.size());
        if (an[a].kind == A_CONV) {
            f.kind = an[a].in[0] == input_id ? LAYER_CONV0 : LAYER_CONV;
            f.conv = a; f.in_anode = an[a].in[0];
            int cur = a, nx;
            owner[a] = id;
            if ((nx = sole_consumer(cur)) >= 0 && an[nx].kind == A_BN) { f.bn = nx; owner[nx] = id; cur = nx; }
            if ((nx = sole_consumer(cur)) >= 0 && (an[nx].kind == A_LEAKY || an[nx].kind == A_MISH)) { f.leaky = nx; owner[nx] = id; cur = nx; }
            if (f.kind == LAYER_CONV && (nx = sole_consumer(cur)) >= 0 && an[nx].kind == A_ADD) {
                const int other = an[nx].in[0] == cur ? an[nx].in[1] : an[nx].in[0];
                if (other != cur && other < a) { f.add = nx; f.residual = other; owner[nx] = id; cur = nx; }
            }
            if (f.kind == LAYER_CONV && (nx = sole_consumer(cur)) >= 0 && an[nx].kind == A_RESIZE) { f.resize = nx; owner[nx] = id; cur = nx; }
            // MaxPool(2, stride 2, no padding) straight after the activation: done in the epilogue of the kernels whose tile is
            // a 16 x 8 pixel patch (each epilogue warp holds whole 2x2 windows): the first convolution (Cout 16 / 32) and the
            // halo-patch layers.  The shape rules mirror conv_halo_supported() / launch_conv0_u8().
            if (fuse_pool && f.add < 0 && f.resize < 0 && (nx = sole_consumer(cur)) >= 0 && an[nx].kind == A_MAXPOOL &&
                an[nx].ksize == 2 && an[nx].stride == 2 && an[nx].pad_lo == 0 && an[nx].pad_hi == 0 && an[a].ksize == 3 &&
                an[a].stride == 1 && an[a].pad_lo == 1 && an[a].pad_hi == 1 && an[a].h % 2 == 0 && an[a].w % 2 == 0) {
                const int cin = an[an[a].in[0]].c, cout = an[a].c;
                const bool first = f.kind == LAYER_CONV0 && (cout == 16 || cout == 32);
                const bool halo = f.kind == LAYER_CONV && (cin == 16 || cin == 32 || cin == 64) && (cout == 32 || cout == 64 || cout == 128) &&
                                  an[a].h >= 64 && an[a].w >= 64;
                if (first || halo) { f.pool = nx; owner[nx] = id; cur = nx; }
            }
            f.final_anode = cur;
        } else if (an[a].kind == A_PAD) {
            const int nx = sole_consumer(a);
            if (nx < 0 || an[nx].kind != A_MAXPOOL) return B.fail("Pad '" + an[a].out_name + "' is only supported directly before MaxPool");
            if (an[nx].pad_lo || an[nx].pad_hi) return B.fail("Pad followed by a padded MaxPool is not supported");
            if (an[a].pads[0] != an[a].pads[1] || an[a].pads[2] != an[a].pads[3]) return B.fail("Pad must be the same for height and width");
            f.kind = LAYER_MAXPOOL; f.pad = a; f.pool = nx; f.in_anode = an[a].in[0]; f.final_anode = nx;
            owner[a] = owner[nx] = id;
        } else if (an[a].kind == A_MAXPOOL) {
            f.kind = LAYER_MAXPOOL; f.pool = a; f.in_anode = an[a].in[0]; f.final_anode = a;
            owner[a] = id;
        } else if (an[a].kind == A_RESIZE) {
            f.kind = LAYER_COPY; f.resize = a; f.in_anode = an[a].in[0]; f.final_anode = a; f.copy_up = 1;
            owner[a] = id;
        } else if (an[a].kind == A_MISH) {
            return B.fail("Mish '" + g.nodes[an[a].node].name + "' cannot be fused into a preceding convolution (it must follow the Conv or its BatchNormalization)");
        } else {
            const char* what = an[a].kind == A_BN ? "BatchNormalization" : an[a].kind == A_LEAKY ? "LeakyRelu" : "Add";
            return B.fail(std::string(what) + " '" + an[a].out_name + "' cannot be fused into a preceding convolution");
        }
        f.anchor = f.final_anode;
        ops.push_back(f);
    }

    // ------------------------------------------------------------------ pass 3: values + placement
    std::vector<Value> vals;
    auto new_value = [&](int anode) {
        Value v;
        v.loc.c = an[anode].c; v.loc.h = an[anode].h; v.loc.w = an[anode].w;
        vals.push_back(v);
        an[anode].value = static_cast<int>(vals.size()) - 1;
        return an[anode].value;
    };
    {
        const int v = new_value(input_id);
        vals[v].is_input = true; vals[v].placed = true;
        vals[v].loc.buf = -2; vals[v].loc.pitch = 3;
    }
    for (auto& f : ops) new_value(f.final_anode);
    for (int a = 0; a < static_cast<int>(an.size()); ++a) if (an[a].kind == A_CONCAT) new_value(a);
    for (int a = 0; a < static_cast<int>(an.size()); ++a) {
        if (an[a].kind != A_VIEW) continue;
        const int src = an[an[a].in[0]].value;
        if (src < 0) return B.fail("internal: the source of channel slice '" + an[a].out_name + "' has no value");
        const int v = new_value(a);
        vals[v].view_of = src;
        vals[v].view_start = an[a].view_start;
        // 16-byte alignment of every read through the view (TMA bases, cp.async)
        if (!an[a].consumers.empty() && (an[a].view_start % 8 || an[a].c % 8))
            return B.fail(g.nodes[an[a].node].name + ": channel slice [" + std::to_string(an[a].view_start) + ", " +
                          std::to_string(an[a].view_start + an[a].c) + ") must start and end on multiples of 8 channels");
    }
    // every consumed anode must carry a value (i.e. nobody reads the inside of a fused chain)
    for (int a = 0; a < static_cast<int>(an.size()); ++a) {
        if (an[a].value >= 0) continue;
        for (int cns : an[a].consumers)
            if (owner[cns] != owner[a]) return B.fail("tensor '" + an[a].out_name + "' is consumed both inside and outside a fused convolution");
        if (an[a].is_output) return B.fail("graph output '" + an[a].out_name + "' lies inside a fused convolution chain");
    }
    // heads: fp32 rows, produced by a plain conv chain
    for (int a : out_anodes) {
        const int op = owner[a];
        if (op < 0 || ops[op].kind != LAYER_CONV || ops[op].resize >= 0 || ops[op].final_anode != a)
            return B.fail("graph output '" + an[a].out_name + "' must be produced by a convolution");
        if (!an[a].consumers.empty()) return B.fail("graph output '" + an[a].out_name + "' is also consumed inside the graph");
        vals[an[a].value].fp32 = true;
    }
    auto new_buffer = [&](int pitch, int h, int w, int fp32) {
        BufferPlan b;
        b.pitch = pitch; b.h = h; b.w = w; b.fp32 = fp32;
        plan->buffers.push_back(b);
        return static_cast<int>(plan->buffers.size()) - 1;
    };
    for (int a = 0; a < static_cast<int>(an.size()); ++a) {
        if (an[a].kind != A_CONCAT) continue;
        const int total = an[a].c;
        if (total % 8) return B.fail("Concat '" + an[a].out_name + "': channel count must be a multiple of 8");
        const int buf = new_buffer(total, an[a].h, an[a].w, 0);
        Value& cv = vals[an[a].value];
        cv.loc.buf = buf; cv.loc.pitch = total; cv.loc.ch_off = 0; cv.placed = true;
        int off = 0;
        for (int in : an[a].in) {
            const int vi = an[in].value;
            if (vi < 0) return B.fail("Concat input '" + an[in].out_name + "' has no materialised value");
            Value& v = vals[vi];
            if (off % 8 || v.loc.c % 8) return B.fail("Concat '" + an[a].out_name + "': slices must start on multiples of 8 channels");
            if (!v.placed && !v.fp32 && v.view_of < 0) {  // (a view's channels are written by its source's producer)
                v.loc.buf = buf; v.loc.pitch = total; v.loc.ch_off = off; v.placed = true;
            } else {
                Fused f;
                f.kind = LAYER_COPY; f.anchor = a; f.final_anode = -1;
                f.copy_src_value = vi; f.copy_dst_buf = buf; f.copy_dst_off = off; f.copy_dst_pitch = total;
                ops.push_back(f);
            }
            off += v.loc.c;
        }
    }
    for (auto& v : vals) {
        if (v.placed || v.view_of >= 0) continue;
        const int pitch = v.fp32 ? (v.loc.c + 3) / 4 * 4 : v.loc.c;
        if (!v.fp32 && pitch % 8) return B.fail("activation channel counts must be multiples of 8");
        v.loc.buf = new_buffer(pitch, v.loc.h, v.loc.w, v.fp32 ? 1 : 0);
        v.loc.pitch = pitch; v.loc.ch_off = 0; v.placed = true;
    }
    // views last: the source may itself live in a concat buffer.  A view of a view was composed at creation.
    for (auto& v : vals) {
        if (v.view_of < 0) continue;
        const TensorLoc& src = vals[v.view_of].loc;
        v.loc.buf = src.buf; v.loc.pitch = src.pitch; v.loc.ch_off = src.ch_off + v.view_start; v.placed = true;
    }
    std::stable_sort(ops.begin(), ops.end(), [](const Fused& x, const Fused& y) { return x.anchor < y.anchor; });

    // ------------------------------------------------------------------ pass 4: layers + packed weights
    auto value_of = [&](int anode) -> const Value& { return vals[an[anode].value]; };
    for (const Fused& f : ops) {
        LayerPlan L;
        L.kind = f.kind;
        if (f.kind == LAYER_COPY && f.final_anode < 0) {  // concat fallback copy
            L.name = "concat_copy";
            L.in = vals[f.copy_src_value].loc;
            L.out = L.in;
            L.out.buf = f.copy_dst_buf; L.out.ch_off = f.copy_dst_off; L.out.pitch = f.copy_dst_pitch;
            plan->layers.push_back(L);
            continue;
        }
        const ANode& fin = an[f.final_anode];
        L.out_name = fin.out_name;
        L.out = value_of(f.final_anode).loc;
        if (an[f.in_anode].value < 0) return B.fail("internal: input of '" + fin.out_name + "' has no value");
        L.in = value_of(f.in_anode).loc;
        if (f.kind == LAYER_COPY) {
            L.name = g.nodes[an[f.resize].node].name;
            L.upsample2x = 1;
        } else if (f.kind == LAYER_MAXPOOL) {
            const ANode& p = an[f.pool];
            L.name = g.nodes[p.node].name;
            L.pool_k = p.ksize; L.pool_s = p.stride;
            if (f.pad >= 0) {
                L.pool_pad_lo = an[f.pad].pads[0]; L.pool_pad_hi = an[f.pad].pads[2];
                L.pad_value = an[f.pad].pad_value;
            } else {
                L.pool_pad_lo = p.pad_lo; L.pool_pad_hi = p.pad_hi;
                L.pad_value = -INFINITY;
            }
        } else {
            const ANode& cv = an[f.conv];
            const OnnxNode& n = g.nodes[cv.node];
            L.name = n.name.empty() ? cv.out_name : n.name;
            const OnnxTensor& W = *B.cst(n.inputs[1]);
            L.cout = static_cast<int>(W.dims[0]); L.cin = static_cast<int>(W.dims[1]);
            L.ksize = cv.ksize; L.stride = cv.stride; L.pad_lo = cv.pad_lo; L.pad_hi = cv.pad_hi;
            L.act = f.leaky < 0 ? 0 : an[f.leaky].kind == A_MISH ? 2 : 1;
            L.alpha = L.act == 1 ? an[f.leaky].alpha : 0.f;
            L.upsample2x = f.resize >= 0 ? 1 : 0;
            L.pool2 = f.pool >= 0 ? 1 : 0;
            L.out_fp32 = value_of(f.final_anode).fp32 ? 1 : 0;
            if (f.residual >= 0) {
                if (an[f.residual].value < 0) return B.fail("residual operand of '" + fin.out_name + "' has no value");
                L.res = value_of(f.residual).loc;
            }
            // fold BatchNormalization (ONNX: y = scale*(x-mean)/sqrt(var+eps) + B) and the conv bias, in fp32
            std::vector<float> scale(L.cout, 1.f), shift(L.cout, 0.f);
            if (n.inputs.size() > 2 && !n.inputs[2].empty()) {
                const OnnxTensor* b = B.cst(n.inputs[2]);
                if (!b || static_cast<int>(b->f.size()) != L.cout) return B.fail(L.name + ": Conv bias must be a constant of size Cout");
                shift = b->f;
            }
            if (f.bn >= 0) {
                const OnnxNode& bn = g.nodes[an[f.bn].node];
                const float eps = bn.attr_f("epsilon", 1e-5f);
                const std::vector<float>& gamma = B.cst(bn.inputs[1])->f;
                const std::vector<float>& beta = B.cst(bn.inputs[2])->f;
                const std::vector<float>& mean = B.cst(bn.inputs[3])->f;
                const std::vector<float>& var = B.cst(bn.inputs[4])->f;
                for (int co = 0; co < L.cout; ++co) {
                    const float inv = gamma[co] / sqrtf(var[co] + eps);
                    scale[co] = inv;
                    shift[co] = beta[co] + (shift[co] - mean[co]) * inv;
                }
            }
            const int k = L.ksize, K = k * k * L.cin;
            L.b_off = plan->bias_f32.size();
            plan->bias_f32.resize(L.b_off + (L.cout + 255) / 256 * 256, 0.f);
            memcpy(plan->bias_f32.data() + L.b_off, shift.data(), sizeof(float) * L.cout);
            if (f.kind == LAYER_CONV0) {
                if (L.stride == 2) {  // only the tensor-core form (conv0_ws_kernel) takes stride 2: dense Cout 16 / 32 rows
                    if (L.cin != 3 || k != 3 || L.pad_lo != 1 || L.pad_hi != 1 || !(L.cout == 16 || L.cout == 32) || L.out.pitch != L.cout ||
                        L.in.h % 2 || L.in.w % 2 || L.upsample2x || L.res.buf != -1 || L.out_fp32)
                        return B.fail(L.name + ": a stride-2 first convolution must be 3x3 pad 1 over 3 channels with Cout 16 or 32, "
                                      "on an even-sized input, into a tensor of its own");
                } else if (L.cin != 3 || k != 3 || L.stride != 1 || L.pad_lo != 1 || L.pad_hi != 1 || L.cout % 8 || L.cout > 64 || L.upsample2x || L.res.buf != -1 || L.out_fp32) {  // (pool2 only with Cout 16 / 32, checked where it is set)
                    return B.fail(L.name + ": the first convolution must be 3x3 stride 1 pad 1 over 3 channels with Cout in {8..64}, or 3x3 stride 2 with Cout 16 or 32");
                }
                L.w_off = plan->conv0_w.size();
                plan->conv0_w.resize(L.w_off + static_cast<size_t>(K) * L.cout);
                for (int co = 0; co < L.cout; ++co)
                    for (int ci = 0; ci < 3; ++ci)
                        for (int r = 0; r < 3; ++r)
                            for (int s = 0; s < 3; ++s)
                                plan->conv0_w[L.w_off + (static_cast<size_t>(r * 3 + s) * 3 + ci) * L.cout + co] =
                                    W.f[((static_cast<size_t>(co) * 3 + ci) * 3 + r) * 3 + s] * scale[co];
            } else {
                if (L.cin % 16) return B.fail(L.name + ": Cin must be a multiple of 16 for the tensor-core path");
                if (!L.out_fp32 && L.cout % 8) return B.fail(L.name + ": Cout must be a multiple of 8");
                L.w_off = (plan->weights_bf16.size() + 63) / 64 * 64;
                plan->weights_bf16.resize(L.w_off + static_cast<size_t>(L.cout) * K, 0);
                uint16_t* dst = plan->weights_bf16.data() + L.w_off;
                for (int co = 0; co < L.cout; ++co)
                    for (int ci = 0; ci < L.cin; ++ci)
                        for (int r = 0; r < k; ++r)
                            for (int s = 0; s < k; ++s)
                                dst[static_cast<size_t>(co) * K + static_cast<size_t>(r * k + s) * L.cin + ci] =
                                    f32_to_bf16_rn(W.f[((static_cast<size_t>(co) * L.cin + ci) * k + r) * k + s] * scale[co]);
            }
            const int ho = cv.h, wo = cv.w;
            L.flops = 2.0 * L.cout * L.cin * k * k * ho * wo;
            plan->conv_flops_per_frame += L.flops;
            plan->num_params += static_cast<size_t>(L.cout) * K + L.cout;
        }
        if (!out_anodes.empty() && fin.is_output) {
            // filled below in graph-output order
        }
        plan->layers.push_back(L);
    }
    // SPP groups: the stride-1 "same" max-pools (pads (k-1)/2 of -inf, from the MaxPool itself) of one tensor whose outputs
    // each go only into the same Concat, placed there directly, on maps whose slab fits the kernel's shared memory.  Up to
    // SPP_MAX_POOLS per launch; layers[i] is the layer of ops[i].
    {
        std::map<std::pair<int, int>, std::vector<int>> groups;  // (input value, Concat anode) -> layers
        for (size_t i = 0; i < ops.size(); ++i) {
            const Fused& f = ops[i];
            if (f.kind != LAYER_MAXPOOL || f.pad >= 0) continue;
            const ANode& p = an[f.pool];
            const LayerPlan& L = plan->layers[i];
            if (p.stride != 1 || p.ksize % 2 == 0 || p.pad_lo != p.ksize / 2 || p.pad_hi != p.ksize / 2) continue;
            if (p.is_output || p.consumers.size() != 1 || an[p.consumers[0]].kind != A_CONCAT) continue;
            if (L.out.buf != vals[an[p.consumers[0]].value].loc.buf || L.in.buf < 0 || !spp_fits(L.in.h, L.in.w)) continue;
            groups[{an[f.in_anode].value, p.consumers[0]}].push_back(static_cast<int>(i));
        }
        for (const auto& kv : groups) {
            const std::vector<int>& mem = kv.second;
            for (size_t s = 0; s + 1 < mem.size(); s += SPP_MAX_POOLS) {
                const size_t e = std::min(mem.size(), s + SPP_MAX_POOLS);
                if (e - s < 2) break;
                for (size_t j = s; j < e; ++j) plan->layers[mem[j]].spp = 1;
                LayerPlan& last = plan->layers[mem[e - 1]];
                last.spp = 2;
                last.spp_members.assign(mem.begin() + s, mem.begin() + e);
            }
        }
    }
    for (int a : out_anodes) {
        int found = -1;
        for (size_t i = 0; i < plan->layers.size(); ++i)
            if (plan->layers[i].out_name == an[a].out_name && plan->layers[i].kind == LAYER_CONV) found = static_cast<int>(i);
        if (found < 0) return B.fail("internal: no layer produces graph output '" + an[a].out_name + "'");
        plan->head_layers.push_back(found);
    }
    return true;
}

}  // namespace fd
