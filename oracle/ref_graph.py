"""oracle/ref_graph.py — CPU fp32/fp64 (and bf16-operand) executor for the ONNX operator subset of the YOLOv3 graphs.

TEST INFRASTRUCTURE ONLY: imported by tests/, __graft_entry__.smoke() and bench.py's CPU-baseline
legs, never by the product path.

This restates, with ONNX-specification semantics, what ``self.model.run(None, {'input': a})`` does at
reference server/detector.py:135.  The arithmetic there lives in a third-party dependency that is
neither vendored nor version-pinned (``onnxruntime-gpu``, reference requirements.txt:3) and is not
installable in this image, and the reference holds no test vectors for it: PARITY UNPINNED at the
onnxruntime boundary.  What pins this file instead: (i) tests/test_oracle_graph.py checks it against
torch eager modules exported to ONNX by torch's own serializer (an independent writer + an independent
implementation of the same operators); (ii) it reads the same ``.onnx`` bytes the native loader reads.

Operators (ONNX opset 9-13 forms): Conv, BatchNormalization (inference), LeakyRelu, Relu, Add, Mul, MaxPool,
Resize / Upsample (nearest, asymmetric, floor), Concat, Pad (constant), Constant, Identity and the integer
shape-arithmetic ops torch's exporter emits around Resize/Pad (Shape, Gather, Cast, Slice, Unsqueeze,
Squeeze, Floor, Div, Sub, ConstantOfShape, Reshape, Transpose).

``dtype="bf16"`` evaluates the arithmetic BASELINE.json's north_star prescribes for the new implementation —
bf16 operands, fp32 accumulation — on the CPU: BatchNormalization is folded into the preceding Conv in fp32
(w' = w * gamma / sqrt(var + eps), b' = beta + (b - mean) * gamma / sqrt(var + eps)), the folded weights and every
convolution input are rounded to bf16 (round-to-nearest-even), products are summed in fp32, and every stored
activation (the value after LeakyRelu, and after a residual Add) is rounded to bf16; graph outputs stay fp32.
It separates the two sources of difference from the fp32 oracle: what the prescribed operand precision costs
(bf16 oracle vs fp32 oracle, a CPU-only comparison: tests/test_oracle_graph.py::test_bf16_operand_floor) and what
the CUDA kernels add on top (GPU vs bf16 oracle: fp32 summation order only).

``GraphExecutor.run_forced`` is the teacher-forced form of the bf16 mode: it evaluates every fused layer in float64 from an
implementation's own values of the layer's inputs, so that each layer of the CUDA path can be held to a rounding bound of
its own (tests/compare.py::layer_bound, tests/test_gpu_layers_exact.py).
"""
from __future__ import annotations

from typing import Dict, List, Optional

import numpy as np
import torch
import torch.nn.functional as F

from . import onnx_min


def _bf16(t: torch.Tensor) -> torch.Tensor:
    """Round-to-nearest-even to bf16, kept in fp32 storage."""
    return t.to(torch.bfloat16).to(torch.float32)


def _t(x, dtype=None):
    if isinstance(x, torch.Tensor):
        return x
    a = np.asarray(x)
    t = torch.from_numpy(a.copy())
    return t


class GraphExecutor:
    """Runs a parsed graph on torch-CPU.  ``dtype`` = torch.float32 (what ORT computes in), float64, or "bf16"
    (bf16 operands / fp32 accumulation, see the module docstring)."""

    def __init__(self, onnx_bytes: bytes, dtype=torch.float32, accumulate=torch.float32, fp32_tail: int = 0):
        """accumulate (bf16 mode): dtype the products are summed in — float64 gives the exactly-summed variant of the same
        bf16-operand arithmetic.  fp32_tail (bf16 mode): the last `fp32_tail` convolutions in front of every graph output
        keep fp32 weights and pass fp32 (unrounded) activations between them."""
        self.graph = onnx_min.load(onnx_bytes)
        self.bf16 = dtype == "bf16"
        self.accumulate = accumulate
        self.fp32_tail = int(fp32_tail)
        if self.bf16:
            dtype = torch.float32
        self.dtype = dtype
        self.consts: Dict[str, torch.Tensor] = {}
        for k, v in self.graph.initializers.items():
            t = torch.from_numpy(np.ascontiguousarray(v))
            if t.is_floating_point():
                t = t.to(dtype)
            self.consts[k] = t
        if "input" not in self.graph.inputs:
            # reference server/detector.py:135 feeds {'input': a}; any other name makes ORT raise
            raise KeyError(f"graph has no input named 'input' (inputs: {self.graph.inputs})")
        self.folded: Dict[str, tuple] = {}   # Conv output name -> (bf16-rounded folded weight, fp32 bias)
        self.bn_identity = set()             # BatchNormalization nodes folded into their producer
        self.round_after = set()             # node outputs that are stored activations (rounded to bf16)
        if self.bf16:
            self._prepare_bf16()

    def _prepare_bf16(self):
        g = self.graph
        consumers: Dict[str, list] = {}
        for n in g.nodes:
            for i in n.inputs:
                consumers.setdefault(i, []).append(n)
        outputs = set(g.outputs)

        def sole(name):
            c = consumers.get(name, [])
            return c[0] if len(c) == 1 and name not in outputs else None

        # the last fp32_tail convolutions in front of every graph output (walking back through the fused chain)
        producer = {n.outputs[0]: n for n in g.nodes}
        tail = set()
        for o in g.outputs:
            name, left = o, self.fp32_tail
            while left > 0 and name in producer:
                n = producer[name]
                if n.op == "Conv":
                    tail.add(id(n))
                    left -= 1
                name = n.inputs[0]
        self.tail = tail
        for n in g.nodes:
            if n.op == "Conv":
                w = self.consts[n.inputs[1]].to(torch.float32)
                b = self.consts[n.inputs[2]].to(torch.float32) if len(n.inputs) > 2 and n.inputs[2] else torch.zeros(w.shape[0])
                last = n
                nx = sole(n.outputs[0])
                if nx is not None and nx.op == "BatchNormalization" and nx.inputs[0] == n.outputs[0]:
                    sc, bb, mean, var = (self.consts[k].to(torch.float32) for k in nx.inputs[1:5])
                    eps = torch.tensor(nx.attrs.get("epsilon", 1e-5), dtype=torch.float32)
                    inv = sc / torch.sqrt(var + eps)
                    w = w * inv.view(-1, 1, 1, 1)
                    b = bb + (b - mean) * inv
                    self.bn_identity.add(id(nx))
                    last = nx
                self.folded[n.outputs[0]] = (w if id(n) in tail else _bf16(w), b)
                nx = sole(last.outputs[0])
                if nx is not None and nx.op in ("LeakyRelu", "Relu"):
                    last = nx
                # the value after the activation is what the conv kernel's epilogue rounds and stores; a graph output
                # (head tensor) is written in fp32
                feeds_tail = any(id(c) in tail for c in consumers.get(last.outputs[0], []))
                if last.outputs[0] not in outputs and not (id(n) in tail and feeds_tail):
                    self.round_after.add(last.outputs[0])
            elif n.op == "Add":
                if n.inputs[0] not in self.consts and n.inputs[1] not in self.consts and n.outputs[0] not in outputs:
                    self.round_after.add(n.outputs[0])  # residual add: bf16 + bf16, rounded once

    # -- single-op semantics -------------------------------------------------
    def _conv(self, n, x, w, b=None):
        a = n.attrs
        if a.get("group", 1) != 1:
            raise NotImplementedError("grouped conv")
        k = a.get("kernel_shape", list(w.shape[2:]))
        strides = a.get("strides", [1, 1])
        dil = a.get("dilations", [1, 1])
        auto = a.get("auto_pad", "NOTSET")
        if auto in ("NOTSET", ""):
            pads = a.get("pads", [0, 0, 0, 0])
        elif auto == "VALID":
            pads = [0, 0, 0, 0]
        else:  # SAME_UPPER / SAME_LOWER
            pads = [0, 0, 0, 0]
            for i, (inp, kk, s) in enumerate(zip(x.shape[2:], k, strides)):
                out = -(-inp // s)
                total = max((out - 1) * s + kk - inp, 0)
                lo = total // 2 if auto == "SAME_UPPER" else total - total // 2
                pads[i], pads[i + 2] = lo, total - lo
        t, l, bt, r = pads
        if (t, l) == (bt, r):
            return F.conv2d(x, w, b, stride=strides, padding=(t, l), dilation=dil)
        x = F.pad(x, (l, r, t, bt))
        return F.conv2d(x, w, b, stride=strides, dilation=dil)

    def _maxpool(self, n, x):
        a = n.attrs
        k = a["kernel_shape"]
        strides = a.get("strides", [1, 1])
        pads = a.get("pads", [0, 0, 0, 0])
        if a.get("ceil_mode", 0):
            raise NotImplementedError("ceil_mode")
        t, l, bt, r = pads
        if any(pads):
            x = F.pad(x, (l, r, t, bt), value=float("-inf"))  # ONNX MaxPool pads never win the max
        return F.max_pool2d(x, kernel_size=k, stride=strides)

    def _resize(self, n, x, ins):
        mode = n.attrs.get("mode", "nearest")
        if mode != "nearest":
            raise NotImplementedError(f"Resize mode {mode}")
        scales = None
        sizes = None
        if n.op == "Upsample":
            scales = ins[1] if len(ins) > 1 else torch.tensor(n.attrs["scales"])
        else:
            if len(ins) == 2:  # opset 10
                scales = ins[1]
            else:
                if len(ins) > 2 and ins[2] is not None and ins[2].numel() > 0:
                    scales = ins[2]
                if len(ins) > 3 and ins[3] is not None and ins[3].numel() > 0:
                    sizes = ins[3]
            ctm = n.attrs.get("coordinate_transformation_mode", "half_pixel")
            nm = n.attrs.get("nearest_mode", "round_prefer_floor")
            if len(ins) > 2 and not (ctm == "asymmetric" and nm == "floor"):
                # for integer upscaling of 2 the common modes coincide except half_pixel+round_prefer_floor,
                # which also equals pixel repetition for scale 2; accept and treat as repetition
                pass
        if sizes is not None:
            oh, ow = int(sizes[2]), int(sizes[3])
        else:
            oh, ow = int(x.shape[2] * float(scales[2])), int(x.shape[3] * float(scales[3]))
        fy, fx = oh // x.shape[2], ow // x.shape[3]
        if fy * x.shape[2] != oh or fx * x.shape[3] != ow:
            raise NotImplementedError("non-integer resize")
        return x.repeat_interleave(fy, dim=2).repeat_interleave(fx, dim=3)

    def _pad(self, n, ins):
        x = ins[0]
        if len(ins) > 1:
            pads = [int(v) for v in ins[1]]
            value = float(ins[2]) if len(ins) > 2 and ins[2] is not None and ins[2].numel() else 0.0
        else:
            pads = n.attrs["pads"]
            value = n.attrs.get("value", 0.0)
        if n.attrs.get("mode", "constant") != "constant":
            raise NotImplementedError("Pad mode")
        r = len(pads) // 2
        tp = []
        for d in reversed(range(r)):
            tp += [pads[d], pads[d + r]]
        return F.pad(x, tp, value=value)

    # -- graph walk ----------------------------------------------------------
    def run(self, x: np.ndarray, keep: Optional[List[str]] = None, all_values: bool = False):
        """x: [N,3,H,W] float array.  Returns the graph outputs as float32 numpy arrays (graph order),
        or a dict name->array when `keep`/`all_values` is given.  bf16 mode with accumulate=float64 keeps the sum, bias,
        activation and residual add in float64 and rounds once where an activation is stored."""
        vals: Dict[str, torch.Tensor] = dict(self.consts)
        vals["input"] = torch.from_numpy(np.ascontiguousarray(x)).to(self.dtype)
        vals[""] = None
        acc64 = self.bf16 and self.accumulate == torch.float64
        with torch.no_grad():
            for n in self.graph.nodes:
                ins = [vals.get(i) if i else None for i in n.inputs]
                out = self._node(n, ins, acc64)
                if n.outputs[0] in self.round_after:
                    out = _bf16(out)
                vals[n.outputs[0]] = out
        if all_values or keep is not None:
            names = keep if keep is not None else [k for k in vals if k and k not in self.consts]
            return {k: vals[k].to(torch.float32).numpy() for k in names if isinstance(vals.get(k), torch.Tensor)}
        return [vals[o].to(torch.float32).numpy() for o in self.graph.outputs]

    def run_forced(self, x: np.ndarray, overrides: Dict[str, np.ndarray], on_value=None):
        """Teacher-forced bf16 evaluation: predicts each fused layer of an implementation from that implementation's OWN
        inputs, so that a layer is judged by its own arithmetic and not by the rounding noise of every layer before it.

        x: [N,3,H,W] network input.  overrides: {value name: array} — the implementation's values of graph tensors (the
        library's fd_layer_desc.out_name of every layer: the value after all ops fused into that layer).  Every Conv uses the
        bf16 semantics of this executor (the folded bf16 weights of `self.folded`, bf16-rounded inputs); the sum, bias,
        activation and residual Add are evaluated in float64 and nothing is rounded to bf16 in between.  When a value named
        in `overrides` has been computed, its record is produced and the value is REPLACED by the override before any later
        node reads it, so Concat / Resize / MaxPool and the next convolutions see exactly the tensors the implementation's
        consumers read.  Record of a value (float64 tensors of the value's shape):
          r       the unrounded value;
          S       magnitude of the sums behind each element: conv(|x|, |w|) + |b| at the Conv (fp32), carried through the
                  activation, + |residual| at an Add, max-pooled / repeated by MaxPool / Resize; None for a value computed
                  exactly from overridden inputs (stand-alone MaxPool, Concat);
          K       cin * kh * kw of the convolution behind it (0 when S is None);
          m       magnitude for the rounding step: |r|, or for a MaxPool output the window maximum of |input|;
          pool    True for a MaxPool output;
          branch, S_branch   (residual Add only) the value after the activation, before the Add, and its S.
        Values not in `overrides` are carried unrounded (a convolution still rounds its input to bf16).
        on_value(name, record) is called for every overridden value; without it the records are returned as a dict."""
        if not self.bf16 or self.tail:
            raise ValueError("run_forced needs dtype='bf16' and fp32_tail=0")
        vals: Dict[str, torch.Tensor] = dict(self.consts)
        vals["input"] = torch.from_numpy(np.ascontiguousarray(x)).to(torch.float32)
        vals[""] = None
        mag: Dict[str, torch.Tensor] = {}   # computed (not overridden) values -> S
        ksz: Dict[str, int] = {}
        recs = {}

        def absval(i):
            return mag[i] if i in mag else vals[i].abs().double()

        with torch.no_grad():
            for n in self.graph.nodes:
                name, op = n.outputs[0], n.op
                ins = [vals.get(i) if i else None for i in n.inputs]
                out = self._node(n, ins, True)
                computed = [i for i in n.inputs if i in mag]
                if op == "Conv":
                    w16, bias = self.folded[name]
                    mag[name] = self._conv(n, _bf16(ins[0].float()).abs(), w16.abs(), bias.abs()).double()
                    ksz[name] = int(w16[0].numel())
                elif computed and op == "BatchNormalization" and id(n) not in self.bn_identity:
                    raise NotImplementedError("run_forced: BatchNormalization that is not folded into a Conv")
                elif computed and op in ("BatchNormalization", "LeakyRelu", "Relu", "Identity"):
                    mag[name], ksz[name] = mag[computed[0]], ksz[computed[0]]
                elif computed and op == "Add":
                    mag[name] = absval(n.inputs[0]) + absval(n.inputs[1])
                    ksz[name] = max(ksz[i] for i in computed)
                elif computed and op in ("MaxPool", "Resize", "Upsample", "Pad", "Concat"):
                    data = range(len(ins)) if op == "Concat" else [0]
                    m_ins = list(ins)
                    for j in data:
                        m_ins[j] = absval(n.inputs[j])
                    mag[name] = self._node(n, m_ins, True)
                    ksz[name] = max(ksz[i] for i in computed)
                if name in overrides:
                    rec = {"r": out.double(), "S": mag.get(name), "K": ksz.get(name, 0), "pool": op == "MaxPool"}
                    rec["m"] = self._maxpool(n, ins[0].double().abs()) if op == "MaxPool" else out.double().abs()
                    if op == "Add" and len(computed) == 1:
                        rec["branch"], rec["S_branch"] = vals[computed[0]].double(), mag[computed[0]]
                    if on_value is not None:
                        on_value(name, rec)
                    else:
                        recs[name] = rec
                    out = torch.as_tensor(np.ascontiguousarray(overrides[name]), dtype=torch.float32)
                    mag.pop(name, None)
                    ksz.pop(name, None)
                vals[name] = out
        return recs

    def _node(self, n, ins, acc64: bool):
        """One node's value.  acc64 (bf16 mode): the convolution sums its bf16 products in float64 and keeps float64."""
        op = n.op
        if op == "Conv" and self.bf16:
            w16, bias = self.folded[n.outputs[0]]
            xin = ins[0] if id(n) in self.tail else _bf16(ins[0])
            if acc64:
                out = self._conv(n, xin.double(), w16.double(), bias.double())
            else:
                out = self._conv(n, xin, w16, bias)
        elif op == "Conv":
            out = self._conv(n, *ins)
        elif op == "BatchNormalization" and id(n) in self.bn_identity:
            out = ins[0]
        elif op == "BatchNormalization":
            xx, sc, bb, mean, var = ins
            eps = n.attrs.get("epsilon", 1e-5)
            shp = (1, -1, 1, 1)
            out = sc.view(shp) * (xx - mean.view(shp)) / torch.sqrt(var.view(shp) + eps) + bb.view(shp)
        elif op == "LeakyRelu":
            out = F.leaky_relu(ins[0], float(np.float32(n.attrs.get("alpha", 0.01))))  # the kernels' fp32 alpha
        elif op == "Relu":
            out = F.relu(ins[0])
        elif op == "Add":
            out = ins[0] + ins[1]
        elif op == "Sub":
            out = ins[0] - ins[1]
        elif op == "Mul":
            out = ins[0] * ins[1]
        elif op == "Div":
            if not ins[0].is_floating_point() and not ins[1].is_floating_point():
                out = torch.div(ins[0], ins[1], rounding_mode="trunc")
            else:
                out = ins[0] / ins[1]
        elif op == "Floor":
            out = torch.floor(ins[0])
        elif op == "MaxPool":
            out = self._maxpool(n, ins[0])
        elif op in ("Resize", "Upsample"):
            out = self._resize(n, ins[0], ins)
        elif op == "Concat":
            axis = n.attrs.get("axis", 1)
            out = torch.cat([i for i in ins], dim=axis)
        elif op == "Pad":
            out = self._pad(n, ins)
        elif op == "Constant":
            v = n.attrs["value"]
            out = torch.from_numpy(np.ascontiguousarray(v))
            if out.is_floating_point():
                out = out.to(self.dtype)
        elif op == "Identity":
            out = ins[0]
        elif op == "Shape":
            out = torch.tensor(list(ins[0].shape), dtype=torch.int64)
        elif op == "Gather":
            axis = n.attrs.get("axis", 0)
            idx = ins[1].to(torch.int64)
            out = torch.index_select(ins[0], axis, idx.reshape(-1)).reshape(
                list(ins[0].shape[:axis]) + list(idx.shape) + list(ins[0].shape[axis + 1:]))
        elif op == "Cast":
            to = n.attrs["to"]
            out = ins[0].to({1: self.dtype, 6: torch.int32, 7: torch.int64, 11: torch.float64}[to])
        elif op == "Slice":
            if len(ins) > 1:
                starts, ends = [int(v) for v in ins[1]], [int(v) for v in ins[2]]
                axes = [int(v) for v in ins[3]] if len(ins) > 3 and ins[3] is not None else list(range(len(starts)))
                steps = [int(v) for v in ins[4]] if len(ins) > 4 and ins[4] is not None else [1] * len(starts)
            else:
                starts, ends = n.attrs["starts"], n.attrs["ends"]
                axes = n.attrs.get("axes", list(range(len(starts))))
                steps = [1] * len(starts)
            arr = ins[0].numpy()
            index = [slice(None)] * arr.ndim
            for s, e, ax, st in zip(starts, ends, axes, steps):
                # numpy slicing clamps exactly like the ONNX Slice specification (INT64 extremes included)
                index[ax] = slice(int(np.clip(s, -2**62, 2**62)), int(np.clip(e, -2**62, 2**62)), st)
                if st < 0 and e < -arr.shape[ax]:
                    index[ax] = slice(int(np.clip(s, -2**62, 2**62)), None, st)
            out = torch.from_numpy(np.ascontiguousarray(arr[tuple(index)]))
        elif op == "Unsqueeze":
            axes = n.attrs.get("axes") or [int(v) for v in ins[1]]
            out = ins[0]
            for ax in sorted(axes):
                out = out.unsqueeze(ax)
        elif op == "Squeeze":
            axes = n.attrs.get("axes") or ([int(v) for v in ins[1]] if len(ins) > 1 else None)
            out = ins[0]
            if axes is None:
                out = out.squeeze()
            else:
                for ax in sorted(axes, reverse=True):
                    out = out.squeeze(ax)
        elif op == "ConstantOfShape":
            v = n.attrs.get("value")
            fill = torch.from_numpy(np.ascontiguousarray(v)).reshape(-1)[0] if v is not None else torch.tensor(0.0)
            out = torch.full([int(d) for d in ins[0]], fill.item(), dtype=fill.dtype)
        elif op == "Reshape":
            out = ins[0].reshape([int(d) for d in ins[1]])
        elif op == "Transpose":
            out = ins[0].permute(n.attrs["perm"])
        else:
            raise NotImplementedError(f"oracle: ONNX op {op}")
        return out


class OrtSubstituteSession:
    """Duck-types the two onnxruntime.InferenceSession calls the reference makes (detector.py:118,135)."""

    def __init__(self, path_or_bytes, dtype=torch.float32):
        if isinstance(path_or_bytes, (bytes, bytearray)):
            data = bytes(path_or_bytes)
        else:
            with open(path_or_bytes, "rb") as fp:
                data = fp.read()
        self.exe = GraphExecutor(data, dtype)

    def run(self, output_names, feeds):
        assert output_names is None
        return self.exe.run(feeds["input"])
