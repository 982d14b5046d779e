"""modelgen.py — synthetic YOLOv3 / YOLOv3-tiny / YOLOv4 / YOLOv4-tiny ONNX files with random-init weights.

The reference ships no model files (``*.onnx`` is git-ignored, reference .gitignore:5; README.md:38-48
names ``yolov3-full.onnx`` / ``yolov3-rsu.onnx`` / ``yolov3-tiny.onnx``), so tests and benchmarks
generate them.  The topologies are the public Darknet ``yolov3.cfg`` / ``yolov3-tiny.cfg`` / ``yolov4.cfg`` /
``yolov4-tiny.cfg``; the graph
contract is what reference server/detector.py:135-140 requires: one input named ``input`` (f32 NCHW,
range [0,1]) and 2 or 3 raw head maps ``[N, 3*(5+nc), S/32*k, S/32*k]``, coarsest first.

The file is written with a small hand protobuf encoder (the ``onnx`` package is not installed); the
exporter variants (BN folded or not, Resize vs Upsample, Pad+MaxPool vs padded MaxPool, initializers
vs Constant nodes, raw vs typed tensor data, Slice vs Split for YOLOv4-tiny's channel groups, one Mish node vs
Softplus -> Tanh -> Mul for YOLOv4's activation) exist so the native
loader is exercised on the forms real exporters emit.
"""
from __future__ import annotations

import struct
from dataclasses import dataclass, field
from typing import Dict, List, Optional, Sequence, Tuple

import numpy as np

# --------------------------------------------------------------------------- protobuf encoding


def _varint(v: int) -> bytes:
    if v < 0:
        v += 1 << 64
    out = bytearray()
    while True:
        b = v & 0x7F
        v >>= 7
        if v:
            out.append(b | 0x80)
        else:
            out.append(b)
            return bytes(out)


def _key(field_no: int, wire: int) -> bytes:
    return _varint((field_no << 3) | wire)


def _f_varint(field_no: int, v: int) -> bytes:
    return _key(field_no, 0) + _varint(v)


def _f_bytes(field_no: int, b: bytes) -> bytes:
    return _key(field_no, 2) + _varint(len(b)) + b


def _f_str(field_no: int, s: str) -> bytes:
    return _f_bytes(field_no, s.encode("utf-8"))


def _f_float(field_no: int, v: float) -> bytes:
    return _key(field_no, 5) + struct.pack("<f", v)


FLOAT, INT64 = 1, 7
ATTR_FLOAT, ATTR_INT, ATTR_STRING, ATTR_TENSOR, ATTR_FLOATS, ATTR_INTS = 1, 2, 3, 4, 6, 7


def tensor_proto(name: str, arr: np.ndarray, raw: bool = True) -> bytes:
    arr = np.asarray(arr)
    out = b""
    for d in arr.shape:
        out += _f_varint(1, int(d))
    if arr.dtype == np.float32:
        out += _f_varint(2, FLOAT)
        if raw:
            out += _f_bytes(9, arr.astype("<f4").tobytes())
        else:  # packed float_data
            out += _f_bytes(4, arr.astype("<f4").tobytes())
    elif arr.dtype == np.int64:
        out += _f_varint(2, INT64)
        if raw:
            out += _f_bytes(9, arr.astype("<i8").tobytes())
        else:  # unpacked int64_data (one varint per element), as torch's serializer writes repeated ints
            for v in arr.reshape(-1):
                out += _f_varint(7, int(v))
    else:
        raise TypeError(arr.dtype)
    if name:
        out += _f_str(8, name)
    return out


def attr_proto(name: str, value, packed: bool = True) -> bytes:
    out = _f_str(1, name)
    if isinstance(value, float):
        out += _f_float(2, value) + _f_varint(20, ATTR_FLOAT)
    elif isinstance(value, int):
        out += _f_varint(3, value) + _f_varint(20, ATTR_INT)
    elif isinstance(value, str):
        out += _f_bytes(4, value.encode()) + _f_varint(20, ATTR_STRING)
    elif isinstance(value, bytes):  # serialized TensorProto
        out += _f_bytes(5, value) + _f_varint(20, ATTR_TENSOR)
    elif isinstance(value, (list, tuple)) and value and isinstance(value[0], float):
        if packed:
            out += _f_bytes(7, b"".join(struct.pack("<f", v) for v in value))
        else:
            for v in value:
                out += _f_float(7, v)
        out += _f_varint(20, ATTR_FLOATS)
    elif isinstance(value, (list, tuple)):
        if packed:
            out += _f_bytes(8, b"".join(_varint(int(v)) for v in value))
        else:
            for v in value:
                out += _f_varint(8, int(v))
        out += _f_varint(20, ATTR_INTS)
    else:
        raise TypeError(type(value))
    return out


def node_proto(op: str, inputs: Sequence[str], outputs: Sequence[str], name: str = "", packed=True, **attrs) -> bytes:
    out = b""
    for i in inputs:
        out += _f_str(1, i)
    for o in outputs:
        out += _f_str(2, o)
    if name:
        out += _f_str(3, name)
    out += _f_str(4, op)
    for k, v in attrs.items():
        out += _f_bytes(5, attr_proto(k, v, packed=packed))
    return out


def value_info(name: str, shape: Sequence, elem_type: int = FLOAT) -> bytes:
    dims = b""
    for d in shape:
        if isinstance(d, str):
            dims += _f_bytes(1, _f_str(2, d))
        else:
            dims += _f_bytes(1, _f_varint(1, int(d)))
    tensor_type = _f_varint(1, elem_type) + _f_bytes(2, dims)
    return _f_str(1, name) + _f_bytes(2, _f_bytes(1, tensor_type))


def model_proto(graph: bytes, opset: int, producer: str = "fastdet_b200.modelgen") -> bytes:
    return (
        _f_varint(1, 7)  # ir_version
        + _f_str(2, producer)
        + _f_str(3, "1")
        + _f_bytes(7, graph)
        + _f_bytes(8, _f_str(1, "") + _f_varint(2, opset))
    )


# --------------------------------------------------------------------------- Darknet topologies


@dataclass
class Layer:
    kind: str  # conv | shortcut | route | upsample | maxpool | yolo
    filters: int = 0
    size: int = 1
    stride: int = 1
    bn: bool = True
    leaky: bool = True
    frm: Tuple[int, ...] = ()  # shortcut: (from,), route: layer indices (darknet-style, may be negative)
    res_tail: bool = False  # conv that closes a residual branch (its output feeds a shortcut)
    groups: int = 1  # route: keep channel group `group_id` of `groups` equal groups (CSP "route groups")
    group_id: int = 0
    mish: bool = False  # conv: Mish activation (then leaky is False)


def yolov3_layers(num_classes: int) -> List[Layer]:
    """Darknet yolov3.cfg: 75 convs, 23 shortcuts, 2 upsamples, 2 route-concats, 3 heads."""
    L: List[Layer] = []
    head_c = 3 * (5 + num_classes)

    def conv(f, k, s=1, bn=True, leaky=True, res_tail=False):
        L.append(Layer("conv", f, k, s, bn, leaky, res_tail=res_tail))

    def res(c):
        conv(c // 2, 1)
        conv(c, 3, res_tail=True)
        L.append(Layer("shortcut", frm=(-3,)))

    conv(32, 3)
    for c, reps in ((64, 1), (128, 2), (256, 8), (512, 8), (1024, 4)):
        conv(c, 3, 2)
        for _ in range(reps):
            res(c)
    # layer indices now match darknet: 36 = last 256-block output, 61 = last 512-block output
    for c in (512,):
        for _ in range(3):
            conv(c, 1)
            conv(c * 2, 3)
    conv(head_c, 1, bn=False, leaky=False)
    L.append(Layer("yolo"))
    L.append(Layer("route", frm=(-4,)))
    conv(256, 1)
    L.append(Layer("upsample", stride=2))
    L.append(Layer("route", frm=(-1, 61)))
    for _ in range(3):
        conv(256, 1)
        conv(512, 3)
    conv(head_c, 1, bn=False, leaky=False)
    L.append(Layer("yolo"))
    L.append(Layer("route", frm=(-4,)))
    conv(128, 1)
    L.append(Layer("upsample", stride=2))
    L.append(Layer("route", frm=(-1, 36)))
    for _ in range(3):
        conv(128, 1)
        conv(256, 3)
    conv(head_c, 1, bn=False, leaky=False)
    L.append(Layer("yolo"))
    return L


def yolov3_tiny_layers(num_classes: int) -> List[Layer]:
    """Darknet yolov3-tiny.cfg: 13 convs, 6 maxpools (the last one stride 1), 1 upsample, 2 heads."""
    L: List[Layer] = []
    head_c = 3 * (5 + num_classes)
    for c in (16, 32, 64, 128, 256):
        L.append(Layer("conv", c, 3, 1))
        L.append(Layer("maxpool", size=2, stride=2))
    L.append(Layer("conv", 512, 3, 1))
    L.append(Layer("maxpool", size=2, stride=1))
    L.append(Layer("conv", 1024, 3, 1))
    L.append(Layer("conv", 256, 1, 1))  # 13: branch point
    L.append(Layer("conv", 512, 3, 1))
    L.append(Layer("conv", head_c, 1, 1, bn=False, leaky=False))
    L.append(Layer("yolo"))
    L.append(Layer("route", frm=(-4,)))
    L.append(Layer("conv", 128, 1, 1))
    L.append(Layer("upsample", stride=2))
    L.append(Layer("route", frm=(-1, 8)))
    L.append(Layer("conv", 256, 3, 1))
    L.append(Layer("conv", head_c, 1, 1, bn=False, leaky=False))
    L.append(Layer("yolo"))
    return L


def yolov4_tiny_layers(num_classes: int) -> List[Layer]:
    """Darknet yolov4-tiny.cfg: 21 convs (the first two stride 2), 3 CSP stages whose route groups take the second
    half of a tensor's channels, 3 maxpools, 1 upsample, 2 heads (coarsest first)."""
    L: List[Layer] = []
    head_c = 3 * (5 + num_classes)
    L.append(Layer("conv", 32, 3, 2))
    L.append(Layer("conv", 64, 3, 2))
    for c in (64, 128, 256):  # layers 2-9, 10-17, 18-25
        L.append(Layer("conv", c, 3, 1))
        L.append(Layer("route", frm=(-1,), groups=2, group_id=1))
        L.append(Layer("conv", c // 2, 3, 1))
        L.append(Layer("conv", c // 2, 3, 1))
        L.append(Layer("route", frm=(-1, -2)))
        L.append(Layer("conv", c, 1, 1))
        L.append(Layer("route", frm=(-6, -1)))
        L.append(Layer("maxpool", size=2, stride=2))
    L.append(Layer("conv", 512, 3, 1))
    L.append(Layer("conv", 256, 1, 1))  # 27: branch point
    L.append(Layer("conv", 512, 3, 1))
    L.append(Layer("conv", head_c, 1, 1, bn=False, leaky=False))
    L.append(Layer("yolo"))
    L.append(Layer("route", frm=(-4,)))
    L.append(Layer("conv", 128, 1, 1))
    L.append(Layer("upsample", stride=2))
    L.append(Layer("route", frm=(-1, 23)))
    L.append(Layer("conv", 256, 3, 1))
    L.append(Layer("conv", head_c, 1, 1, bn=False, leaky=False))
    L.append(Layer("yolo"))
    return L


def yolov4_layers(num_classes: int) -> List[Layer]:
    """Darknet yolov4.cfg: 162 layers, 110 convs (72 Mish in the CSPDarknet53 backbone, 35 leaky in the neck, 3 linear
    heads), an SPP block (stride-1 max-pools 5, 9, 13 of one tensor, concatenated), a PAN neck.  The cfg lists the
    heads finest first; build_onnx emits them coarsest first, as the reference's decoder expects."""
    L: List[Layer] = []
    head_c = 3 * (5 + num_classes)

    def conv(f, k, s=1, act="mish", res_tail=False):
        L.append(Layer("conv", f, k, s, leaky=act == "leaky", mish=act == "mish", res_tail=res_tail))

    def route(*frm):
        L.append(Layer("route", frm=frm))

    def shortcut():
        L.append(Layer("shortcut", frm=(-3,)))

    conv(32, 3)                                   # 0
    conv(64, 3, 2)                                # 1
    conv(64, 1); route(-2); conv(64, 1)           # 2-4
    conv(32, 1); conv(64, 3, res_tail=True); shortcut()  # 5-7
    conv(64, 1); route(-1, -7); conv(64, 1)       # 8-10
    for c, reps, back in ((128, 2, -10), (256, 8, -28), (512, 8, -28), (1024, 4, -16)):  # ends at 23, 54, 85, 104
        conv(c, 3, 2)
        conv(c // 2, 1); route(-2); conv(c // 2, 1)
        for _ in range(reps):
            conv(c // 2, 1); conv(c // 2, 3, res_tail=True); shortcut()
        conv(c // 2, 1); route(-1, back); conv(c, 1)
    lk = "leaky"
    conv(512, 1, act=lk); conv(1024, 3, act=lk); conv(512, 1, act=lk)   # 105-107
    for i, k in enumerate((5, 9, 13)):                                  # SPP, 108-113
        if i:
            route(-2 * i)
        L.append(Layer("maxpool", size=k, stride=1))
    route(-1, -3, -5, -6)
    conv(512, 1, act=lk); conv(1024, 3, act=lk); conv(512, 1, act=lk)   # 114-116
    for c, lateral in ((256, 85), (128, 54)):                           # 117-126, 127-136
        conv(c, 1, act=lk); L.append(Layer("upsample", stride=2)); route(lateral); conv(c, 1, act=lk); route(-1, -3)
        for _ in range(2):
            conv(c, 1, act=lk); conv(2 * c, 3, act=lk)
        conv(c, 1, act=lk)
    for c, back in ((128, None), (256, -16), (512, -37)):              # heads at 52, 26, 13 (finest first, as in the cfg)
        if back is not None:
            route(-4); conv(c, 3, 2, act=lk); route(-1, back)
            for _ in range(2):
                conv(c, 1, act=lk); conv(2 * c, 3, act=lk)
            conv(c, 1, act=lk)
        conv(2 * c, 3, act=lk)
        L.append(Layer("conv", head_c, 1, 1, bn=False, leaky=False))
        L.append(Layer("yolo"))
    return L


ARCHS = {"full": yolov3_layers, "rsu": yolov3_layers, "tiny": yolov3_tiny_layers, "tiny4": yolov4_tiny_layers, "v4": yolov4_layers}


def conv_gflops(arch: str, num_classes: int, size: int) -> float:
    """Algorithmic conv FLOPs per frame (2*MACs), the figure the tensor roofline uses."""
    layers = ARCHS[arch](num_classes)
    shapes: List[Tuple[int, int]] = []  # (channels, spatial)
    c, s = 3, size
    fl = 0.0
    for i, l in enumerate(layers):
        if l.kind == "conv":
            so = s // l.stride
            fl += 2.0 * l.filters * c * l.size * l.size * so * so
            c, s = l.filters, so
        elif l.kind == "maxpool":
            s = s // l.stride
        elif l.kind == "upsample":
            s = s * 2
        elif l.kind == "route":
            idx = [j if j >= 0 else i + j for j in l.frm]
            c = sum(shapes[j][0] for j in idx) // l.groups
            s = shapes[idx[0]][1]
        elif l.kind == "shortcut":
            pass
        shapes.append((c, s))
    return fl * 1e-9


# --------------------------------------------------------------------------- ONNX emission


@dataclass
class ExportOptions:
    fold_bn: bool = True  # True: Conv(+bias) -> LeakyRelu ; False: Conv -> BatchNormalization -> LeakyRelu
    upsample_op: str = "Resize"  # "Resize" (opset 11, scales input) | "Upsample" (opset 9, scales input)
    pool_pad: str = "attr"  # "attr": MaxPool pads=[0,0,1,1] ; "pad_node": Pad(-inf..) is not valid ONNX, so
    # "pad_node" emits Pad(constant, value=-3.0e38) + MaxPool, the explicit form some converters use
    const_as: str = "initializer"  # "initializer" | "constant_node"
    raw_data: bool = True
    packed_attrs: bool = True
    batch: object = "N"  # declared batch dim: symbolic or an int (Unity export pins 1)
    bn_eps: float = 1e-5
    obj_fraction: float = 0.005  # share of anchor boxes whose objectness clears 0.11 on the calibration frames
    obj_spread: float = 1.5  # standard deviation of the objectness logits over positions
    head_gain: float = 1.0  # RMS of the head logits (calibrated)
    opset: int = 11
    split_op: str = "Slice"  # route groups: "Slice" (constant starts / ends inputs) | "Split" (sizes as the `split`
    # attribute below opset 13, as an input from 13 on)
    mish_op: str = "Mish"  # Mish layers: "Mish" (the ONNX op, opset 18) | "softplus" (Softplus -> Tanh -> Mul, as torch's
    # exporter writes nn.Mish at opsets below 18)
    mish_as_leaky: bool = False  # the same graph with LeakyRelu(0.1) in place of every Mish (the A/B twin for timing)


def _he_sigma(fan_in: int) -> float:
    # variance-preserving for LeakyReLU(0.1): E[f(x)^2] = (1 + 0.01)/2 * var
    return float(np.sqrt(2.0 / (1.01 * fan_in)))


def _he_sigma_mish(fan_in: int) -> float:
    # variance-preserving for Mish: E[mish(x)^2] = 0.452 * var for x ~ N(0, var)
    return float(np.sqrt(1.0 / (0.452 * fan_in)))


def _leaky(x):
    return np.where(x > 0, x, np.float32(0.1) * x)


def build_onnx(arch: str, num_classes: int, size: int = 416, seed: int = 0,
               opts: Optional[ExportOptions] = None) -> bytes:
    """Serialized ModelProto for `arch` in {"tiny", "full", "rsu", "tiny4", "v4"} with seeded random weights.

    Weights are the SURVEY §8d recipe — He-normal convs, BatchNorm gamma~U(.8,1.2), beta~N(0,.1),
    mean~N(0,.1), var~U(.8,1.2) — followed by one scalar per layer, fitted on two synthetic frames: each
    BatchNorm's affine pair (gamma, beta) is multiplied by k so the activation RMS after the LeakyReLU is ~1,
    residual branches end at 0.3x the RMS of the stream they are added to, and head logits have RMS
    `head_gain`, with the objectness channels biased so ~`obj_fraction` of the boxes become candidates.  Without the scalars
    the 23 residual adds let the RMS drift by three orders of magnitude, exp(tw) overflows and the boxes are
    garbage.  The statistics are deliberately NOT fitted per channel: subtracting a data-fitted per-channel
    mean from an untrained random net makes it amplify any perturbation (fp32-vs-fp64 noise grows 12x, bf16
    rounding reaches 10% at the heads in a CPU emulation), which says nothing about the kernels."""
    import torch
    import torch.nn.functional as F

    opts = opts or ExportOptions()
    layers = ARCHS[arch](num_classes)
    rng = np.random.default_rng(seed)
    nodes: List[bytes] = []
    inits: List[bytes] = []
    outputs: List[Tuple[str, Tuple]] = []
    names: List[str] = []  # output tensor name per darknet layer
    chans: List[int] = []
    spatial: List[int] = []
    acts: List = []  # calibration activations per darknet layer (torch f32 [1,C,H,W])

    def add_const(name: str, arr: np.ndarray):
        if opts.const_as == "constant_node":
            nodes.append(node_proto("Constant", [], [name], name=name + "_const",
                                    value=tensor_proto("", arr, raw=opts.raw_data)))
        else:
            inits.append(tensor_proto(name, arr, raw=opts.raw_data))

    def rms(t) -> float:
        return float(torch.sqrt(torch.mean(t.double() ** 2)))

    calib = np.stack([synthetic_frame(987654321 + seed + k, size) for k in range(2)])
    x = torch.from_numpy(np.ascontiguousarray((calib / 255).astype(np.float32).transpose(0, 3, 1, 2)))
    cur, c, s = "input", 3, size
    head_c = 3 * (5 + num_classes)
    n_conv = 0
    with torch.no_grad():
        for i, l in enumerate(layers):
            if l.kind == "conv":
                n_conv += 1
                tag = f"conv{n_conv}"
                fan_in = c * l.size * l.size
                pad = l.size // 2
                sigma = _he_sigma_mish(fan_in) if l.mish and not opts.mish_as_leaky else _he_sigma(fan_in)
                w = rng.normal(0.0, sigma, size=(l.filters, c, l.size, l.size)).astype(np.float32)
                conv_attrs = dict(dilations=[1, 1], group=1, kernel_shape=[l.size, l.size],
                                  pads=[pad, pad, pad, pad], strides=[l.stride, l.stride])
                out = f"{tag}_out"
                raw = F.conv2d(x, torch.from_numpy(w), None, stride=l.stride, padding=pad)
                if l.bn:
                    gamma = rng.uniform(0.8, 1.2, l.filters).astype(np.float32)
                    beta = rng.normal(0.0, 0.1, l.filters).astype(np.float32)
                    mean = rng.normal(0.0, 0.1, l.filters).astype(np.float32)
                    var = rng.uniform(0.8, 1.2, l.filters).astype(np.float32)
                    inv = 1.0 / np.sqrt(var + np.float32(opts.bn_eps))
                    y = (raw - torch.from_numpy(mean).view(1, -1, 1, 1)) * torch.from_numpy(gamma * inv).view(1, -1, 1, 1) \
                        + torch.from_numpy(beta).view(1, -1, 1, 1)
                    mish = l.mish and not opts.mish_as_leaky
                    a = F.mish(y) if mish else F.leaky_relu(y, 0.1) if (l.leaky or l.mish) else y
                    target = 1.0
                    if l.res_tail:
                        target = 0.3 * rms(acts[i - 2])  # the stream this branch is added to (shortcut from -3)
                    k = np.float32(target / max(rms(a), 1e-12))
                    gamma, beta = (gamma * k).astype(np.float32), (beta * k).astype(np.float32)
                    a = a * float(k)
                    if opts.fold_bn:
                        g_inv = (gamma * inv).astype(np.float32)
                        add_const(f"{tag}_w", (w * g_inv[:, None, None, None]).astype(np.float32))
                        add_const(f"{tag}_b", (beta - mean * g_inv).astype(np.float32))
                        nodes.append(node_proto("Conv", [cur, f"{tag}_w", f"{tag}_b"], [out], name=tag,
                                                packed=opts.packed_attrs, **conv_attrs))
                    else:
                        add_const(f"{tag}_w", w)
                        nodes.append(node_proto("Conv", [cur, f"{tag}_w"], [f"{tag}_raw"], name=tag,
                                                packed=opts.packed_attrs, **conv_attrs))
                        for nm, arr in (("gamma", gamma), ("beta", beta), ("mean", mean), ("var", var)):
                            add_const(f"{tag}_bn_{nm}", arr)
                        nodes.append(node_proto(
                            "BatchNormalization",
                            [f"{tag}_raw", f"{tag}_bn_gamma", f"{tag}_bn_beta", f"{tag}_bn_mean", f"{tag}_bn_var"],
                            [out], name=tag + "_bn", epsilon=float(opts.bn_eps), momentum=0.9))
                else:  # detection head: linear, bias, logits of RMS head_gain
                    k = np.float32(opts.head_gain / max(rms(raw), 1e-12))
                    w = (w * k).astype(np.float32)
                    b = np.zeros(l.filters, np.float32)
                    gain = np.full(l.filters, k, np.float32)
                    # objectness channels: a random net's channel is a big frame-wide offset plus a small
                    # position-dependent part, so a fixed bias yields either zero or thousands of candidates all
                    # sitting on the threshold.  Standardise these channels on the calibration frames (spread
                    # `obj_spread`) and place the bias so ~`obj_fraction` of the boxes clear sigmoid(obj) >= 0.11.
                    cut = float(np.log(0.11 / 0.89))
                    for ch in range(4, l.filters, 5 + num_classes):
                        v = raw[:, ch].reshape(-1).double()
                        # (capped: a channel that barely varies over positions would otherwise turn bf16
                        # rounding of its large common-mode part into logit noise)
                        gain[ch] = np.float32(min(opts.obj_spread / max(float(v.std()), 1e-12), 4.0 * float(k)))
                        b[ch] = cut - float(torch.quantile(v * float(gain[ch]), 1.0 - opts.obj_fraction))
                    w = (w * (gain / k)[:, None, None, None]).astype(np.float32)
                    raw = raw * torch.from_numpy(gain / k).view(1, -1, 1, 1)
                    a = raw * float(k) + torch.from_numpy(b).view(1, -1, 1, 1)
                    add_const(f"{tag}_w", w)
                    add_const(f"{tag}_b", b)
                    nodes.append(node_proto("Conv", [cur, f"{tag}_w", f"{tag}_b"], [out], name=tag,
                                            packed=opts.packed_attrs, **conv_attrs))
                if l.mish and not opts.mish_as_leaky:
                    if opts.mish_op == "Mish":
                        nodes.append(node_proto("Mish", [out], [f"{tag}_act"], name=tag + "_mish"))
                    elif opts.mish_op == "softplus":
                        nodes.append(node_proto("Softplus", [out], [f"{tag}_sp"], name=tag + "_softplus"))
                        nodes.append(node_proto("Tanh", [f"{tag}_sp"], [f"{tag}_tanh"], name=tag + "_tanh"))
                        nodes.append(node_proto("Mul", [out, f"{tag}_tanh"], [f"{tag}_act"], name=tag + "_mish"))
                    else:
                        raise ValueError(opts.mish_op)
                    out = f"{tag}_act"
                elif l.leaky or l.mish:
                    nodes.append(node_proto("LeakyRelu", [out], [f"{tag}_act"], name=tag + "_leaky", alpha=0.1))
                    out = f"{tag}_act"
                cur, c, s, x = out, l.filters, s // l.stride, a
            elif l.kind == "shortcut":
                j = i + l.frm[0]
                out = f"add{i}_out"
                nodes.append(node_proto("Add", [cur, names[j]], [out], name=f"add{i}"))
                cur, x = out, x + acts[j]
            elif l.kind == "route":
                idx = [j if j >= 0 else i + j for j in l.frm]
                if l.groups > 1:  # one channel group of one tensor: Slice or Split on axis 1
                    src, cs = names[idx[0]], chans[idx[0]]
                    gc = cs // l.groups
                    out = f"route{i}_out"
                    if opts.split_op == "Slice":
                        add_const(f"route{i}_starts", np.array([gc * l.group_id], np.int64))
                        add_const(f"route{i}_ends", np.array([gc * (l.group_id + 1) if l.group_id + 1 < l.groups else 2**63 - 1], np.int64))
                        add_const(f"route{i}_axes", np.array([1], np.int64))
                        nodes.append(node_proto("Slice", [src, f"route{i}_starts", f"route{i}_ends", f"route{i}_axes"], [out],
                                                name=f"route{i}"))
                    elif opts.split_op == "Split":
                        outs = [out if g == l.group_id else f"route{i}_part{g}" for g in range(l.groups)]
                        if opts.opset >= 13:
                            add_const(f"route{i}_split", np.full(l.groups, gc, np.int64))
                            nodes.append(node_proto("Split", [src, f"route{i}_split"], outs, name=f"route{i}", axis=1))
                        else:
                            nodes.append(node_proto("Split", [src], outs, name=f"route{i}", packed=opts.packed_attrs, axis=1,
                                                    split=[gc] * l.groups))
                    else:
                        raise ValueError(opts.split_op)
                    cur, c, s = out, gc, spatial[idx[0]]
                    x = acts[idx[0]][:, gc * l.group_id:gc * (l.group_id + 1)]
                elif len(idx) == 1:
                    cur, c, s, x = names[idx[0]], chans[idx[0]], spatial[idx[0]], acts[idx[0]]
                else:
                    out = f"concat{i}_out"
                    nodes.append(node_proto("Concat", [names[j] for j in idx], [out], name=f"concat{i}", axis=1))
                    cur, c, s = out, sum(chans[j] for j in idx), spatial[idx[0]]
                    x = torch.cat([acts[j] for j in idx], dim=1)
            elif l.kind == "upsample":
                out = f"up{i}_out"
                scales = np.array([1.0, 1.0, 2.0, 2.0], np.float32)
                add_const(f"up{i}_scales", scales)
                if opts.upsample_op == "Resize":
                    add_const(f"up{i}_roi", np.zeros((0,), np.float32))
                    nodes.append(node_proto("Resize", [cur, f"up{i}_roi", f"up{i}_scales"], [out], name=f"up{i}",
                                            coordinate_transformation_mode="asymmetric", mode="nearest",
                                            nearest_mode="floor"))
                elif opts.upsample_op == "Upsample":
                    nodes.append(node_proto("Upsample", [cur, f"up{i}_scales"], [out], name=f"up{i}", mode="nearest"))
                else:
                    raise ValueError(opts.upsample_op)
                cur, s = out, s * 2
                x = x.repeat_interleave(2, dim=2).repeat_interleave(2, dim=3)
            elif l.kind == "maxpool":
                out = f"pool{i}_out"
                if l.stride == 1 and l.size % 2:  # SPP: "same" padding of (k-1)/2 on every side
                    p = l.size // 2
                    nodes.append(node_proto("MaxPool", [cur], [out], name=f"pool{i}", packed=opts.packed_attrs,
                                            kernel_shape=[l.size, l.size], pads=[p, p, p, p], strides=[1, 1]))
                    x = F.max_pool2d(x, l.size, 1, p)
                elif l.stride == 1:
                    if opts.pool_pad == "pad_node":
                        pads = np.array([0, 0, 0, 0, 0, 0, 1, 1], np.int64)
                        add_const(f"pool{i}_pads", pads)
                        add_const(f"pool{i}_padval", np.array(-3.0e38, np.float32))
                        nodes.append(node_proto("Pad", [cur, f"pool{i}_pads", f"pool{i}_padval"],
                                                [f"pool{i}_padded"], name=f"pool{i}_pad", mode="constant"))
                        nodes.append(node_proto("MaxPool", [f"pool{i}_padded"], [out], name=f"pool{i}",
                                                packed=opts.packed_attrs, kernel_shape=[2, 2], pads=[0, 0, 0, 0],
                                                strides=[1, 1]))
                    else:
                        nodes.append(node_proto("MaxPool", [cur], [out], name=f"pool{i}", packed=opts.packed_attrs,
                                                kernel_shape=[2, 2], pads=[0, 0, 1, 1], strides=[1, 1]))
                    x = F.max_pool2d(F.pad(x, (0, 1, 0, 1), value=float("-inf")), 2, 1)
                else:
                    nodes.append(node_proto("MaxPool", [cur], [out], name=f"pool{i}", packed=opts.packed_attrs,
                                            kernel_shape=[l.size, l.size], pads=[0, 0, 0, 0],
                                            strides=[l.stride, l.stride]))
                    s = s // l.stride
                    x = F.max_pool2d(x, l.size, l.stride)
                cur = out
            elif l.kind == "yolo":
                outputs.append((cur, (opts.batch, head_c, s, s)))
            names.append(cur)
            chans.append(c)
            spatial.append(s)
            acts.append(x)

    if arch == "v4":
        outputs.reverse()  # coarsest first: the reference pairs graph output i with ANCHORS[3][i]
    graph = b"".join(_f_bytes(1, n) for n in nodes)
    graph += _f_str(2, {"tiny4": "yolov4-tiny", "v4": "yolov4"}.get(arch, f"yolov3-{arch}"))
    graph += b"".join(_f_bytes(5, t) for t in inits)
    graph += _f_bytes(11, value_info("input", (opts.batch, 3, size, size)))
    for name, shape in outputs:
        graph += _f_bytes(12, value_info(name, shape))
    opset = opts.opset if opts.upsample_op == "Resize" else 9
    if any(l.mish for l in layers) and opts.mish_op == "Mish" and not opts.mish_as_leaky:
        opset = max(opset, 18)  # (the Mish operator's first opset; Resize and MaxPool keep their meaning there)
    return model_proto(graph, opset)


def write_model(path: str, arch: str, num_classes: int, size: int = 416, seed: int = 0,
                opts: Optional[ExportOptions] = None) -> str:
    data = build_onnx(arch, num_classes, size, seed, opts)
    with open(path, "wb") as fp:
        fp.write(data)
    return path


def synthetic_frame(seed: int, size: int = 416) -> np.ndarray:
    """'dog-shaped' synthetic frame: matches the first two moments of the reference's testdata/dog.jpg
    (per-channel mean ~[135,136,116], sigma ~54; SURVEY §8d) with image-like spatial structure: a coarse
    16-pixel block pattern (sigma 50) plus 3x3-blurred pixel noise (sigma ~18), clipped to u8."""
    rng = np.random.default_rng(seed)
    mu = np.array([135.0, 136.0, 116.0])
    g = (size + 15) // 16
    coarse = rng.normal(0.0, 50.0, size=(g, g, 3)).repeat(16, axis=0).repeat(16, axis=1)[:size, :size]
    a = rng.normal(0.0, 54.0, size=(size + 2, size + 2, 3))
    fine = np.zeros((size, size, 3))
    for dy in range(3):
        for dx in range(3):
            fine += a[dy:dy + size, dx:dx + size]
    return np.clip(np.rint(mu + coarse + fine / 9.0), 0, 255).astype(np.uint8)


if __name__ == "__main__":
    import argparse

    ap = argparse.ArgumentParser(description="write a synthetic YOLOv3 ONNX file")
    ap.add_argument("arch", choices=sorted(ARCHS))
    ap.add_argument("path")
    ap.add_argument("-c", "--classes", type=int, default=80)
    ap.add_argument("-s", "--size", type=int, default=416)
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--unfolded-bn", action="store_true")
    a = ap.parse_args()
    write_model(a.path, a.arch, a.classes, a.size, a.seed, ExportOptions(fold_bn=not a.unfolded_bn))
    print(a.path, f"{conv_gflops(a.arch, a.classes, a.size):.3f} GFLOP/frame")
