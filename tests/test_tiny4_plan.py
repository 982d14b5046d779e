"""YOLOv4-tiny on the host side: channel Split / Slice as views, the stride-2 first convolution, and the generator.

CPU only: the planner runs on plan-only models (device=-1) and the oracle on torch-CPU."""
import hashlib

import numpy as np
import pytest
import torch
import torch.nn as nn
import torch.nn.functional as F

from fastdet_b200 import _native, modelgen
from fastdet_b200.modelgen import ExportOptions, model_proto, node_proto, tensor_proto, value_info
from oracle import ref_graph, ref_post
from tests import torch_export
from tests.split_oracle import SplitExecutor

KEYS = ("kind", "c", "h", "w", "cin", "ksize", "stride", "act", "has_residual", "upsample2x", "out_fp32", "flops")


def _layers(data, nc=80, size=416):
    m = _native.Model(data, nc, (size, size), device=-1)
    try:
        return [[l[k] for k in KEYS] for l in m.layers()]
    finally:
        m.close()


def test_tiny4_plan():
    data = modelgen.build_onnx("tiny4", 80, 416, seed=1)
    m = _native.Model(data, 80, (416, 416), device=-1)
    info = m.info
    # 21 convolutions, 3 stand-alone max-pools over concat buffers, one concat copy (layer 23 feeds two Concats);
    # the four route-group slices are views and launch nothing
    assert info.n_conv == 21 and info.n_layers == 25
    L = m.layers()
    assert [l["kind"] for l in L].count(2) == 3 and [l["kind"] for l in L].count(3) == 1
    assert m.head_shapes == [(255, 13, 13), (255, 26, 26)]
    assert (L[0]["kind"], L[0]["stride"], L[0]["c"], L[0]["h"], L[0]["w"], L[0]["cin"]) == (0, 2, 32, 208, 208, 3)
    assert round(info.conv_flops_per_frame * 1e-9, 3) == 6.908
    assert abs(info.conv_flops_per_frame * 1e-9 - modelgen.conv_gflops("tiny4", 80, 416)) < 1e-9
    assert round(modelgen.conv_gflops("tiny4", 80, 416), 3) == 6.908
    for n in (1, 64):
        assert m.planned_fusions(n) == (False, -1)
    m.close()


def test_tiny4_export_forms_plan_alike():
    base = _layers(modelgen.build_onnx("tiny4", 80, 416, seed=1))
    for opts in (ExportOptions(split_op="Split"), ExportOptions(split_op="Split", opset=13),
                 ExportOptions(split_op="Slice", opset=13), ExportOptions(fold_bn=False),
                 ExportOptions(split_op="Split", packed_attrs=False, const_as="constant_node", raw_data=False)):
        assert _layers(modelgen.build_onnx("tiny4", 80, 416, seed=1, opts=opts)) == base, opts


# build_onnx bytes of the YOLOv3 graphs at the seeds the tests and the benchmark use, recorded before YOLOv4-tiny was added
SHA256 = {
    ("full", 80, 416, 2): "ed59d0b3d25abd76ca8e8742a42b5a7ef7bae83d5ba5bb2b02e3179762fb0e00",
    ("rsu", 9, 416, 3): "0c0fe52faab6adb06a829fd5ff26d3f1c275b12a5b39bb435418ecaa1731a09d",
    ("tiny", 80, 416, 1): "0aef1788e4048ba366ed5ec6e17bff1950492ec0905433a639186008498406f8",
    ("full", 80, 160, 3): "d18af95be3de162e22acc1b3e4694ff6cbb0fd92b73a436a17f5aac1cae8b8be",
    ("rsu", 9, 160, 3): "7c7cd66b1864330aa9da16e793379f8cfc52b718cb36fe8127fd42a5c690a716",
    ("tiny", 5, 96, 2): "b1704ede1ffbd774c25818404de97db82beab11429c1d47da4969dded1668274",
    ("tiny", 3, 64, 1): "32e34bb24072e71405c06e07d0213b323b5b74202a0609fb699f19edc6556e73",
}


@pytest.mark.parametrize("key", sorted(SHA256))
def test_yolov3_graph_bytes_unchanged(key):
    arch, nc, size, seed = key
    assert hashlib.sha256(modelgen.build_onnx(arch, nc, size, seed)).hexdigest() == SHA256[key]


# ------------------------------------------------------------------------------------------- torch-exported channel slices
class CspNet(nn.Module):
    """Every way a PyTorch source writes a CSP route group: a constant slice, a slice through the tensor's own shape
    (Shape -> Gather -> Div -> Slice), torch.chunk and torch.split (Split); a stride-2 first convolution."""

    def __init__(self, nc=4):
        super().__init__()
        self.nc = nc
        conv = lambda ci, co, k, s=1: nn.Sequential(nn.Conv2d(ci, co, k, s, k // 2, bias=False), nn.BatchNorm2d(co))
        self.c1, self.c2 = conv(3, 32, 3, 2), conv(32, 64, 3)
        self.c3, self.c4, self.c5 = conv(32, 32, 3), conv(16, 32, 3), conv(32, 64, 3)
        self.h1 = nn.Conv2d(48, 3 * (5 + nc), 1)
        self.h2 = nn.Conv2d(64, 3 * (5 + nc), 1)
        for mod in self.modules():
            if isinstance(mod, nn.BatchNorm2d):
                nn.init.uniform_(mod.weight, 0.8, 1.2)
                nn.init.normal_(mod.bias, 0.0, 0.1)
                mod.running_mean.normal_(0.0, 0.1)
                mod.running_var.uniform_(0.8, 1.2)

    def forward(self, x):
        act = lambda t: F.leaky_relu(t, 0.1)
        a = act(self.c2(act(self.c1(x))))            # 64 @ S/2
        c = a.shape[1]
        b = act(self.c3(a[:, c // 2:]))              # constant slice -> 32
        d = act(self.c4(b[:, b.shape[1] // 2:]))     # slice through the shape chain -> 16 in, 32 out
        f = torch.cat([d, a[:, c // 2:]], 1)         # a view as a Concat input: 64
        g1, g2 = torch.chunk(F.max_pool2d(f, 2, 2), 2, dim=1)   # Split, equal parts: 32 @ S/4
        e = act(self.c5(g2))                         # 64
        _, h = torch.split(e, [16, 48], dim=1)       # Split with sizes
        return self.h1(F.max_pool2d(h, 2, 2)), self.h2(torch.cat([g1, g1], 1))


@pytest.mark.parametrize("opset", [11, 13])
def test_torch_exported_slices(opset):
    torch.manual_seed(0)
    net = CspNet().eval()
    data = torch_export.export(net, 64, opset=opset)
    x = torch.rand(2, 3, 64, 64)
    with torch.no_grad():
        want = [t.numpy() for t in net(x)]
    got = SplitExecutor(data).run(x.numpy())
    for g, w in zip(got, want):
        assert g.shape == w.shape
        np.testing.assert_allclose(g, w, rtol=1e-4, atol=1e-4 * np.abs(w).max())
    m = _native.Model(data, 4, (64, 64), device=-1)
    assert m.head_shapes == [(27, 8, 8), (27, 16, 16)]
    L = m.layers()
    assert L[0]["kind"] == 0 and L[0]["stride"] == 2 and m.info.n_conv == 7
    m.close()


# ------------------------------------------------------------------------------------------------ hand-built small graphs
class G:
    """A graph written node by node with the generator's protobuf helpers."""

    def __init__(self, seed=0):
        self.nodes, self.inits, self.rng, self.k = [], [], np.random.default_rng(seed), 0

    def const(self, arr):
        self.k += 1
        name = f"k{self.k}"
        self.inits.append(tensor_proto(name, np.asarray(arr)))
        return name

    def conv(self, x, cin, cout, k=3, s=1, pads=None, act=True, name=None):
        self.k += 1
        name = name or f"conv{self.k}"
        w = self.const(self.rng.normal(0, 0.2, (cout, cin, k, k)).astype(np.float32))
        b = self.const(self.rng.normal(0, 0.1, cout).astype(np.float32))
        p = pads if pads is not None else [k // 2] * 4
        self.nodes.append(node_proto("Conv", [x, w, b], [name + "_out"], name=name, kernel_shape=[k, k], pads=p, strides=[s, s]))
        if not act:
            return name + "_out"
        self.nodes.append(node_proto("LeakyRelu", [name + "_out"], [name + "_act"], name=name + "_leaky", alpha=0.1))
        return name + "_act"

    def op(self, op, ins, name, n_out=1, **attrs):
        outs = [f"{name}_out{i}" for i in range(n_out)] if n_out > 1 else [name + "_out"]
        self.nodes.append(node_proto(op, ins, outs, name=name, **attrs))
        return outs if n_out > 1 else outs[0]

    def slice(self, x, start, end, axis=1, step=None, name="cut"):
        ins = [x, self.const(np.array([start], np.int64)), self.const(np.array([end], np.int64)), self.const(np.array([axis], np.int64))]
        if step is not None:
            ins.append(self.const(np.array([step], np.int64)))
        return self.op("Slice", ins, name)

    def model(self, outputs, size):
        graph = b"".join(modelgen._f_bytes(1, n) for n in self.nodes) + modelgen._f_str(2, "g")
        graph += b"".join(modelgen._f_bytes(5, t) for t in self.inits)
        graph += modelgen._f_bytes(11, value_info("input", ("N", 3, size, size)))
        for o, c, s in outputs:
            graph += modelgen._f_bytes(12, value_info(o, ("N", c, s, s)))
        return model_proto(graph, 11)


def _net(cut=None, first=None, head_cut=False, size=64):
    """input -> conv 3->32 (s1, or `first` = (stride, pads, cout)) -> conv 32->64 s2 -> [cut(t)] -> conv -> two heads (nc = 1)."""
    g = G()
    s, pads, c0 = first or (1, [1, 1, 1, 1], 32)
    a = g.conv("input", 3, c0, 3, s, pads, name="first")
    r = size // s
    b = g.conv(a, c0, 64, 3, 2)
    x = cut(g, b) if cut else g.slice(b, 32, 64)
    c = g.conv(x, 32, 64, 3, 2)
    h1 = g.conv(c, 64, 18, 1, act=False, name="head1")
    h2 = g.conv(b, 64, 18, 1, act=False, name="head2")
    outs = [(h1, 18, r // 4), (h2, 18, r // 2)]
    if head_cut:
        outs[1] = (g.slice(h2, 0, 16, name="headcut"), 16, r // 2)
    return g.model(outs, size)


def test_small_net_plans():
    m = _native.Model(_net(), 1, (64, 64), device=-1)
    L = m.layers()
    assert m.info.n_layers == 5 and L[2]["cin"] == 32 and L[2]["h"] == 16
    m.close()


@pytest.mark.parametrize("case,want", [
    ("slice_h", ["cut", "axis 2"]),
    ("step2", ["cut", "step 2"]),
    ("start4", ["cut", "multiples of 8"]),
    ("input", ["cut", "network input"]),
    ("head", ["headcut", "channel slice"]),
    ("stride2_pads", ["first", "stride-2"]),
    ("stride2_cout64", ["first", "stride-2"]),
])
def test_planner_refusals(case, want):
    data = {
        "slice_h": lambda: _net(lambda g, t: g.slice(t, 0, 8, axis=2)),
        "step2": lambda: _net(lambda g, t: g.slice(t, 0, 64, step=2)),
        "start4": lambda: _net(lambda g, t: g.slice(t, 4, 36)),
        "input": lambda: _net(lambda g, t: g.conv(g.slice("input", 0, 3), 3, 32)),
        "head": lambda: _net(head_cut=True),
        "stride2_pads": lambda: _net(first=(2, [0, 0, 1, 1], 32)),
        "stride2_cout64": lambda: _net(first=(2, [1, 1, 1, 1], 64)),
    }[case]()
    with pytest.raises(_native.NativeError) as e:
        _native.Model(data, 1, (64, 64), device=-1)
    assert e.value.code == _native.FD_ERR_MODEL
    for w in want:
        assert w in e.value.msg, e.value.msg


def test_stride2_first_conv_plans():
    for cout in (16, 32):
        m = _native.Model(_net(first=(2, [1, 1, 1, 1], cout)), 1, (64, 64), device=-1)
        L0 = m.layers()[0]
        assert (L0["kind"], L0["stride"], L0["c"], L0["h"]) == (0, 2, cout, 32)
        m.close()


def test_split_outputs_nobody_reads():
    def cut(g, t):
        parts = g.op("Split", [t], "sp", n_out=3, axis=1, split=[4, 28, 32])  # misaligned, unread parts are fine
        return parts[2]
    m = _native.Model(_net(cut), 1, (64, 64), device=-1)
    assert m.info.n_layers == 5
    m.close()


def _block_net(slice_mid):
    """YOLOv3's first residual block shape (1x1 64->32, 3x3 32->64 + Add at 80x80): fused by conv_block_kernel unless
    the block's middle tensor has another reader, here a channel slice of it."""
    g = G(1)
    a = g.conv("input", 3, 32, 3)
    b = g.conv(a, 32, 64, 3, 2)                      # block input (160 -> 80)
    mid = g.conv(b, 64, 32, 1, name="mid")           # 1x1
    c = g.conv(mid, 32, 64, 3, name="tail")
    add = g.op("Add", [c, b], "add")
    side = g.conv(g.slice(mid if slice_mid else b, 16, 32), 16, 16, 1)
    cat = g.op("Concat", [add, side], "cat", axis=1)
    h1 = g.conv(g.conv(add, 64, 64, 3, 2), 64, 18, 1, act=False, name="head1")
    h2 = g.conv(cat, 80, 18, 1, act=False, name="head2")
    return g.model([(h1, 18, 40), (h2, 18, 80)], 160)


def test_sliced_block_middle_is_not_fused():
    m = _native.Model(_block_net(False), 1, (160, 160), device=-1)
    assert m.planned_fusions(8)[1] == 2  # control: the block's input may be sliced, the pair still fuses
    m.close()
    m = _native.Model(_block_net(True), 1, (160, 160), device=-1)
    L = m.layers()
    assert L[2]["name"] == "mid" and m.planned_fusions(8)[1] == -1
    m.close()


# ---------------------------------------------------------------------------------------------------- oracle and floor
def test_oracle_split_and_slice_forms_agree():
    x = ref_post.normalise(modelgen.synthetic_frame(200, 128))
    outs = [SplitExecutor(modelgen.build_onnx("tiny4", 80, 128, seed=1, opts=o)).run(x)
            for o in (None, ExportOptions(split_op="Split"), ExportOptions(split_op="Split", opset=13))]
    for o in outs[1:]:
        for a, b in zip(outs[0], o):
            assert np.array_equal(a, b)


def test_forced_oracle_reads_views_of_the_forced_tensors():
    """run_forced on the Slice form (the executor as it is) and on the Split form (Split parts) gives the same records
    when every layer's value is forced: each view is taken from the forced tensor of its source."""
    x = ref_post.normalise(modelgen.synthetic_frame(201, 128))
    slice_data = modelgen.build_onnx("tiny4", 80, 128, seed=1)
    m = _native.Model(slice_data, 80, (128, 128), device=-1)
    names = [l["out_name"] for l in m.layers() if l["out_name"]]
    m.close()
    vals = ref_graph.GraphExecutor(slice_data, dtype="bf16").run(x, keep=names)
    over = {k: (v + np.float32(1 / 64)).astype(np.float32) for k, v in vals.items()}  # forced values differ from computed ones
    recs = []
    for exe in (ref_graph.GraphExecutor(slice_data, dtype="bf16"),
                SplitExecutor(modelgen.build_onnx("tiny4", 80, 128, seed=1, opts=ExportOptions(split_op="Split", opset=13)), dtype="bf16")):
        recs.append(exe.run_forced(x, over))
    assert sorted(recs[0]) == sorted(recs[1]) == sorted(names)
    for k in names:
        assert torch.equal(recs[0][k]["r"], recs[1][k]["r"]), k


def tiny4_floor(frames=3, seed=1):
    """Detection spread of the bf16-operand oracle against the fp32 oracle on tiny4 (the measure of
    tests/test_oracle_graph.py::test_bf16_operand_floor): (head err, IoUs, |dconf|s, candidates per frame)."""
    data = modelgen.build_onnx("tiny4", 80, 416, seed)
    e32, e16 = ref_graph.GraphExecutor(data), ref_graph.GraphExecutor(data, dtype="bf16")
    herr, ious, dconfs, cands = [], [], [], []
    for s in range(frames):
        x = ref_post.normalise(modelgen.synthetic_frame(200 + s, 416))
        h32, h16 = e32.run(x), e16.run(x)
        herr.append(max(float(np.abs(a - b).max() / np.abs(a).max()) for a, b in zip(h32, h16)))
        i, d = ref_post.detection_spread(h32, h16, 80, (416, 416), 0.1)
        ious.extend(i)
        dconfs.extend(d)
        cands.append(len(ref_post.detect_from_heads(h32, 0, 80, (416, 416), 0.1)[0]))
    return max(herr), np.array(ious), np.array(dconfs), cands


def test_tiny4_bf16_operand_floor():
    herr, ious, dconfs, cands = tiny4_floor()
    print(f"tiny4 bf16-operand vs fp32 oracle: head err {herr:.4f}, {len(ious)} matched boxes, IoU min {ious.min():.4f} "
          f"median {np.median(ious):.4f}, |dconf| max {dconfs.max():.4f}; detections per frame {cands}")
    assert herr <= 2e-2
    assert min(cands) >= 10  # calibrated like the other archs: tens of detections per frame at 0.1
    assert ious.min() >= 0.95 and np.median(ious) >= 0.98 and dconfs.max() <= 1e-2
