"""YOLOv4 on the host side: Mish (one node, or Softplus -> Tanh -> Mul) as a fused convolution's activation, the SPP
max-pools as one launch, the generator's v4 arch, the Mish oracle and the Mish form of the rounding model.

CPU only: the planner runs on plan-only models (device=-1) and the oracle on torch-CPU."""
import hashlib

import numpy as np
import pytest
import torch
import torch.nn as nn
import torch.nn.functional as F

from fastdet_b200 import _native, modelgen
from fastdet_b200.modelgen import ExportOptions
from oracle import ref_graph, ref_post
from tests import torch_export
from tests.compare import U
from tests.mish_compare import MISH_C, check_layer
from tests.mish_oracle import MishExecutor
from tests.test_tiny4_plan import G

KEYS = ("kind", "c", "h", "w", "cin", "ksize", "stride", "act", "has_residual", "upsample2x", "out_fp32", "flops")


def _layers(data, nc=80, size=416):
    m = _native.Model(data, nc, (size, size), device=-1)
    try:
        return [[l[k] for k in KEYS] for l in m.layers()]
    finally:
        m.close()


def test_v4_plan():
    data = modelgen.build_onnx("v4", 80, 416, seed=1)
    m = _native.Model(data, 80, (416, 416), device=-1)
    info, L = m.info, m.layers()
    # 110 convolutions and the 3 SPP pools; the route concats are shared buffers, the x2 upsamples fused into their convs
    assert info.n_conv == 110 and info.n_layers == 113
    # one launch per layer + 2 (post-processing), less the two SPP pools the group's launch computes
    assert info.launches_per_detect == info.n_layers + 2 - 2
    assert m.head_shapes == [(255, 13, 13), (255, 26, 26), (255, 52, 52)]  # coarsest first
    assert abs(info.conv_flops_per_frame * 1e-9 - modelgen.conv_gflops("v4", 80, 416)) < 1e-9
    assert round(modelgen.conv_gflops("v4", 80, 416), 2) == 60.10
    acts = [l["act"] for l in L if l["kind"] in (0, 1)]
    assert acts.count(2) == 72 and acts.count(1) == 35 and acts.count(0) == 3
    assert L[0]["kind"] == 0 and L[0]["act"] == 2  # the first layer is a Mish layer
    pools = [(i, l["name"]) for i, l in enumerate(L) if l["kind"] == 2]
    assert [n for _, n in pools] == ["pool108", "pool110", "pool112"] and pools[2][0] - pools[0][0] == 2
    for n in (1, 64):  # YOLOv4's first layers have the fused stem's and block's shapes, but those kernels are LeakyReLU only
        assert m.planned_fusions(n) == (False, -1)
    m.close()
    twin = _native.Model(modelgen.build_onnx("v4", 80, 416, seed=1, opts=ExportOptions(mish_as_leaky=True)), 80, (416, 416), device=-1)
    assert [l["act"] for l in twin.layers() if l["kind"] in (0, 1)].count(1) == 107
    assert twin.planned_fusions(64) == (True, 4)  # the leaky twin does take them (block: the first CSP block's 1x1 + 3x3)
    twin.close()


def test_v4_generator_layers():
    L = modelgen.yolov4_layers(80)
    assert len(L) == 162 and sum(l.kind == "conv" for l in L) == 110 and sum(l.mish for l in L) == 72
    assert [l.size for l in L if l.kind == "maxpool"] == [5, 9, 13]


def test_v4_export_forms_plan_alike():
    base = _layers(modelgen.build_onnx("v4", 80, 160, seed=1), size=160)
    for opts in (ExportOptions(mish_op="softplus"), ExportOptions(mish_op="softplus", opset=13), ExportOptions(fold_bn=False),
                 ExportOptions(mish_op="softplus", fold_bn=False)):
        assert _layers(modelgen.build_onnx("v4", 80, 160, seed=1, opts=opts), size=160) == base, opts


# build_onnx bytes of YOLOv4-tiny, recorded before YOLOv4 was added (the YOLOv3 graphs are pinned in test_tiny4_plan.py)
SHA256 = {
    ("tiny4", 80, 416, 1): "bb72bef67e3de338d02f9c549f43fca46043014873f694044a24b76309e7cf17",
    ("tiny4", 80, 128, 1): "aade0b2f7cd464c95634c858c3e0b4467392d3bfe3a103ce3127f3cabfc7a603",
}


@pytest.mark.parametrize("key", sorted(SHA256))
def test_tiny4_graph_bytes_unchanged(key):
    arch, nc, size, seed = key
    assert hashlib.sha256(modelgen.build_onnx(arch, nc, size, seed)).hexdigest() == SHA256[key]


# ------------------------------------------------------------------------------------- torch-exported Mish and SPP
class MishSpp(nn.Module):
    """nn.Mish after conv + BN (a residual Add after one of them), a stride-2 conv, and an SPP block (max-pools 5, 9, 13 of
    one tensor, concatenated with it) between a leaky conv and two linear heads."""

    def __init__(self, nc=4):
        super().__init__()
        conv = lambda ci, co, k, s=1: nn.Sequential(nn.Conv2d(ci, co, k, s, k // 2, bias=False), nn.BatchNorm2d(co))
        self.c1, self.c2, self.c3, self.c4 = conv(3, 32, 3), conv(32, 64, 3, 2), conv(64, 32, 1), conv(32, 64, 3)
        self.c5, self.c6 = conv(64, 32, 1), conv(128, 64, 1)
        self.h1 = nn.Conv2d(64, 3 * (5 + nc), 1)
        self.h2 = nn.Conv2d(64, 3 * (5 + nc), 1)
        self.mish = nn.Mish()
        for mod in self.modules():
            if isinstance(mod, nn.BatchNorm2d):
                nn.init.uniform_(mod.weight, 0.8, 1.2)
                nn.init.normal_(mod.bias, 0.0, 0.1)
                mod.running_mean.normal_(0.0, 0.1)
                mod.running_var.uniform_(0.8, 1.2)

    def forward(self, x):
        a = self.mish(self.c2(self.mish(self.c1(x))))        # 64 @ S/2
        a = self.mish(self.c4(self.mish(self.c3(a)))) + a     # residual after the Mish
        b = F.leaky_relu(self.c5(a), 0.1)                     # 32
        spp = torch.cat([F.max_pool2d(b, 13, 1, 6), F.max_pool2d(b, 9, 1, 4), F.max_pool2d(b, 5, 1, 2), b], 1)
        c = F.leaky_relu(self.c6(spp), 0.1)
        return self.h1(F.max_pool2d(c, 2, 2)), self.h2(c)


@pytest.mark.parametrize("opset", [11, 13])
def test_torch_exported_mish_and_spp(opset):
    torch.manual_seed(0)
    net = MishSpp().eval()
    data = torch_export.export(net, 32, opset=opset)  # (SPP at 16 x 16: a 32 x 32 slab would not fit the kernel)
    ops = {n.op for n in __import__("oracle.onnx_min", fromlist=["load"]).load(data).nodes}
    assert {"Softplus", "Tanh", "Mul"} <= ops  # nn.Mish as torch writes it below opset 18
    x = torch.rand(2, 3, 32, 32)
    with torch.no_grad():
        want = [t.numpy() for t in net(x)]
    got = MishExecutor(data).run(x.numpy())
    for g, w in zip(got, want):
        assert g.shape == w.shape
        np.testing.assert_allclose(g, w, rtol=1e-4, atol=1e-4 * np.abs(w).max())
    m = _native.Model(data, 4, (32, 32), device=-1)
    assert m.head_shapes == [(27, 8, 8), (27, 16, 16)]
    L = m.layers()
    assert [l["act"] for l in L if l["kind"] in (0, 1)] == [2, 2, 2, 2, 1, 1, 0, 0]
    assert [l["has_residual"] for l in L if l["kind"] == 1][2] == 1
    assert m.info.launches_per_detect == m.info.n_layers + 2 - 2  # three SPP pools, one launch
    m.close()


def test_mish_oracle_forms_agree():
    """The Mish-node and Softplus-chain files give the same values in every mode, and run_forced tags the Mish layers."""
    x = ref_post.normalise(modelgen.synthetic_frame(200, 96))
    a = modelgen.build_onnx("v4", 80, 96, seed=1)
    b = modelgen.build_onnx("v4", 80, 96, seed=1, opts=ExportOptions(mish_op="softplus"))
    for kw in ({}, {"dtype": "bf16"}):
        for u, v in zip(MishExecutor(a, **kw).run(x), MishExecutor(b, **kw).run(x)):
            assert np.array_equal(u, v)
    m = _native.Model(a, 80, (96, 96), device=-1)
    L = m.layers()
    m.close()
    names = [l["out_name"] for l in L]
    vals = MishExecutor(a, dtype="bf16").run(x, keep=names)
    recs = MishExecutor(a, dtype="bf16").run_forced(x, vals)
    assert sorted(recs) == sorted(names)
    tagged = {n for n, r in recs.items() if r.get("act") == "mish"}
    assert tagged == {l["out_name"] for l in L if l["act"] == 2}


# ------------------------------------------------------------------------------------------------ hand-built refusals
def _refused(build, want):
    g = G()
    a = g.conv("input", 3, 32, 3, name="first")
    out = build(g, a)
    data = g.model([(g.conv(out, 32, 18, 1, act=False, name="head"), 18, 64)], 64)
    with pytest.raises(_native.NativeError) as e:
        _native.Model(data, 1, (64, 64), device=-1)
    assert e.value.code == _native.FD_ERR_MODEL
    for w in want:
        assert w in e.value.msg, e.value.msg


def _raw_conv(g, x, name):
    return g.conv(x, 32, 32, 3, act=False, name=name)


def _chain(g, x, mul_other=None, name="m"):
    sp = g.op("Softplus", [x], name + "_sp")
    th = g.op("Tanh", [sp], name + "_tanh")
    return g.op("Mul", [th, mul_other or x], name + "_mul")


@pytest.mark.parametrize("case,want", [
    ("mul_other", ["m_mul", "other than x"]),
    ("tanh_alone", ["lone_tanh", "Tanh"]),
    ("softplus_alone", ["lone_sp", "Softplus"]),
    ("mish_after_add", ["late_mish", "cannot be fused"]),
    ("chain_after_add", ["m_mul", "cannot be fused"]),
    ("tanh_two_readers", ["m_tanh", "Tanh"]),
])
def test_mish_refusals(case, want):
    def build(g, a):
        c = _raw_conv(g, a, "c")
        if case == "mul_other":
            return _chain(g, c, mul_other=_raw_conv(g, a, "d"))
        if case == "tanh_alone":
            return g.op("Tanh", [c], "lone_tanh")
        if case == "softplus_alone":
            return g.op("Mul", [c, g.op("Softplus", [c], "lone_sp")], "spmul")
        if case == "mish_after_add":
            return g.op("Mish", [g.op("Add", [c, a], "add")], "late_mish")
        if case == "chain_after_add":
            return _chain(g, g.op("Add", [c, a], "add"))
        if case == "tanh_two_readers":
            m = _chain(g, c)
            return g.op("Add", [m, "m_tanh_out"], "add2")
    _refused(build, want)


def test_mish_forms_plan():
    for form in ("node", "chain", "chain_swapped"):
        def build(g, a, form=form):
            c = _raw_conv(g, a, "c")
            if form == "node":
                return g.op("Mish", [c], "mish")
            sp = g.op("Tanh", [g.op("Softplus", [c], "sp")], "th")
            return g.op("Mul", [c, sp] if form == "chain" else [sp, c], "mul")
        g = G()
        a = g.conv("input", 3, 32, 3, name="first")
        data = g.model([(g.conv(build(g, a), 32, 18, 1, act=False, name="head"), 18, 64)], 64)
        m = _native.Model(data, 1, (64, 64), device=-1)
        assert [l["act"] for l in m.layers()] == [1, 2, 0], form
        m.close()


# --------------------------------------------------------------------------------------------------- rounding model
LOG2E = np.float32(1.44269504088896341)


def _fma32(a, b, c):
    return (a.astype(np.float64) * b.astype(np.float64) + c.astype(np.float64)).astype(np.float32)


def device_mish(x):
    """fastdet_b200/csrc/act.cuh in float32 (ex2.approx taken as exp2 rounded to float32)."""
    x = np.asarray(x, np.float32)
    with np.errstate(over="ignore", invalid="ignore"):
        e = np.exp2((x * LOG2E).astype(np.float32)).astype(np.float32)
        n = (e * (e + np.float32(2))).astype(np.float32)
        d = (n + np.float32(2)).astype(np.float32)
        r = (np.int32(0x7EF311C3) - d.view(np.int32)).view(np.float32)
        for _ in range(3):
            r = _fma32(r, _fma32(-d, r, np.ones_like(d)), r)
        y = (x * (n * r).astype(np.float32)).astype(np.float32)
    return np.where(x > 20, x, y)


def _exact_mish(x):
    x = np.asarray(x, np.float64)
    return x * np.tanh(np.logaddexp(x, 0.0))


def _bf16(v):
    return torch.from_numpy(np.asarray(v, np.float32)).to(torch.bfloat16).float().numpy()


def _sweep():
    x = np.linspace(-40, 40, 800001, dtype=np.float32)
    return np.concatenate([x, np.float32([-100, -88, -87, -20, -1e-30, 0, 1e-30, 19.999, 20, 20.001, 44, 89, 1e4])])


def _judge(g, x):
    rec = {"r": _exact_mish(x), "S": np.abs(x.astype(np.float64)), "K": 0, "m": np.abs(_exact_mish(x)), "act": "mish"}
    return check_layer(g, rec)


def test_reciprocal_first_guess():
    d = np.float32(2) ** np.linspace(1, 60, 400001, dtype=np.float32)
    r0 = (np.int32(0x7EF311C3) - d.view(np.int32)).view(np.float32).astype(np.float64)
    assert np.abs(r0 * d - 1).max() < 1 / 8


def test_rounding_model_mish():
    x = _sweep()
    ok, st = _judge(_bf16(device_mish(x)), x)
    print(f"device Mish, bf16 output: worst/bound {st['ratio']:.3f}")
    assert ok, st
    # the fp32 result itself, against the formula's own term (MISH_C * U relative) plus the x * log2(e) rounding
    y, r = device_mish(x).astype(np.float64), _exact_mish(x)
    assert np.all(np.abs(y - r) <= MISH_C * U * np.abs(r) + 1.09 * U * np.abs(x.astype(np.float64)) + 1e-45)
    # what the bound must catch
    for name, wrong in (("bf16 Mish", lambda v: _bf16(v * _bf16(np.tanh(_bf16(np.logaddexp(_bf16(v), 0)))))),
                        ("x tanh(x)", lambda v: v * np.tanh(v)),
                        ("softplus without tanh", lambda v: v * np.logaddexp(v, 0)),
                        ("LeakyReLU", lambda v: np.where(v > 0, v, np.float32(0.1) * v))):
        ok, st = _judge(_bf16(wrong(x.astype(np.float32)).astype(np.float32)), x)
        assert not ok, name


# ---------------------------------------------------------------------------------------------------- bf16 floor
def test_v4_bf16_operand_floor():
    size, frames = 256, 2
    data = modelgen.build_onnx("v4", 80, size, seed=1)
    e32, e16 = MishExecutor(data), MishExecutor(data, dtype="bf16")
    herr, ious, dconfs, cands = [], [], [], []
    for s in range(frames):
        x = ref_post.normalise(modelgen.synthetic_frame(200 + s, size))
        h32, h16 = e32.run(x), e16.run(x)
        herr.append(max(float(np.abs(a - b).max() / np.abs(a).max()) for a, b in zip(h32, h16)))
        i, d = ref_post.detection_spread(h32, h16, 80, (size, size), 0.1)
        ious.extend(i)
        dconfs.extend(d)
        cands.append(len(ref_post.detect_from_heads(h32, 0, 80, (size, size), 0.1)[0]))
    ious, dconfs = np.array(ious), np.array(dconfs)
    print(f"v4 {size} bf16-operand vs fp32 oracle: head err {max(herr):.4f}, {len(ious)} matched boxes, IoU min {ious.min():.4f} "
          f"median {np.median(ious):.4f}, |dconf| max {dconfs.max():.4f}; detections per frame {cands}")
    assert max(herr) <= 2e-2
    assert min(cands) >= 10
    assert ious.min() >= 0.95 and np.median(ious) >= 0.98 and dconfs.max() <= 1e-2
