"""CPU-side checks of the native library: it loads, exports every symbol include/fastdet_b200.h declares,
plans ONNX graphs (host logic only) and refuses — loudly — to compute without a CUDA device."""
import ctypes
import os
import re

import numpy as np
import pytest
import torch

from fastdet_b200 import _native, modelgen
from fastdet_b200 import detector as fdet
from tests import torch_export

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HAS_GPU = torch.cuda.is_available()


def test_library_exports_every_declared_symbol():
    header = open(os.path.join(ROOT, "include", "fastdet_b200.h")).read()
    declared = set(re.findall(r"\b(fd_[a-z0-9_]+)\s*\(", header))
    assert len(declared) >= 18
    lib = _native.lib()
    for name in sorted(declared):
        assert hasattr(lib, name), f"{name} declared in the header but not exported"
    assert declared == set(_native._PROTOS), "ctypes prototypes and header disagree"
    assert lib.fd_abi_version() == 4
    assert ctypes.sizeof(_native.FdDet) == 48


@pytest.mark.parametrize("arch,nc,convs,layers", [("tiny", 80, 13, 16), ("full", 80, 75, 75), ("rsu", 9, 75, 75)])
def test_planner_on_generated_models(arch, nc, convs, layers):
    size = 416 if arch == "tiny" else 160
    data = modelgen.build_onnx(arch, nc, size, seed=3)
    m = _native.Model(data, nc, (size, size), device=-1)
    info = m.info
    # every Add/Resize/Concat fused away; tiny-416: the three max-pools behind conv1..conv3 (16x8-patch kernels) are fused
    # into those convolutions' epilogues, the pools at 52 / 26 / 13 remain launches
    assert info.n_conv == convs and info.n_layers == layers
    assert info.n_heads == (2 if arch == "tiny" else 3)
    g = size // 32
    assert m.head_shapes == [(3 * (5 + nc), g * (1 << i), g * (1 << i)) for i in range(info.n_heads)]
    assert info.boxes_per_frame == sum(3 * h * w for _, h, w in m.head_shapes)
    assert abs(info.conv_flops_per_frame * 1e-9 - modelgen.conv_gflops(arch, nc, size)) < 1e-6
    L = m.layers()
    assert L[0]["kind"] == 0 and L[0]["cin"] == 3
    if arch != "tiny":
        assert sum(l["has_residual"] for l in L) == 23 and sum(l["upsample2x"] for l in L) == 2
    anchors = np.array(info.anchors).reshape(4, 3, 2)
    want = fdet.ONNXDetector.ANCHORS[info.n_heads]
    assert np.array_equal(anchors[:info.n_heads], np.array(want, np.float32))
    m.close()
    if arch == "tiny":
        with _native.option("fuse_pool", 0):
            m = _native.Model(data, nc, (size, size), device=-1)
            assert m.info.n_layers == 19 and sum(l["kind"] == 2 for l in m.layers()) == 6
            m.close()


def test_flop_table_matches_survey():
    assert round(modelgen.conv_gflops("tiny", 80, 416), 3) == 5.565
    assert round(modelgen.conv_gflops("full", 80, 416), 3) == 65.864
    assert round(modelgen.conv_gflops("rsu", 9, 416), 3) == 65.348
    assert round(modelgen.conv_gflops("full", 80, 608), 3) == 140.692


def test_planner_accepts_every_exporter_form():
    base = _native.Model(modelgen.build_onnx("tiny", 5, 96, seed=2), 5, (96, 96), device=-1).layers()
    alt = modelgen.ExportOptions(fold_bn=False, upsample_op="Upsample", pool_pad="pad_node", const_as="constant_node",
                                 raw_data=False, packed_attrs=False, batch=1)
    other = _native.Model(modelgen.build_onnx("tiny", 5, 96, seed=2, opts=alt), 5, (96, 96), device=-1).layers()
    keys = ("kind", "c", "h", "w", "cin", "ksize", "stride", "act", "has_residual", "upsample2x", "out_fp32")
    assert [[l[k] for k in keys] for l in base] == [[l[k] for k in keys] for l in other]
    for training_form in (False, True):  # torch's own serializer: Pad built from Shape/Gather/Slice/Transpose chains
        net = torch_export.MiniYolo(nc=4, width=16).eval()
        m = _native.Model(torch_export.export(net, 64, training_form=training_form), 4, (64, 64), device=-1)
        assert m.info.n_layers == 12 and m.head_shapes == [(27, 16, 16), (27, 32, 32)]


def test_planner_errors():
    good = modelgen.build_onnx("tiny", 3, 64, seed=1)
    with pytest.raises(_native.NativeError) as e:
        _native.Model(b"not an onnx file at all", 3, (64, 64), device=-1)
    assert e.value.code == _native.FD_ERR_MODEL
    with pytest.raises(_native.NativeError) as e:  # head channels do not match num_classes
        _native.Model(good, 80, (64, 64), device=-1)
    assert e.value.code == _native.FD_ERR_MODEL and "num_classes" in e.value.msg
    with pytest.raises(_native.NativeError) as e:  # reference feeds {'input': a}: any other input name fails
        _native.Model(good.replace(b"\x0a\x05input", b"\x0a\x05inpux"), 3, (64, 64), device=-1)
    assert "input" in e.value.msg
    with pytest.raises(_native.NativeError) as e:
        _native.Model(good, 3, (70, 64), device=-1)
    assert e.value.code == _native.FD_ERR_ARG
    with pytest.raises(_native.NativeError) as e:  # truncated file
        _native.Model(good[: len(good) // 2], 3, (64, 64), device=-1)
    assert e.value.code == _native.FD_ERR_MODEL


def test_no_cpu_fallback():
    data = modelgen.build_onnx("tiny", 3, 64, seed=1)
    m = _native.Model(data, 3, (64, 64), device=-1)
    frames = np.zeros((1, 64, 64, 3), np.uint8)
    for call in (lambda: m.forward(1), lambda: m.detect(frames, 0.1), lambda: m.normalise(frames),
                 lambda: m.heads(1), lambda: m.preprocess(frames, 1, (64, 64)), lambda: m.detect_jpeg([b"\xff\xd8"], 0.1),
                 lambda: m.decode_jpeg([b"\xff\xd8"]), lambda: m.submit_jpeg(0, [b"\xff\xd8"], 0.1),
                 lambda: m.submit(0, frames, 0.1)):
        with pytest.raises(_native.NativeError) as e:
            call()
        assert e.value.code == _native.FD_ERR_CUDA
    if not HAS_GPU:
        assert _native.device_count() == 0
        with pytest.raises(_native.NativeError) as e:  # the product path never falls back to a CPU implementation
            fdet.ONNXDetector(data, num_classes=3, image_size=(64, 64))
        assert e.value.code == _native.FD_ERR_CUDA and "no CPU fallback" in e.value.msg


def test_product_never_imports_the_oracle():
    pkg = os.path.join(ROOT, "fastdet_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cc", ".h", ".cuh")):
                text = open(os.path.join(dirpath, f), errors="replace").read()
                assert not re.search(r"^\s*(from|import)\s+oracle\b", text, re.M), f"{f} imports the oracle"
                assert "oracle/" not in text or f in ("build.py",), f"{f} references oracle/"


def test_dummy_detector_golden(golden_dir):
    z = np.load(os.path.join(golden_dir, "kat.npz"))
    got = fdet.DummyDetector().perform(b"anything")
    assert np.array_equal(np.array(got, np.float64), z["dummy"])  # (16, 1.0, 208.0, 208.0, 166.4, 166.4)
    assert repr(fdet.DummyDetector()) == "<DummyDetector>"


def test_dbgout_dump(tmp_path):
    p = tmp_path / "dump.bin"
    fdet.DummyDetector(dbgout=str(p)).perform(b"\x01\x02\x03")
    assert p.read_bytes() == b"\x01\x02\x03"


def test_stem_normalisation_formula():
    """conv_stem.cu normalises without a table: fma(2^23 + k, c, -2^23 c) with c = float32(1 / 255), rounded to bf16.  For every
    byte that equals bf16(float32(k / 255.0)) — the reference's float64 division rounded to float32
    (/root/reference/server/detector.py:134), rounded once more for the tensor core — which is what the table in
    conv0_ws_kernel holds.  The fma is emulated exactly: both products are exact in float64 (24-bit x 24-bit)."""
    k = np.arange(256)
    table = torch.tensor((k / 255.0).astype(np.float32)).to(torch.bfloat16)
    c = np.float32(1.0) / np.float32(255.0)
    x = np.float32(8388608.0) + k.astype(np.float32)
    assert np.array_equal(x.view(np.uint32), 0x4B000000 | k.astype(np.uint32))  # the PRMT builds this bit pattern from the byte
    fma = (x.astype(np.float64) * np.float64(c) - np.float64(8388608.0) * np.float64(c)).astype(np.float32)
    assert torch.equal(torch.tensor(fma).to(torch.bfloat16).view(torch.int16), table.view(torch.int16))


def test_planned_fusions_host_logic():
    """Which layer pairs go to the fused kernels (conv_stem.cu: layers 0 + 1; conv_block.cu: a 1x1 + 3x3 + residual block) is
    decided on the host from the plan alone: YOLOv3-shaped graphs at 416 and 608 get both, YOLOv3-tiny (max-pool behind the
    first convolution, no residuals) neither, maps under 64 x 64 keep the separate kernels, and the options switch each
    fusion off."""
    full = _native.Model(modelgen.build_onnx("full", 80, 416, seed=2), 80, (416, 416), device=-1)
    L = full.layers()
    assert full.planned_fusions(64) == (True, 2) and full.planned_fusions(1) == (True, 2)
    # the fused block = the 1x1 (64 -> 32) and the 3x3 (32 -> 64) + residual of the first residual block
    assert (L[2]["ksize"], L[2]["cin"], L[2]["c"], L[3]["ksize"], L[3]["cin"], L[3]["c"], L[3]["has_residual"]) == (1, 64, 32, 3, 32, 64, 1)
    assert (L[0]["kind"], L[0]["c"], L[1]["ksize"], L[1]["stride"], L[1]["c"]) == (0, 32, 3, 2, 64)
    with _native.option("stem", 0):
        assert full.planned_fusions(64) == (False, 2)
    with _native.option("block", 0):
        assert full.planned_fusions(64) == (True, -1)
    full.close()
    for arch, nc, size, want in (("rsu", 9, 416, (True, 2)), ("full", 80, 608, (True, 2)), ("tiny", 80, 416, (False, -1)),
                                 ("full", 80, 96, (False, -1))):  # 96: conv2's map is 48 x 48
        m = _native.Model(modelgen.build_onnx(arch, nc, size, seed=2), nc, (size, size), device=-1)
        assert m.planned_fusions(8) == want, (arch, size, m.planned_fusions(8))
        m.close()


def test_option_names():
    """Every plan-time option round-trips through fd_set_option / fd_get_option; the retired A/B switches are unknown
    names, refused by both calls with FD_ERR_ARG."""
    for name in ("strip", "stem", "block", "fuse_pool", "nms_general", "jpeg_threads", "server_inflight"):
        old = _native.get_option(name)
        try:
            _native.set_option(name, old + 3)
            assert _native.get_option(name) == old + 3, name
        finally:
            _native.set_option(name, old)
        assert _native.get_option(name) == old, name
    for name in ("strip_min_w", "swap", "two_cta", "split_k", "split_k_min_kb", "split_k_max", "latency_bn", "b_resident",
                 "halo", "halo_skew", "halo_slots", "pdl", "graph", "exact_batch", "detect_overlap"):
        for call in (lambda: _native.set_option(name, 1), lambda: _native.get_option(name)):
            with pytest.raises(_native.NativeError) as e:
                call()
            assert e.value.code == _native.FD_ERR_ARG, name
