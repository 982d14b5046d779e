"""GPU parity tests of the kernel forms the BENCHMARKED configurations run (-m gpu).

The library picks a kernel form per layer and per batch-size bucket (fd_layer_exec_info): small batches take the
im2col / split-K forms, the batch-64 serving configuration takes the strip form of the CTA-pair kernel for every 3x3
stride-1 layer with >= 64-channel inputs (29 of YOLOv3's 75 convolutions, about half of the step's device time); the
synchronous fd_detect call runs the first four layers quarter batch by quarter batch behind the pieces of its frame copy.
These tests put exactly those forms under the CPU oracle:
  * the strip form forced at a small batch (option strip=2), per layer, for the 416 and the 608 grids
    (strip widths W+1 = 53 / 27 / 14 and 77 / 39 / 20);
  * the default plan at batch 8 per layer (52x52 strips by the library's own choice);
  * the production batch 64 (rsu-416-9, BASELINE config 3): heads and detections of 8 of the 64 frames;
  * full-608 at a batch whose 76x76 layers take strips by default (BASELINE config 4's per-GPU shard, reduced);
  * the stand-alone kernel checker (csrc/dev/test_conv.cu: every kernel form, the production split-K shapes included,
    against a float64 CPU loop under the rounding model of tests/compare.py).
Every test first asserts, through fd_layer_exec_info, that the layers really took the form it means to check.
The per-layer checks here are RMS-relative against the fp32 oracle's own chain (drift from fp32); the element-wise check of
every layer against a float64 prediction from the layer's own GPU inputs, at every batch bucket, is
tests/test_gpu_layers_exact.py.
"""
import os
import subprocess

import numpy as np
import pytest

from fastdet_b200 import _native, modelgen
from oracle import ref_graph, ref_post
from tests.test_gpu_parity import DetectionTally, _check_heads, frames_for

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def strip_candidates(m):
    """Layers the strip form is built for: 3x3, stride 1, Cin % 64 == 0, Cout > 128, bf16 output."""
    return [i for i, L in enumerate(m.layers())
            if L["kind"] == 1 and L["ksize"] == 3 and L["stride"] == 1 and L["cin"] % 64 == 0 and L["c"] > 128 and not L["out_fp32"]]


def forms(m, n):
    return [e["kernel_name"] for e in m.exec_info(n)]


@pytest.mark.parametrize("size,batch", [(416, 2), (608, 1)])
def test_strip_form_forced_small_batch_per_layer(size, batch):
    data = modelgen.build_onnx("full", 80, size, seed=2)
    with _native.option("strip", 2):
        m = _native.Model(data, 80, (size, size), device=0)
        f = forms(m, batch)
        cands = strip_candidates(m)
        assert len(cands) == 29
        assert all(f[i] == "tc_pair_strip" for i in cands), [(i, f[i]) for i in cands if f[i] != "tc_pair_strip"]
        _check_heads(data, m, frames_for(batch, size, first_seed=140), per_layer=True)
    m.close()


def test_default_plan_batch8_per_layer():
    """Batch 8, default options: the library itself puts the 52x52 3x3 layers on strips (88 strip tiles >= 74 CTA pairs);
    every layer's output against the oracle."""
    data = modelgen.build_onnx("full", 80, 416, seed=2)
    m = _native.Model(data, 80, (416, 416), device=0)
    f = forms(m, 8)
    L = m.layers()
    strips52 = [i for i in strip_candidates(m) if L[i]["h"] == 52]
    assert len(strips52) == 11 and all(f[i] == "tc_pair_strip" for i in strips52)
    info = m.exec_info(8)
    # conv1 runs inside conv2's kernel (conv_stem.cu), conv3 inside conv4's (conv_block.cu)
    assert f[:4] == ["fused_next", "stem", "fused_next", "block"]
    assert all(e["launches"] == (0 if e["kernel_name"] == "fused_next" else 1) for e in info)  # no chunking by default
    _check_heads(data, m, frames_for(8, 416, first_seed=150), per_layer=True)
    m.close()


def test_production_batch64_against_oracle():
    """BASELINE config 3 (rsu-416-9, batch 64) — the configuration bench.py times: all 29 strip layers in strip form by
    the library's own choice; heads of 8 of the 64 frames against the fp32 oracle (2e-2 * max|ref|) and their
    detections against the fp32 and the bf16-operand oracle (see test_detections_match_oracle)."""
    nc = 9
    data = modelgen.build_onnx("rsu", nc, 416, seed=3)
    m = _native.Model(data, nc, (416, 416), device=0)
    f = forms(m, 64)
    cands = strip_candidates(m)
    assert len(cands) == 29 and all(f[i] == "tc_pair_strip" for i in cands), [(i, f[i]) for i in cands]
    frames = frames_for(64, 416, first_seed=100)  # 64 distinct frames, seeds 100..163 (SURVEY 8d config 3)
    m.preprocess(frames, 64, (416, 416))
    m.forward(64)
    heads = m.heads(64)
    m.postprocess(64, 0.1, max_det=512)
    dets, counts, total = m.fetch(64)
    assert (total == counts).all()
    exe, exe16 = ref_graph.GraphExecutor(data), ref_graph.GraphExecutor(data, dtype="bf16")
    t32, t16 = DetectionTally(nc), DetectionTally(nc)
    picks = [0, 7, 13, 21, 30, 42, 55, 63]
    for fidx in picks:
        x = ref_post.normalise(frames[fidx])
        want = exe.run(x)
        for g, r in zip(heads, want):
            err = np.abs(g[fidx] - r[0]).max()
            assert err <= 2e-2 * np.abs(r).max(), (fidx, err, np.abs(r).max())
        h16 = exe16.run(x)
        t32.add(want, dets[fidx, :counts[fidx]])
        t32.add_floor(want, h16)
        t16.add(h16, dets[fidx, :counts[fidx]])
    t32.check("rsu bs64 vs fp32 oracle")
    t16.check("rsu bs64 vs bf16-operand oracle")
    # the synchronous call (frame copy in four pieces overlapped with conv1..conv4 quarter by quarter, then the captured
    # tail graph) and the pipelined pair return the very same records as the staged path above
    d2, c2 = m.detect(frames, 0.1, max_det=512)
    assert np.array_equal(c2, counts) and all(np.array_equal(d2[f, :c2[f]], dets[f, :counts[f]]) for f in range(64))
    m.submit(0, frames, 0.1, max_det=512)
    d3, c3, _ = m.collect(0)
    assert np.array_equal(c3, counts) and all(np.array_equal(d3[f, :c3[f]], dets[f, :counts[f]]) for f in range(64))
    m.close()


def test_full_608_batch_with_strips_against_oracle():
    """full-608-80 (BASELINE config 4) at batch 4: the eleven 76x76 3x3 layers (27 % of the FLOPs) take strips of
    128 + 2*77 + 2 = 284 positions by the library's own choice; heads of every frame against the oracle."""
    data = modelgen.build_onnx("full", 80, 608, seed=2)
    m = _native.Model(data, 80, (608, 608), device=0)
    f = forms(m, 4)
    L = m.layers()
    s76 = [i for i in strip_candidates(m) if L[i]["h"] == 76]
    assert len(s76) == 11 and all(f[i] == "tc_pair_strip" for i in s76), [(i, f[i]) for i in s76]
    _check_heads(data, m, frames_for(4, 608, first_seed=1000))
    m.close()


def test_fused_maxpool_equals_the_pool_kernel():
    """YOLOv3-tiny: MaxPool(2, 2) in the epilogue of conv1 (conv0_ws_kernel) and conv2 / conv3 (halo-patch kernel) gives the
    very values the stand-alone pool kernel gives (a maximum of bf16 values is exact), layer by layer and at the heads;
    batch 5 so that edge tiles and several frames are involved."""
    data = modelgen.build_onnx("tiny", 80, 416, seed=1)
    frames = frames_for(5, 416, first_seed=230)
    m = _native.Model(data, 80, (416, 416), device=0)
    L = m.layers()
    assert len(L) == 16 and [l["h"] for l in L[:3]] == [208, 104, 52]  # conv1..conv3 write the pooled maps
    got, _ = _check_heads(data, m, frames, per_layer=True)
    pooled = {l["out_name"]: m.layer_output(i, 5) for i, l in enumerate(L[:3])}
    m.close()
    with _native.option("fuse_pool", 0):
        m2 = _native.Model(data, 80, (416, 416), device=0)
        L2 = m2.layers()
        assert len(L2) == 19
        m2.preprocess(frames, 5, (416, 416))
        m2.forward(5)
        for i, l in enumerate(L2):
            if l["out_name"] in pooled:
                assert l["kind"] == 2 and np.array_equal(m2.layer_output(i, 5), pooled[l["out_name"]]), l["out_name"]
        for a, b in zip(got, m2.heads(5)):
            assert np.array_equal(a, b)
        m2.close()


def test_nms_general_path_equals_register_path():
    """Option nms_general forces the global-memory Soft-NMS loop: same records as the one-candidate-per-thread path."""
    data = modelgen.build_onnx("tiny", 80, 416, seed=1)
    m = _native.Model(data, 80, (416, 416), device=0)
    frames = frames_for(3, 416, first_seed=210)
    a, ca = m.detect(frames, 0.1, max_det=256)
    with _native.option("nms_general", 1):
        b, cb = m.detect(frames, 0.1, max_det=256)
    assert np.array_equal(ca, cb) and ca.sum() > 0
    for i in range(3):
        assert np.array_equal(a[i, :ca[i]], b[i, :cb[i]])
    m.close()


def test_fused_stem_and_block_against_the_unfused_path():
    """conv_stem_kernel (/255 + conv1 + conv2 in one kernel) and conv_block_kernel (conv3 + conv4 + residual in one kernel) — the
    default for YOLOv3-shaped graphs — against the four kernels they replace (options stem=0, block=0: conv0_ws_kernel,
    conv_halo_kernel<32, 2>, conv_tc_kernel, conv_halo_kernel<32, 1>).  conv2's output agrees up to rare bf16 rounding flips
    (the same products added in another order before conv1's rounding); conv4's to one bf16 step (the fused block adds the
    residual in fp32 and rounds once, the halo kernel rounds the branch value first).  The tensors the fused forms never
    materialise (conv1, conv3) are still served by the parity hook, and both plans pass the oracle check, layer by layer and at
    the heads.  Batch 3 (bucket 4) of full-416 and batch 1 of full-608."""
    for size, batch in ((416, 3), (608, 1)):
        data = modelgen.build_onnx("full", 80, size, seed=2)
        frames = frames_for(batch, size, first_seed=400)
        m = _native.Model(data, 80, (size, size), device=0)
        info = m.exec_info(batch)
        assert [e["kernel_name"] for e in info[:4]] == ["fused_next", "stem", "fused_next", "block"]
        assert [e["launches"] for e in info[:4]] == [0, 1, 0, 1]
        _check_heads(data, m, frames, per_layer=True, layers=range(5))
        fused = [m.layer_output(i, batch) for i in range(4)]
        m.close()
        with _native.option("stem", 0), _native.option("block", 0):
            m2 = _native.Model(data, 80, (size, size), device=0)
            names = [e["kernel_name"] for e in m2.exec_info(batch)[:4]]
            assert names[0] == "conv0" and names[1] == "halo" and names[3] == "halo" and "fused_next" not in names
            _check_heads(data, m2, frames, per_layer=True, layers=range(5))
            plain = [m2.layer_output(i, batch) for i in range(4)]
            m2.close()
        assert np.array_equal(plain[0], fused[0])  # conv1: the hook runs the very kernel of the unfused plan
        d1 = np.abs(plain[1] - fused[1])
        assert (d1 > 0).mean() < 1e-3 and d1.max() <= 2.0 ** -6 * max(1.0, np.abs(fused[1]).max()), ((d1 > 0).mean(), d1.max())
        d2 = np.abs(plain[2] - fused[2])
        assert (d2 > 0).mean() < 1e-2, (d2 > 0).mean()  # conv3 from the hook: same kernel, inputs differ by conv2's rare flips
        d3 = np.abs(plain[3] - fused[3])
        assert d3.max() <= 2.0 ** -6 * max(1.0, np.abs(fused[3]).max()), d3.max()


def test_stem_checker():
    """csrc/dev/test_stem: the fused stem and the fused residual block against a float64 CPU loop (every border pixel, tile seams,
    random interior pixels) and against the kernels they replace, on ten shapes (ragged maps, odd heights, pad (1, 0), many
    tiles per CTA)."""
    exe = os.path.join(ROOT, "build", "test_stem")
    if not os.path.exists(exe):
        from fastdet_b200 import build
        exe = build.build_stem_harness()
    r = subprocess.run([exe, "check"], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=600)
    assert r.returncode == 0 and "check: 0 failing case(s)" in r.stdout and "block 208" in r.stdout, "\n".join(r.stdout.splitlines()[-20:])


def test_kernel_checker_all_forms():
    """csrc/dev/test_conv: every conv kernel form (single CTA, CTA pair, swapped, split-K incl. the production 13x13 / 26x26
    shapes, strips incl. the 608 widths, halo-patch) against a float64 CPU loop, each element held to the rounding model of
    tests/compare.py (half a bf16 step + 2^-23 (K + 4) S)."""
    exe = os.path.join(ROOT, "build", "test_conv")
    if not os.path.exists(exe):
        from fastdet_b200 import build
        exe = build.build_dev_harness()
    r = subprocess.run([exe, "check"], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=600)
    tail = "\n".join(r.stdout.splitlines()[-60:])
    assert r.returncode == 0 and "check: 0 failing case(s)" in r.stdout, tail
    assert "x2 strip" in r.stdout  # the strip cases really took the strip form
    # the split-K cases really split (which also runs the check that a relaunch finds its counters back at zero)
    split_cases = [l for l in r.stdout.splitlines() if l.startswith("[splitK")]
    assert len(split_cases) == 4 and all(" splitK " in l for l in split_cases), "\n".join(split_cases)
    assert all("x2 splitK" in l for l in split_cases if l.startswith("[splitK 2cta")), "\n".join(split_cases)  # the CTA pair
