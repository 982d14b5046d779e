"""YOLOv4 on the GPU (-m gpu): Mish in every convolution kernel form and the SPP max-pools as one launch, against the
teacher-forced float64 oracle per layer (tests/mish_oracle.py through check_layers_exact), the fp32 oracle at the heads and
in the detections, and through the drop-in detector and the serving lanes."""
import io

import numpy as np
import pytest
from PIL import Image

from fastdet_b200 import _native, modelgen
from fastdet_b200 import detector as fdet
from oracle import ref_graph, ref_post
from tests import mish_compare, test_gpu_layers_exact
from tests.compare import same_detections
from tests.mish_oracle import MishExecutor
from tests.test_gpu_layers_exact import _front_layers, _pooled, _records, _run_path, check_layers_exact
from tests.test_gpu_parity import DetectionTally, frames_for
from tests.test_gpu_tiny4 import _reference_jpegs, _synthetic_jpegs

pytestmark = pytest.mark.gpu
SEED = 1
THR = 0.1

# id: (net (w, h), batch, path, checked frames (None: all), strip option (None: default))
ROWS = {
    "416-n1": ((416, 416), 1, "forward", None, None),
    "416-n5-bucket8": ((416, 416), 5, "forward", None, None),
    "416-n64": ((416, 416), 64, "forward", [0, 37, 63], None),
    "416-strip-n2": ((416, 416), 2, "forward", None, 2),
    "416x256-n3": ((416, 256), 3, "forward", [0, 2], None),
    "256x416-n2": ((256, 416), 2, "forward", [1], None),
    "416-n20-detect": ((416, 416), 20, "detect", [0, 9, 19], None),
}
# every form a Mish layer must have run in over the rows ("halo s2": the stride-2 halo kernel; "split_k": a split launch)
MISH_FORMS = {"conv0", "halo", "halo s2", "tc_single", "tc_swapped", "tc_pair", "tc_pair_strip", "split_k"}
_data = {}
_models = {}


@pytest.fixture(scope="module", autouse=True)
def _release_models():
    yield
    for m in _models.values():
        m.close()
    _models.clear()


def _v4(opts=None):
    key = repr(opts)
    if key not in _data:
        _data[key] = modelgen.build_onnx("v4", 80, 416, SEED, opts)
    return _data[key]


def _model(wh, strip=None):
    key = (wh, strip)
    if key not in _models:
        if strip is None:
            _models[key] = _native.Model(_v4(), 80, wh, device=0)
        else:
            with _native.option("strip", strip):
                _models[key] = _native.Model(_v4(), 80, wh, device=0)
    return _models[key]


def _exec_info(m, n, strip):
    if strip is None:
        return m.exec_info(n)
    with _native.option("strip", strip):
        return m.exec_info(n)


def _mish_forms(L, info):
    out = set()
    for l, e in zip(L, info):
        if l["act"] != 2:
            continue
        name = e["kernel_name"]
        out.add(name + (" s2" if name == "halo" and l["stride"] == 2 else ""))
        if e["split_k"] > 1:
            out.add("split_k")
    return out


@pytest.mark.parametrize("row", list(ROWS))
def test_v4_layers_exact(row, monkeypatch):
    wh, n, path, picks, strip = ROWS[row]
    # check_layers_exact builds the oracle and applies the bound through these names
    monkeypatch.setattr(ref_graph, "GraphExecutor", MishExecutor)
    monkeypatch.setattr(test_gpu_layers_exact, "check_layer", mish_compare.check_layer)
    picks = list(range(n)) if picks is None else picks
    frames = frames_for(n, wh, first_seed=700)
    data, m = _v4(), _model(wh, strip)
    records = _run_path(m, frames, path) if strip is None else None
    if strip is not None:
        with _native.option("strip", strip):
            _run_path(m, frames, path)
    L = m.layers()
    front = _front_layers(L, _pooled(data), wh[1]) if path == "detect" else frozenset()
    check_layers_exact(data, m, frames, picks, "v4 " + row, front)
    info = _exec_info(m, n, strip)
    # the SPP block: one launch at the last pool, which check_layers_exact held to the oracle exactly (bound 0)
    assert [e["kernel_name"] for l, e in zip(L, info) if l["kind"] == 2] == ["fused_next", "fused_next", "spp"]
    assert [e["launches"] for l, e in zip(L, info) if l["kind"] == 2] == [0, 0, 1]
    assert info[0]["kernel_name"] == "conv0" and L[0]["act"] == 2
    if strip is not None:
        assert "tc_pair_strip" in _mish_forms(L, info)
    if records is not None:  # the staged path on the same frames returns the very same records
        m.preprocess(frames, n, wh)
        m.forward(n)
        staged = _records(m, n)
        for f in range(n):
            assert np.array_equal(records[f], staged[f]), f


def test_v4_rows_run_mish_in_every_form():
    seen = set()
    for wh, n, path, picks, strip in ROWS.values():
        m = _model(wh, strip)
        seen |= _mish_forms(m.layers(), _exec_info(m, n, strip))
    print("Mish layers ran as:", sorted(seen))
    assert MISH_FORMS <= seen, sorted(MISH_FORMS - seen)


def test_v4_heads_against_fp32_oracle():
    frames = frames_for(2, 416)
    m = _model((416, 416))
    m.preprocess(frames, 2, (416, 416))
    m.forward(2)
    x = np.concatenate([ref_post.normalise(f) for f in frames])
    for g, r in zip(m.heads(2), MishExecutor(_v4()).run(x)):
        assert g.shape == r.shape
        err = np.abs(g - r).max()
        assert err <= 2e-2 * np.abs(r).max(), (err, np.abs(r).max())
    # the Softplus -> Tanh -> Mul export computes exactly what the Mish-node export does
    m2 = _native.Model(_v4(modelgen.ExportOptions(mish_op="softplus")), 80, (416, 416), device=0)
    m2.preprocess(frames, 2, (416, 416))
    m2.forward(2)
    for a, b in zip(m.heads(2), m2.heads(2)):
        assert np.array_equal(a, b)
    m2.close()


def test_v4_detections_match_oracle():
    det = fdet.ONNXDetector(_v4(), num_classes=80)
    exe, exe16 = MishExecutor(_v4()), MishExecutor(_v4(), dtype="bf16")
    t32, t16 = DetectionTally(80, THR), DetectionTally(80, THR)
    for s in range(3):
        frame = modelgen.synthetic_frame(200 + s, 416)
        buf = io.BytesIO()
        Image.fromarray(frame, "RGB").save(buf, format="PNG")
        got = det.perform(buf.getvalue(), threshold=THR)
        dets, counts = det.model.detect(frame[None], THR)
        assert counts[0] == len(got)
        x = ref_post.normalise(frame)
        h32, h16 = exe.run(x), exe16.run(x)
        t32.add(h32, dets[0, :counts[0]])
        t32.add_floor(h32, h16)
        t16.add(h16, dets[0, :counts[0]])
    t32.check("v4 vs fp32 oracle")
    t16.check("v4 vs bf16-operand oracle")


def test_v4_batch_sizes_agree():
    m = _model((416, 416))
    frames = frames_for(64, 416)
    d64, c64 = m.detect(frames, THR)
    for f in (0, 31, 63):
        d1, c1 = m.detect(frames[f:f + 1], THR)
        tup = lambda d, c: [(int(r["klass"]), float(r["conf"]), float(r["x"]), float(r["y"]), float(r["w"]), float(r["h"])) for r in d[:c]]
        assert c1[0] > 0
        assert same_detections(tup(d1[0], c1[0]), tup(d64[f], c64[f]), THR), f


def test_v4_dropin_on_reference_images(tmp_path):
    path = tmp_path / "yolov4.onnx"
    path.write_bytes(_v4())
    det = fdet.ONNXDetector(str(path), num_classes=80)
    exe, exe16 = MishExecutor(_v4()), MishExecutor(_v4(), dtype="bf16")
    tally = DetectionTally(80, THR)
    for jpg in _reference_jpegs():
        got = det.perform(jpg, threshold=THR)
        pixels = np.asarray(Image.open(io.BytesIO(jpg)).convert("RGB"))
        dets, counts = det.model.detect(pixels[None], THR)
        assert [(int(d["klass"]), float(d["conf"])) for d in dets[0, :counts[0]]] == [(g[0], g[1]) for g in got]
        x = ref_post.normalise(pixels)
        h32, h16 = exe.run(x), exe16.run(x)
        tally.add(h32, dets[0, :counts[0]])
        tally.add_floor(h32, h16)
    tally.check("v4 drop-in on the reference images", min_solid=1)


def test_v4_server_jpeg_equals_detect_jpeg():
    from fastdet_b200.server import DetectServer
    from tests.test_server_jpeg import run_concurrently
    data = _v4()
    payloads = _reference_jpegs() + [buf.getvalue() for buf in _synthetic_jpegs(5)]
    srv = DetectServer({"v4": (data, 80)}, devices=[0], max_batch=8, max_det=256, max_delay_ms=200.0)
    res = run_concurrently(srv.perform_jpeg_records, [("v4", 0, p, THR) for p in payloads])
    assert srv.lane_stats()[(0, "v4")] == (1, 8)
    srv.close()
    m = _native.Model(data, 80, (416, 416), device=0)
    dets, counts = m.detect_jpeg(payloads, THR, max_det=256)
    total = 0
    for i in range(len(payloads)):
        assert not isinstance(res[i], BaseException), res[i]
        assert res[i].tobytes() == dets[i, :counts[i]].tobytes(), i
        total += int(counts[i])
    assert total > 0
    m.close()
