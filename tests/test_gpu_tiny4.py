"""YOLOv4-tiny on the GPU (-m gpu): the stride-2 first convolution on tensor cores and the convolutions that read channel
views (Slice / Split of a tensor that lives in a concat buffer), against the teacher-forced float64 oracle per layer, the fp32
oracle at the heads and in the detections, and through the drop-in detector and the serving lanes."""
import io
import os

import numpy as np
import pytest
from PIL import Image

from fastdet_b200 import _native, modelgen
from fastdet_b200 import detector as fdet
from oracle import onnx_min, ref_graph, ref_post
from tests.compare import same_detections
from tests.split_oracle import SplitExecutor
from tests.test_gpu_layers_exact import _front_layers, _pooled, _records, _run_path, check_layers_exact
from tests.test_gpu_parity import DetectionTally, frames_for

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))
SEED = 1
THR = 0.1

# id: (net (w, h), batch, path, checked frames (None: all))
ROWS = {
    "416-n1": ((416, 416), 1, "forward", None),
    "416-n5-bucket8": ((416, 416), 5, "forward", None),
    "416-n64": ((416, 416), 64, "forward", [0, 37, 63]),
    "416x256-n5": ((416, 256), 5, "forward", None),
    "256x416-n3": ((256, 416), 3, "forward", None),
    "96x160-n2": ((96, 160), 2, "forward", None),
    "416-n20-detect": ((416, 416), 20, "detect", [0, 9, 19]),
}
_models = {}


@pytest.fixture(scope="module", autouse=True)
def _release_models():
    yield
    for _, m in _models.values():
        m.close()
    _models.clear()


def _model(wh, split_op="Slice"):
    key = (wh, split_op)
    if key not in _models:
        data = modelgen.build_onnx("tiny4", 80, 416, SEED, modelgen.ExportOptions(split_op=split_op))
        _models[key] = (data, _native.Model(data, 80, wh, device=0))
    return _models[key]


def _view_readers(data, L):
    """Layers whose input is a channel view: {layer index: first channel of the view inside its source}."""
    g = onnx_min.load(data)
    producer = {o: n for n in g.nodes for o in n.outputs}
    consts = dict(g.initializers)
    out = {}
    for i, l in enumerate(L):
        node = next((n for n in g.nodes if n.name == l["name"]), None)
        if node is None or node.op != "Conv":
            continue
        src = producer.get(node.inputs[0])
        if src is not None and src.op == "Slice":
            out[i] = int(consts[src.inputs[1]][0])
        elif src is not None and src.op == "Split":
            k = src.outputs.index(node.inputs[0])
            out[i] = sum(int(v) for v in src.attrs["split"][:k])
    return out


class _WithoutLayer:
    """The model seen without one layer: the concat copy, which produces no graph value of its own (it moves layer 23's
    output into the second Concat's buffer) and is checked on its own, for bit equality with its source."""

    def __init__(self, m, skip):
        self.m, self.keep = m, [i for i in range(m.info.n_layers) if i != skip]

    def layers(self):
        L = self.m.layers()
        return [L[i] for i in self.keep]

    def exec_info(self, n):
        X = self.m.exec_info(n)
        return [X[i] for i in self.keep]

    def layer_output(self, i, n):
        return self.m.layer_output(self.keep[i], n)


def _copy_and_source(data, L):
    """(index of the concat copy, index of the layer whose output it copies)."""
    copy = next(i for i, l in enumerate(L) if l["kind"] == 3 and not l["upsample2x"])
    src = next(n for n in onnx_min.load(data).nodes if n.op == "Concat" and n.name == "concat34").inputs[1]
    return copy, next(i for i, l in enumerate(L) if l["out_name"] == src)


@pytest.mark.parametrize("row", list(ROWS))
def test_tiny4_layers_exact(row):
    wh, n, path, picks = ROWS[row]
    picks = list(range(n)) if picks is None else picks
    frames = frames_for(n, wh, first_seed=700)
    data, m = _model(wh)
    records = _run_path(m, frames, path)
    L = m.layers()
    front = _front_layers(L, _pooled(data), wh[1]) if path == "detect" else frozenset()
    if path == "detect":
        assert front == {0}  # the stride-2 first layer is a down-sampling layer: the quarter-batch front ends at layer 1
    copy, src = _copy_and_source(data, L)
    assert copy > src
    check_layers_exact(data, _WithoutLayer(m, copy), frames, picks, "tiny4 " + row, front)
    assert np.array_equal(m.layer_output(copy, n)[picks], m.layer_output(src, n)[picks])
    info = m.exec_info(n)
    assert L[0]["stride"] == 2 and info[0]["kernel_name"] == "conv0"
    readers = _view_readers(data, L)
    assert len(readers) == 3 and all(v > 0 for v in readers.values()), readers  # routes 3, 11, 19: the second half
    for i in readers:
        big = L[i]["h"] >= 64 and L[i]["w"] >= 64
        want = ("halo",) if big and L[i]["cin"] == 32 else ("tc_single", "tc_swapped", "tc_pair", "tc_pair_strip")
        assert info[i]["kernel_name"] in want, (i, L[i]["name"], info[i]["kernel_name"])
    if wh == (416, 416):
        assert info[min(readers)]["kernel_name"] == "halo"  # the 32-channel 104x104 convolution
    names = [e["kernel_name"] for e in info]
    assert names.count("maxpool") == 3 and names.count("copy") == 1
    if records is not None:  # the staged path on the same frames returns the very same records
        m.preprocess(frames, n, wh)
        m.forward(n)
        staged = _records(m, n)
        for f in range(n):
            assert np.array_equal(records[f], staged[f]), f


def test_tiny4_heads_slice_and_split():
    frames = frames_for(2, 416)
    x = np.concatenate([ref_post.normalise(f) for f in frames])
    heads = {}
    for op in ("Slice", "Split"):
        data, m = _model((416, 416), op)
        m.preprocess(frames, 2, (416, 416))
        m.forward(2)
        heads[op] = m.heads(2)
        for g, r in zip(heads[op], SplitExecutor(data).run(x)):
            assert g.shape == r.shape
            err = np.abs(g - r).max()
            assert err <= 2e-2 * np.abs(r).max(), (op, err, np.abs(r).max())
    for a, b in zip(heads["Slice"], heads["Split"]):
        assert np.array_equal(a, b)


def test_tiny4_detections_match_oracle():
    data, _ = _model((416, 416))
    det = fdet.ONNXDetector(data, num_classes=80)
    exe, exe16 = ref_graph.GraphExecutor(data), ref_graph.GraphExecutor(data, dtype="bf16")
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
    t32.check("tiny4 vs fp32 oracle")
    t16.check("tiny4 vs bf16-operand oracle")


def test_tiny4_batch_sizes_agree():
    data, m = _model((416, 416))
    frames = frames_for(64, 416)
    d64, c64 = m.detect(frames, THR)
    for f in (0, 31, 63):
        d1, c1 = m.detect(frames[f:f + 1], THR)
        tup = lambda d, c: [(int(r["klass"]), float(r["conf"]), float(r["x"]), float(r["y"]), float(r["w"]), float(r["h"])) for r in d[:c]]
        assert c1[0] > 0
        assert same_detections(tup(d1[0], c1[0]), tup(d64[f], c64[f]), THR), f


def _reference_jpegs():
    z = np.load(os.path.join(HERE, "golden", "ref_images.npz"))
    return [z[n + "_jpg"].tobytes() for n in ("dog", "rsu1", "rsu2")]


def test_tiny4_dropin_on_reference_images(tmp_path):
    data, _ = _model((416, 416))
    path = tmp_path / "yolov4-tiny.onnx"
    path.write_bytes(data)
    det = fdet.ONNXDetector(str(path), num_classes=80)
    exe, exe16 = ref_graph.GraphExecutor(data), ref_graph.GraphExecutor(data, dtype="bf16")
    tally = DetectionTally(80, THR)
    for jpg in _reference_jpegs():
        got = det.perform(jpg, threshold=THR)
        pixels = np.asarray(Image.open(io.BytesIO(jpg)).convert("RGB"))
        dets, counts = det.model.detect(pixels[None], THR)  # the reference's route: PIL pixels
        assert [(int(d["klass"]), float(d["conf"])) for d in dets[0, :counts[0]]] == [(g[0], g[1]) for g in got]
        x = ref_post.normalise(pixels)
        h32, h16 = exe.run(x), exe16.run(x)
        tally.add(h32, dets[0, :counts[0]])
        tally.add_floor(h32, h16)
    tally.check("tiny4 drop-in on the reference images", min_solid=1)


def test_tiny4_server_jpeg_equals_detect_jpeg():
    from fastdet_b200.server import DetectServer
    from tests.test_server_jpeg import run_concurrently
    data, _ = _model((416, 416))
    payloads = _reference_jpegs() + [buf.getvalue() for buf in _synthetic_jpegs(5)]
    srv = DetectServer({"v4t": (data, 80)}, devices=[0], max_batch=8, max_det=256, max_delay_ms=200.0)
    res = run_concurrently(srv.perform_jpeg_records, [("v4t", 0, p, THR) for p in payloads])
    assert srv.lane_stats()[(0, "v4t")] == (1, 8)  # one batch of 8: the same bucket as the fd_detect_jpeg call below
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


def _synthetic_jpegs(k):
    out = []
    for i in range(k):
        buf = io.BytesIO()
        Image.fromarray(modelgen.synthetic_frame(800 + i, 416), "RGB").save(buf, format="JPEG", quality=85)
        out.append(buf)
    return out
