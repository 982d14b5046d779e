"""JPEG requests on the multi-GPU dispatcher (fd_server_perform_jpeg) and per-frame thresholds in the post kernels.

CPU: the stand-in backend runs the real host half (parse + entropy decode into the lane's JPEG batch); its records say which
frame (first quantised luma DC coefficient), which batch size and which threshold each caller was served with.
GPU (-m gpu): fd_postprocess_thresholds against the oracle and against fd_postprocess at each frame's threshold, and the
lanes' JPEG batches against fd_detect_jpeg and the reference detector's perform()."""
import io
import os
import threading
import time

import numpy as np
import pytest
from PIL import Image

from fastdet_b200 import _native, modelgen
from fastdet_b200.server import DetectServer

HERE = os.path.dirname(os.path.abspath(__file__))
FIELDS = ["klass", "conf", "x", "y", "w", "h"]


def encode(a, fmt="JPEG", **kw):
    buf = io.BytesIO()
    Image.fromarray(a).save(buf, fmt, **kw)
    return buf.getvalue()


def picture(size, seed):
    rng = np.random.default_rng(seed)
    a = np.full((size, size, 3), 30 + 25 * seed, np.float64) + rng.normal(0, 30, (size, size, 3))
    return np.clip(a, 0, 255).astype(np.uint8)


def dc_tag(data):
    """What the stand-in backend reports as klass: the frame's first quantised luma DC coefficient."""
    _, planes = _native.jpeg_coefficients(data)
    return int(planes[0][0, 0, 0, 0])


def run_concurrently(fn, args, delays=None):
    out = {}

    def call(i, a):
        if delays and delays[i]:
            time.sleep(delays[i])
        try:
            out[i] = fn(*a)
        except Exception as e:  # noqa: BLE001
            out[i] = e

    threads = [threading.Thread(target=call, args=(i, a)) for i, a in enumerate(args)]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    return [out[i] for i in range(len(args))]


# ------------------------------------------------------------------------------------------ stand-in backend (CPU)
def test_thresholds_share_a_jpeg_batch():
    srv = DetectServer.fake(n_models=1, n_devices=1, image_size=(32, 32), max_batch=8, max_delay_ms=100.0, latency_us=1000)
    datas = [encode(picture(32, i), quality=90) for i in range(6)]
    tags = [dc_tag(d) for d in datas]
    assert len(set(tags)) == 6
    thr = [0.1 if i % 2 else 0.3 for i in range(6)]
    res = run_concurrently(srv.perform_jpeg_records, [(0, 0, datas[i], thr[i]) for i in range(6)])
    for i, r in enumerate(res):
        assert not isinstance(r, BaseException), r
        assert len(r) == 1 and r[0]["klass"] == tags[i] and r[0]["w"] == thr[i]  # its own frame, its own threshold
        assert r[0]["box"] == 6  # all six rode in one batch
    assert srv.lane_stats()[(0, "m0")] == (1, 6)
    srv.close()


def test_refused_payloads_never_enter_a_batch_and_damage_stays_with_its_caller():
    srv = DetectServer.fake(n_models=1, n_devices=1, image_size=(32, 32), max_batch=8, max_delay_ms=100.0, latency_us=1000)
    a = picture(32, 1)
    refused = {"png": (encode(a, "PNG"), _native.FD_JPEG_NOT_JPEG),
               "progressive": (encode(a, quality=80, progressive=True), _native.FD_JPEG_UNSUPPORTED),
               "grey": (encode(a[..., 0], quality=80), _native.FD_JPEG_UNSUPPORTED)}
    for name, (data, status) in refused.items():
        with pytest.raises(_native.JpegRefused) as e:
            srv.perform_jpeg_records(0, 0, data, 0.1)
        assert e.value.status.tolist() == [status], name
    assert srv.lane_stats()[(0, "m0")] == (0, 0)
    big = encode(picture(208, 2), quality=80)
    with pytest.raises(ValueError, match="^invalid image size$"):
        srv.detector(0, 0).perform(big, 0.1)
    with pytest.raises(ValueError, match="^invalid image size$"):
        srv.perform_jpeg_records(0, 0, big, 0.1)
    assert srv.lane_stats()[(0, "m0")] == (0, 0)

    good = [encode(picture(32, 3 + i), quality=95) for i in range(4)]
    broken = good[0][:len(good[0]) * 2 // 3]  # the header parses, the entropy data ends early
    assert _native.jpeg_probe(broken).status == _native.FD_JPEG_OK
    datas = [good[0], good[1], broken, good[2], good[3]]
    res = run_concurrently(srv.perform_jpeg_records, [(0, 0, d, 0.2) for d in datas])
    for i, (d, r) in enumerate(zip(datas, res)):
        if d is broken:
            assert isinstance(r, _native.JpegRefused) and r.status.tolist() == [_native.FD_JPEG_CORRUPT]
        else:
            assert not isinstance(r, BaseException), r
            assert r[0]["klass"] == dc_tag(d) and r[0]["box"] == 5  # one batch; the damaged frame rode along
    assert srv.lane_stats()[(0, "m0")] == (1, 5)
    srv.close()


def test_rgb_and_jpeg_callers_on_one_lane():
    srv = DetectServer.fake(n_models=1, n_devices=1, image_size=(32, 32), max_batch=8, max_delay_ms=20.0, latency_us=500)
    datas = [encode(picture(32, 10 + i), quality=90) for i in range(4)]

    def call(i):
        if i % 2:
            f = np.zeros((32, 32, 3), np.uint8)
            f[0, 0, 0] = 200 + i
            return "rgb", srv.perform_records(0, 0, f, 0.1)
        return "jpeg", srv.perform_jpeg_records(0, 0, datas[i // 2], 0.1 + i / 100)

    res = run_concurrently(call, [(i,) for i in range(8)])
    for i, r in enumerate(res):
        assert not isinstance(r, BaseException), r
        kind, rec = r
        if kind == "rgb":
            assert rec[0]["klass"] == 200 + i
        else:
            assert rec[0]["klass"] == dc_tag(datas[i // 2]) and rec[0]["w"] == 0.1 + i / 100
    b, f = srv.lane_stats()[(0, "m0")]
    assert f == 8 and b >= 2  # an RGB and a JPEG frame never share a batch
    srv.close()


# ------------------------------------------------------------------------------------------ B200
def _fixture_heads(path):
    from tests.test_gpu_parity import _golden_heads
    z = np.load(path)
    return z, _golden_heads(z)


def _post_batch(m, heads_list, thrs, nc, size):
    """Stage heads_list (one frame each) as one batch; frame f at thrs[f].  Each frame must equal the oracle at its threshold
    and fd_postprocess at that threshold bit for bit."""
    from oracle import ref_post
    heads = [np.concatenate([h[k] for h in heads_list]) for k in range(len(heads_list[0]))]
    n = m.set_heads(heads)
    md = m.info.boxes_per_frame
    m.postprocess_thresholds(thrs, max_det=md)
    dets, counts, total = m.fetch(n)
    for f in range(n):
        want, want_idx, _ = ref_post.detect_from_heads(heads, f, nc, (size, size), thrs[f])
        assert counts[f] == total[f] == len(want), (f, thrs[f])
        d = dets[f, :counts[f]]
        assert [int(k) for k in d["klass"]] == [r[0] for r in want]
        assert [int(b) for b in d["box"]] == want_idx
        if len(want):
            got = np.stack([d["conf"], d["x"], d["y"], d["w"], d["h"]], axis=1)
            np.testing.assert_allclose(got, np.array([r[1:] for r in want], np.float64), rtol=1e-12, atol=1e-12)
    for t in sorted(set(thrs)):
        m.postprocess(n, t, max_det=md)
        d2, c2, _ = m.fetch(n)
        for f in range(n):
            if thrs[f] == t:
                assert c2[f] == counts[f] and d2[f, :c2[f]].tobytes() == dets[f, :counts[f]].tobytes(), (f, t)
    return counts


@pytest.mark.gpu
@pytest.mark.parametrize("nms_general", [0, 1])
def test_per_frame_thresholds_on_the_golden_heads(nms_general):
    groups = [["post_tiny80.npz", "post_empty.npz"], ["post_dense.npz"], ["post_full80_small.npz"], ["post_rsu9.npz"]]
    with _native.option("nms_general", nms_general):
        for names in groups:
            fixtures = [_fixture_heads(os.path.join(HERE, "golden", n)) for n in names]
            z0, h0 = fixtures[0]
            nc, size = int(z0["num_classes"]), h0[0].shape[2] * 32
            m = _native.Model(modelgen.build_onnx("tiny" if len(h0) == 2 else "full", nc, size, seed=11), nc, (size, size), device=0)
            heads_list, thrs = [], []
            for z, h in fixtures:
                at_score = [float(z["results"][len(z["results"]) // 2, 1])] if len(z["results"]) else []
                exhaustive = [0.0] if h[0].shape[2] <= 16 else []  # every box a candidate: the oracle's Python Soft-NMS is O(boxes^2)
                for t in exhaustive + [1.0, float(z["threshold"]), 0.2] + at_score:
                    heads_list.append(h)
                    thrs.append(t)
            counts = _post_batch(m, heads_list, thrs, nc, size)
            assert counts.sum() > 0, names
            m.close()


@pytest.mark.gpu
@pytest.mark.parametrize("n", [8, 64])
def test_per_frame_thresholds_after_a_forward_pass(n):
    data = modelgen.build_onnx("full", 80, 416, 2)
    m = _native.Model(data, 80, (416, 416), device=0)
    frames = np.stack([modelgen.synthetic_frame(700 + i, 416) for i in range(n)])
    m.detect(frames, 0.1, max_det=256)  # forward pass on the batch; heads stay in place
    thrs = [(0.05, 0.1, 0.3, 0.5, 0.1, 0.05, 0.7, 0.3)[i % 8] for i in range(n)]
    m.postprocess_thresholds(thrs, max_det=256)
    dets, counts, _ = m.fetch(n)
    assert counts.sum() > 0
    for t in sorted(set(thrs)):
        m.postprocess(n, t, max_det=256)
        d2, c2, _ = m.fetch(n)
        for f in range(n):
            if thrs[f] == t:
                assert c2[f] == counts[f] and d2[f, :c2[f]].tobytes() == dets[f, :counts[f]].tobytes(), (n, f, t)
    m.close()


def _reference_payloads():
    z = np.load(os.path.join(HERE, "golden", "ref_images.npz"))
    refs = [z[n + "_jpg"].tobytes() for n in ("dog", "rsu1", "rsu2")]
    synth = [encode(modelgen.synthetic_frame(800 + i, 416), quality=q, subsampling=sub, restart_marker_blocks=rst)
             for i, (sub, q, rst) in enumerate([(0, 85, 3), (1, 80, 5), (2, 75, 2), (2, 90, 7), (0, 70, 1)])]
    return refs + synth


_full = {}


def full416():
    if "data" not in _full:
        _full["data"] = modelgen.build_onnx("full", 80, 416, 2)
    return _full["data"]


def _records(dets, counts, f):
    return dets[f, :counts[f]]


@pytest.mark.gpu
def test_lane_jpeg_batch_equals_detect_jpeg():
    data = full416()
    payloads = _reference_payloads()
    thr = [0.3 if i % 2 == 0 else 0.1 for i in range(8)]
    srv = DetectServer({"full": (data, 80)}, devices=[0], max_batch=8, max_det=256, max_delay_ms=200.0)
    res = run_concurrently(srv.perform_jpeg_records, [("full", 0, payloads[i], thr[i]) for i in range(8)])
    assert srv.lane_stats()[(0, "full")] == (1, 8)
    srv.close()
    m = _native.Model(data, 80, (416, 416), device=0)
    want = {t: m.detect_jpeg(payloads, t, max_det=256) for t in (0.1, 0.3)}
    rev = {t: m.detect_jpeg(payloads[::-1], t, max_det=256) for t in (0.1, 0.3)}
    total = 0
    for i in range(8):
        assert not isinstance(res[i], BaseException), res[i]
        w = _records(*want[thr[i]], i)
        assert res[i].tobytes() == w.tobytes(), i
        assert _records(*rev[thr[i]], 7 - i).tobytes() == w.tobytes(), i  # a frame's position in the batch does not matter
        total += len(w)
    assert total > 0
    m.close()


@pytest.mark.gpu
def test_lane_refusals_take_the_reference_route(tmp_path):
    from fastdet_b200 import detector as fdet
    data = full416()
    path = tmp_path / "full.onnx"
    path.write_bytes(data)
    ref = fdet.ONNXDetector(str(path), num_classes=80, max_det=256)
    payloads = _reference_payloads()
    prog = encode(modelgen.synthetic_frame(830, 416), quality=80, progressive=True)
    broken = payloads[4][:len(payloads[4]) // 3]
    assert _native.jpeg_probe(broken).status == _native.FD_JPEG_OK
    callers = payloads[:4] + [broken] + payloads[5:8]  # 7 JPEG callers (one damaged) + the progressive one below
    thr = [0.3 if i % 2 == 0 else 0.1 for i in range(8)]
    srv = DetectServer({"full": (data, 80)}, devices=[0], max_batch=8, max_det=256, max_delay_ms=200.0)

    def call(i):
        if i == 7:
            return srv.detector("full", 0).perform(prog, thr[i])
        if callers[i] is broken:
            return srv.detector("full", 0).perform(broken, thr[i])
        return srv.perform_jpeg_records("full", 0, callers[i], thr[i])

    # the progressive caller comes last (its PIL decode and RGB frame would otherwise close the JPEG batch early)
    res = run_concurrently(call, [(i,) for i in range(8)], delays=[0] * 7 + [0.05])
    assert srv.lane_stats()[(0, "full")] == (2, 8)  # the JPEG batch of seven, then the progressive frame on its own
    srv.close()

    def reference(d, t):
        try:
            return ref.perform(d, t)
        except Exception as e:  # noqa: BLE001
            return e

    for i in (4, 7):
        d = prog if i == 7 else broken
        want = reference(d, thr[i])
        if isinstance(want, BaseException):
            assert type(res[i]) is type(want) and str(res[i]) == str(want), (res[i], want)
        else:
            assert res[i] == want
    assert isinstance(res[4], BaseException)  # PIL raises on the truncated stream, as in the reference
    stand_in = payloads[:4] + [payloads[0]] + payloads[5:7]  # any good payload in the damaged one's place
    m = _native.Model(data, 80, (416, 416), device=0)
    want = {t: m.detect_jpeg(stand_in, t, max_det=256) for t in (0.1, 0.3)}
    for i in (0, 1, 2, 3, 5, 6):
        assert not isinstance(res[i], BaseException), res[i]
        assert res[i].tobytes() == _records(*want[thr[i]], i).tobytes(), i
    m.close()


@pytest.mark.gpu
def test_bound_detector_equals_the_reference_detector(tmp_path):
    from fastdet_b200 import detector as fdet
    data = full416()
    path = tmp_path / "full.onnx"
    path.write_bytes(data)
    ref = fdet.ONNXDetector(str(path), num_classes=80, max_det=256)
    srv = DetectServer({"full": (data, 80)}, devices=[0], max_batch=8, max_det=256, max_delay_ms=0.0)
    payloads = _reference_payloads()[:3] + [encode(modelgen.synthetic_frame(840, 416), "PNG"),
                                            encode(modelgen.synthetic_frame(841, 320), quality=80)]
    for s, d in enumerate(payloads):
        for thr in (0.1, 0.3):
            try:
                want = ref.perform(d, thr)
            except Exception as e:  # noqa: BLE001
                want = e
            if isinstance(want, BaseException):
                with pytest.raises(type(want)) as e:
                    srv.detector("full", s).perform(d, thr)
                assert str(e.value) == str(want)
            else:
                assert srv.detector("full", s).perform(d, thr) == want, (s, thr)
    assert isinstance(want, ValueError) and str(want) == "invalid image size"
    srv.close()
