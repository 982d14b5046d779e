"""CPU tests of the two SURVEY §8f "next" rows built so far: the wire-format packer (native, host-only) against the
reference's struct.pack lines, and the micro-batching service's host logic with a stand-in detector."""
import io
import struct
import threading

import numpy as np
import pytest

from fastdet_b200 import _native, service
from oracle import ref_wire


def _dets(rows):
    a = np.zeros(len(rows), _native.DET_DTYPE)
    for i, (k, c, x, y, w, h) in enumerate(rows):
        a[i] = (k, i, c, x, y, w, h)
    return a


def test_pack_matches_reference_dummy_detector_answer():
    # the one fixed answer the reference ships: DummyDetector.perform (server/detector.py:83-92) at 416x416
    results = [(16, 1.0, 208.0, 208.0, 166.4, 166.4)]
    want = ref_wire.pack_results(results, reqid=7, msec=12)
    assert want == struct.pack('>4sLLL', b'YOLO', 7, 12, 10) + struct.pack('>BBhhhh', 16, 255, 208, 208, 166, 166)
    assert _native.pack_wire(_dets(results), 7, 12) == want


def test_pack_random_detections_bit_exact():
    rng = np.random.default_rng(5)
    rows = [(int(rng.integers(1, 81)), float(rng.random()), float(rng.uniform(-500, 900)), float(rng.uniform(-500, 900)),
             float(rng.uniform(0, 3000)), float(rng.uniform(0, 3000))) for _ in range(300)]
    rows += [(1, 0.999999, -0.99, 0.99, 32767.9, -32768.9), (255, 0.0, -32768.0, 32767.0, 0.0, 0.0)]  # truncation toward zero, extremes
    assert _native.pack_wire(_dets(rows), 0xFFFFFFFF, 123456) == ref_wire.pack_results(rows, 0xFFFFFFFF, 123456)
    assert _native.pack_wire(_dets([]), 1, 2) == ref_wire.pack_results([], 1, 2)


def test_pack_out_of_range_like_struct_pack_or_saturating():
    bad = [(3, 0.5, 40000.0, 0.0, 10.0, 10.0)]
    with pytest.raises(struct.error):
        ref_wire.pack_results(bad, 0, 0)
    with pytest.raises(struct.error):
        _native.pack_wire(_dets(bad), 0, 0)
    sat = _native.pack_wire(_dets(bad + [(300, 0.5, -40000.0, 1.0, 2.0, 3.0)]), 0, 0, saturate=True)
    assert sat[16:] == struct.pack('>BBhhhh', 3, 127, 32767, 0, 10, 10) + struct.pack('>BBhhhh', 255, 127, -32768, 1, 2, 3)


class _FakeDetector:
    """perform_frames returns, per frame, a result that identifies the frame and the batch it rode in."""
    image_size = (8, 8)

    def __init__(self):
        self.batches = []

    def perform_frames(self, frames, threshold=0.1):
        self.batches.append((len(frames), threshold))
        if threshold == 0.99:
            raise RuntimeError("boom")
        return [[(1, float(threshold), float(f[0, 0, 0]), 0.0, 1.0, 1.0)] for f in frames]


def _png(value):
    from PIL import Image
    buf = io.BytesIO()
    Image.fromarray(np.full((8, 8, 3), value, np.uint8), "RGB").save(buf, format="PNG")
    return buf.getvalue()


def test_batching_service_groups_concurrent_callers():
    det = _FakeDetector()
    svc = service.BatchingService(det, max_batch=16, max_delay=0.2)
    out = {}

    def call(i):
        out[i] = svc.perform(_png(i), threshold=0.1 if i % 4 else 0.25)

    threads = [threading.Thread(target=call, args=(i,)) for i in range(12)]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    for i in range(12):  # every caller gets its own frame's answer with its own threshold
        assert out[i] == [(1, 0.1 if i % 4 else 0.25, float(i), 0.0, 1.0, 1.0)]
    assert svc.frames_run == 12 and svc.batches_run < 12  # requests were grouped
    assert all(thr in (0.1, 0.25) for _, thr in det.batches)
    # errors: bad size is raised in the caller like the reference's ValueError; a failing batch reaches its callers
    from PIL import Image
    buf = io.BytesIO()
    Image.fromarray(np.zeros((4, 8, 3), np.uint8), "RGB").save(buf, format="PNG")
    with pytest.raises(ValueError, match="invalid image size"):
        svc.perform(buf.getvalue())
    with pytest.raises(RuntimeError, match="boom"):
        svc.perform(_png(1), threshold=0.99)
    assert svc.perform(_png(9), threshold=0.1) == [(1, 0.1, 9.0, 0.0, 1.0, 1.0)]  # the worker survived
    svc.close()
    with pytest.raises(RuntimeError):
        svc.perform(_png(1))


class _RefusingDetector:
    """Pipelined stand-in whose submit refuses batches that contain a 'bad' payload, naming it in a per-frame status
    like fastdet_b200._native.JpegRefused does; on its own the bad payload raises OSError (what PIL raises)."""
    image_size = (8, 8)

    class Refused(RuntimeError):
        def __init__(self, status):
            super().__init__("refused")
            self.status = status

    def __init__(self):
        self.slots, self.submitted, self.single = {}, [], []

    def jpeg_probe(self, data):
        return 'device'

    def _answer(self, d):
        return [(1, 0.5, float(len(d)), 0.0, 1.0, 1.0)]

    def perform_jpegs(self, datas, threshold=0.1):
        self.single.append(len(datas))
        for d in datas:
            if d.startswith(b"bad"):
                raise OSError("cannot identify image file")
        return [self._answer(d) for d in datas]

    def perform_frames(self, frames, threshold=0.1):
        raise AssertionError("not used")

    def submit_jpegs(self, slot, datas, threshold=0.1, strict=False):
        assert strict and slot not in self.slots
        status = [2 if d.startswith(b"bad") else 0 for d in datas]
        if any(status):
            raise self.Refused(status)
        self.submitted.append(len(datas))
        self.slots[slot] = [self._answer(d) for d in datas]

    def submit_frames(self, slot, frames, threshold=0.1):
        raise AssertionError("not used")

    def collect(self, slot):
        return self.slots.pop(slot)


def test_one_bad_payload_fails_only_its_own_caller():
    """ADVICE r1: a damaged payload queued with 15 good ones must not fail (or serialise) the others: the refusal's
    per-frame status singles it out, its caller alone gets the reference's exception, the rest runs as ONE batch."""
    det = _RefusingDetector()
    svc = service.BatchingService(det, max_batch=16, max_delay=0.3)
    out, errs = {}, {}

    def call(i):
        data = (b"bad" if i == 5 else b"ok") + bytes(i)
        try:
            out[i] = svc.perform(data)
        except Exception as e:  # noqa: BLE001
            errs[i] = e

    threads = [threading.Thread(target=call, args=(i,)) for i in range(16)]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    svc.close()
    assert list(errs) == [5] and isinstance(errs[5], OSError)
    assert sorted(out) == [i for i in range(16) if i != 5]
    for i, res in out.items():
        assert res == [(1, 0.5, float(2 + i), 0.0, 1.0, 1.0)]
    assert svc.isolated == 1 and det.single == [1]           # only the offender went through the one-by-one route
    assert sum(det.submitted) == 15 and len(det.submitted) <= 3  # the good ones were re-batched, not serialised


def test_letterbox_geometry_and_unmapping():
    """Extension (SURVEY 8f rank 4): frames of another size are letterboxed; fd_unmap_letterbox takes the boxes back to
    the caller's pixels.  Restated here: scale = min(net/src) with the long side filling the network, centred."""
    import numpy as np
    from fastdet_b200 import _native
    for (NW, NH) in [(416, 416), (416, 256), (256, 416)]:  # on the non-square nets either side can limit a source
        for (sw, sh) in [(640, 480), (480, 640), (416, 416), (1920, 1080), (97, 1031), (1, 1), (832, 416), (416, 256), (13, 500)]:
            nw, nh, ox, oy = _native.letterbox_geometry((sw, sh), (NW, NH))
            if sw * NH >= sh * NW:
                want = (NW, max(1, (sh * NW + sw // 2) // sw))
            else:
                want = (max(1, (sw * NH + sh // 2) // sh), NH)
            assert (nw, nh) == want and (ox, oy) == ((NW - nw) // 2, (NH - nh) // 2), ((sw, sh), (NW, NH))
            d = np.zeros(3, _native.DET_DTYPE)
            d['x'], d['y'], d['w'], d['h'] = [ox, ox + nw / 2, 10.0], [oy, oy + nh / 2, 20.0], [nw, 5.0, 1.0], [nh, 7.0, 2.0]
            d['klass'], d['conf'] = [1, 2, 3], [0.9, 0.8, 0.7]
            u = _native.unmap_letterbox(d, (sw, sh), (NW, NH))
            assert np.allclose(u['x'], (d['x'] - ox) * sw / nw, rtol=0, atol=1e-9) and np.allclose(u['w'], d['w'] * sw / nw, rtol=0, atol=1e-9)
            assert np.allclose(u['y'], (d['y'] - oy) * sh / nh, rtol=0, atol=1e-9) and np.allclose(u['h'], d['h'] * sh / nh, rtol=0, atol=1e-9)
            assert u['x'][0] == 0 and u['y'][0] == 0 and abs(u['w'][0] - sw) < 1e-9 and abs(u['h'][0] - sh) < 1e-9  # the whole picture
            assert np.array_equal(u['klass'], d['klass']) and np.array_equal(u['conf'], d['conf'])
