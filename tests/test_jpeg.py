"""JPEG front end (SURVEY §8f rank 2; reference server/detector.py:128-133 = PIL/libjpeg decode inside perform()).

CPU part (default run): the numpy restatement in oracle/ref_jpeg.py is pinned against Pillow (committed fixture + streams
generated here), and the library's host half — marker parse + Huffman decode, through the C ABI — is checked against it
coefficient by coefficient, plus the refusal behaviour.  GPU part (-m gpu): the device half against Pillow, bit-exact,
and the end-to-end equivalence fd_detect_jpeg(bytes) == fd_detect(PIL-decoded frames).
"""
import io
import os
import threading

import numpy as np
import pytest
from PIL import Image

from fastdet_b200 import _native, modelgen
from fastdet_b200.service import BatchingService
from oracle import ref_jpeg

HERE = os.path.dirname(os.path.abspath(__file__))


def encode(a, **kw):
    buf = io.BytesIO()
    Image.fromarray(a).save(buf, 'JPEG', **kw)
    return buf.getvalue()


def picture(h, w, seed):
    rng = np.random.default_rng(seed)
    yy, xx = np.mgrid[0:h, 0:w]
    img = np.stack([127 + 100 * np.sin(xx / 9.0 + seed) * np.cos(yy / 13.0), 127 + 120 * np.sin((xx - yy) / 6.0),
                    (xx * 2 + yy * 7 + seed * 31) % 256], -1).astype(np.float64)
    img += rng.normal(0, 20, img.shape)
    return np.clip(img, 0, 255).astype(np.uint8)


def golden():
    z = np.load(os.path.join(HERE, 'golden', 'jpeg.npz'))
    return [(z[f'jpeg{i}'].tobytes(), z[f'rgb{i}'], tuple(z[f'meta{i}'])) for i in range(int(z['count']))]


# ------------------------------------------------------------------------------------------ oracle pinned to Pillow
def test_restatement_matches_committed_pillow_output():
    for data, rgb, meta in golden():
        assert np.array_equal(ref_jpeg.decode(data), rgb), meta
        assert np.array_equal(ref_jpeg.decode_reference(data), rgb), meta  # this image's Pillow still agrees


@pytest.mark.parametrize('sub', [0, 1, 2])
def test_restatement_matches_pillow_generated(sub):
    for (h, w, q, rst) in [(40, 56, 85, 0), (23, 41, 60, 2), (33, 18, 97, 0)]:
        kw = dict(restart_marker_blocks=rst) if rst else {}
        data = encode(picture(h, w, q), quality=q, subsampling=sub, **kw)
        assert np.array_equal(ref_jpeg.decode(data), ref_jpeg.decode_reference(data)), (h, w, q, rst)


def test_committed_damaged_streams():
    """Pillow's pixels for damaged streams (fixture): the restatement on the NATIVE coefficients reproduces them, so the
    overflow behaviour of libjpeg-turbo's SIMD IDCT is pinned independently of the Pillow build on the test machine."""
    z = np.load(os.path.join(HERE, 'golden', 'jpeg.npz'))
    assert int(z['damaged_count']) >= 8
    for i in range(int(z['damaged_count'])):
        d = z[f'damaged_jpeg{i}'].tobytes()
        info, planes = _native.jpeg_coefficients(d)
        assert np.array_equal(ref_jpeg.reconstruct(ref_jpeg.parse(d), planes), z[f'damaged_rgb{i}']), i


def test_idct_known_answers():
    # DC only: every sample = clamp(descale(dc * q) + 128); a full-range DC saturates through the range-limit table
    q = np.full((8, 8), 16, np.int64)
    for dc, want in [(0, 128), (1, 130), (-1, 126), (8, 144), (63, 254), (64, 255), (-64, 0), (-100, 0)]:
        c = np.zeros((8, 8), np.int16)
        c[0, 0] = dc
        assert np.all(ref_jpeg.idct_islow(c, q) == want), dc
    # upsampling edge rules (jdsample.c): ends copied, 3:1 inside with the +1 / +2 rounding pair
    row = np.array([[10, 20, 40]])
    assert ref_jpeg.h2v1_fancy(row).tolist() == [[10, 13, 17, 25, 35, 40]]
    assert ref_jpeg.h2v2_fancy(np.array([[16, 32, 64]])).tolist() == [[16, 20, 28, 40, 56, 64]] * 2
    # colour: grey stays grey, saturated chroma hits the clamps
    assert ref_jpeg.ycc_to_rgb(np.array([77]), np.array([128]), np.array([128])).tolist() == [[77, 77, 77]]
    assert ref_jpeg.ycc_to_rgb(np.array([128]), np.array([255]), np.array([0])).tolist() == [[0, 176, 255]]


# ------------------------------------------------------------------------------------------ host half of the library
def test_native_huffman_equals_oracle_on_golden():
    for data, rgb, meta in golden():
        info, planes = _native.jpeg_coefficients(data)
        hdr, coefs = ref_jpeg.entropy_decode(data)
        assert (info.width, info.height) == (hdr['width'], hdr['height'])
        assert (info.h_samp, info.v_samp) == hdr['comps'][0][1:3]
        assert info.restart_interval == hdr['restart_interval']
        for c in range(3):
            assert np.array_equal(planes[c], coefs[c]), (meta, c)
            assert np.array_equal(np.array(info.quant[c * 64:(c + 1) * 64]).reshape(8, 8), hdr['qt'][hdr['comps'][c][3]])
        # and the rest of the restatement on top of the NATIVE coefficients lands on Pillow's pixels
        assert np.array_equal(ref_jpeg.reconstruct(hdr, planes), rgb), meta


@pytest.mark.parametrize('sub,q,rst', [(0, 75, 0), (1, 75, 0), (2, 75, 0), (2, 95, 7), (2, 20, 0), (0, 100, 1)])
def test_native_huffman_full_size_frames(sub, q, rst):
    """416x416 (the reference's frame size): native coefficients -> numpy reconstruction == Pillow, bit for bit."""
    kw = dict(restart_marker_blocks=rst) if rst else {}
    data = encode(modelgen.synthetic_frame(100 + sub + q, 416), quality=q, subsampling=sub, **kw)
    info, planes = _native.jpeg_coefficients(data)
    assert info.status == _native.FD_JPEG_OK and (info.width, info.height) == (416, 416)
    hdr = ref_jpeg.parse(data)
    assert np.array_equal(ref_jpeg.reconstruct(hdr, planes), ref_jpeg.decode_reference(data))


def test_optimised_huffman_tables_and_16bit_codes():
    data = encode(picture(64, 64, 5), quality=98, subsampling=0, optimize=True)
    info, planes = _native.jpeg_coefficients(data)
    hdr, coefs = ref_jpeg.entropy_decode(data)
    assert all(np.array_equal(p, c) for p, c in zip(planes, coefs))


def test_refusals():
    a = picture(64, 64, 1)
    ok = encode(a, quality=80)
    assert _native.jpeg_probe(ok).status == _native.FD_JPEG_OK
    cases = {
        'progressive': (encode(a, quality=80, progressive=True), _native.FD_JPEG_UNSUPPORTED),
        'grey': (encode(a[..., 0], quality=80), _native.FD_JPEG_UNSUPPORTED),
        'headers only': (ok[:ok.index(b'\xff\xda')], _native.FD_JPEG_CORRUPT),
        'empty': (b'', _native.FD_JPEG_NOT_JPEG),
    }
    buf = io.BytesIO()
    Image.fromarray(a).save(buf, 'PNG')
    cases['png'] = (buf.getvalue(), _native.FD_JPEG_NOT_JPEG)
    buf = io.BytesIO()
    Image.fromarray(a).convert('CMYK').save(buf, 'JPEG', quality=80)
    cases['cmyk'] = (buf.getvalue(), _native.FD_JPEG_UNSUPPORTED)
    for name, (data, want) in cases.items():
        assert _native.jpeg_probe(data).status == want, name
        with pytest.raises(_native.JpegRefused):
            _native.jpeg_coefficients(data)
    # damage that only the entropy decoder can see: truncated scan, missing EOI, a marker in the middle of the data
    for name, data in {'truncated': ok[:len(ok) * 2 // 3], 'no EOI': ok[:-2],
                       'marker inside': ok[:len(ok) - 200] + b'\xff\xd9' + ok[len(ok) - 198:]}.items():
        assert _native.jpeg_probe(data).status == _native.FD_JPEG_OK, name
        with pytest.raises(_native.JpegRefused) as e:
            _native.jpeg_coefficients(data)
        assert e.value.status[0] == _native.FD_JPEG_CORRUPT, name
    # trailing bytes after EOI are ignored, as Pillow ignores them
    info, planes = _native.jpeg_coefficients(ok + b'\x00\x01\x02')
    assert info.status == _native.FD_JPEG_OK


def test_random_damage_never_crashes():
    rng = np.random.default_rng(7)
    ok = bytearray(encode(picture(48, 64, 2), quality=70, restart_marker_blocks=2))
    for trial in range(300):
        d = bytearray(ok)
        for _ in range(int(rng.integers(1, 6))):
            d[int(rng.integers(2, len(d)))] = int(rng.integers(0, 256))
        try:
            _native.jpeg_coefficients(bytes(d))
        except _native.JpegRefused:
            pass


def damaged_streams(seed, trials, mods=4):
    """Random byte / bit damage on valid streams; yields the ones the library still accepts."""
    rng = np.random.default_rng(seed)
    for trial in range(trials):
        sub, rst = int(rng.integers(0, 3)), int(rng.integers(0, 3))
        kw = dict(restart_marker_blocks=rst) if rst else {}
        d = bytearray(encode(picture(40, 56, trial % 7), quality=int(rng.integers(20, 98)), subsampling=sub, **kw))
        for _ in range(int(rng.integers(1, mods))):
            pos = int(rng.integers(2, len(d)))
            if rng.random() < 0.5:
                d[pos] ^= 1 << int(rng.integers(0, 8))
            else:
                d[pos] = int(rng.integers(0, 256))
        d = bytes(d)
        try:
            info, planes = _native.jpeg_coefficients(d)
        except (_native.JpegRefused, MemoryError):  # (MemoryError: damaged dimensions, the test hook's numpy buffer)
            continue
        yield d, planes


def test_accepted_damaged_streams_decode_like_pillow():
    """Whatever the library does not refuse must come out exactly as Pillow decodes it — including the places where
    libjpeg-turbo's SIMD IDCT overflows differently from the C code (16-bit lanes, saturating packs, the DC-only
    shortcut) and a DC predictor that has run away.  Before those were restated, 5 % of the accepted streams differed."""
    import warnings
    accepted = 0
    with warnings.catch_warnings():
        warnings.simplefilter('ignore')
        for d, planes in damaged_streams(21, 700):
            accepted += 1
            want = ref_jpeg.decode_reference(d)  # must not raise: what Pillow cannot open, the library must refuse
            assert np.array_equal(ref_jpeg.reconstruct(ref_jpeg.parse(d), planes), want)
    assert accepted > 150


class _FakeDetector:
    """perform_jpegs / perform_frames stand-ins that record how each payload arrived."""
    image_size = (64, 64)

    def __init__(self):
        self.jpeg_batches, self.frame_batches = [], []

    def jpeg_probe(self, data):
        info = _native.jpeg_probe(bytes(data))
        if info.status != _native.FD_JPEG_OK:
            return 'host'
        return 'device' if (info.width, info.height) == self.image_size else 'size'

    def perform_jpegs(self, datas, threshold=0.1):
        self.jpeg_batches.append(len(datas))
        return [[(1, 0.5, float(len(d)), 0.0, 1.0, 1.0)] for d in datas]

    def perform_frames(self, frames, threshold=0.1):
        self.frame_batches.append(len(frames))
        return [[(2, 0.5, float(f.sum() % 1000), 0.0, 1.0, 1.0)] for f in frames]


class _FakePipelinedDetector(_FakeDetector):
    """Adds the two-slot submit / collect surface; checks the service never overruns a slot."""

    def __init__(self):
        super().__init__()
        self.slots = {}

    def submit_jpegs(self, slot, datas, threshold=0.1):
        assert slot in (0, 1) and slot not in self.slots
        self.slots[slot] = self.perform_jpegs(datas, threshold)

    def submit_frames(self, slot, frames, threshold=0.1):
        assert slot in (0, 1) and slot not in self.slots
        self.slots[slot] = self.perform_frames(frames, threshold)

    def collect(self, slot):
        return self.slots.pop(slot)


@pytest.mark.parametrize('fake', ['sync', 'pipelined'])
def test_service_routes_jpeg_bytes_to_the_library_and_other_formats_to_pil(fake):
    det = _FakeDetector() if fake == 'sync' else _FakePipelinedDetector()
    svc = BatchingService(det, max_batch=8, max_delay=0.05)
    a = picture(64, 64, 3)
    jpg = encode(a, quality=80)
    buf = io.BytesIO()
    Image.fromarray(a).save(buf, 'PNG')
    png = buf.getvalue()
    out = {}

    def call(i, data):
        out[i] = svc.perform(data)

    threads = [threading.Thread(target=call, args=(i, jpg if i % 2 == 0 else png)) for i in range(6)]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    svc.close()
    assert sum(det.jpeg_batches) == 3 and sum(det.frame_batches) == 3
    for i in range(6):
        if i % 2 == 0:
            assert out[i] == [(1, 0.5, float(len(jpg)), 0.0, 1.0, 1.0)]
        else:
            assert out[i] == [(2, 0.5, float(a.sum() % 1000), 0.0, 1.0, 1.0)]
    svc2 = BatchingService(det, max_batch=2, max_delay=0.001)
    with pytest.raises(ValueError, match='invalid image size'):
        svc2.perform(encode(picture(32, 64, 1), quality=80))
    svc2.close()


# ------------------------------------------------------------------------------------------ device half (B200)
_model = {}


def gpu_model(wh=(416, 416)):
    if wh not in _model:
        data = modelgen.build_onnx('tiny', 80, 416, 1)
        _model[wh] = (data, _native.Model(data, 80, wh, device=0))
    return _model[wh]


@pytest.mark.gpu
def test_device_decode_bit_exact_against_pillow():
    _, m = gpu_model()
    datas = []
    for i, (sub, q, rst) in enumerate([(0, 75, 0), (1, 75, 0), (2, 75, 0), (2, 95, 7), (2, 10, 0), (0, 100, 1), (1, 50, 3),
                                       (2, 85, 0)]):
        kw = dict(restart_marker_blocks=rst) if rst else {}
        datas.append(encode(modelgen.synthetic_frame(200 + i, 416), quality=q, subsampling=sub, **kw))
    want = np.stack([ref_jpeg.decode_reference(d) for d in datas])
    got = m.decode_jpeg(datas)  # one batch mixing all three chroma layouts
    for i in range(len(datas)):
        assert np.array_equal(got[i], want[i]), i
    for i in (0, 2, 5):  # and one at a time (batch size 1 takes its own execution state)
        assert np.array_equal(m.decode_jpeg([datas[i]])[0], want[i])
    # flat and extreme pictures: saturated colours exercise the clamps of the colour conversion
    extreme = [np.zeros((416, 416, 3), np.uint8), np.full((416, 416, 3), 255, np.uint8),
               np.tile(np.array([[[255, 0, 0], [0, 255, 0]], [[0, 0, 255], [255, 255, 0]]], np.uint8), (208, 208, 1))]
    for a in extreme:
        for sub in (0, 2):
            d = encode(a, quality=90, subsampling=sub)
            assert np.array_equal(m.decode_jpeg([d])[0], ref_jpeg.decode_reference(d))
    # a 416x256 net decoding 416x256 JPEGs (no letterbox): the chroma rows, the MCU grid (26x16 4:2:0 MCUs) and the output
    # rows follow the frame's own width and height
    _, m = gpu_model((416, 256))
    datas = [encode(modelgen.synthetic_frame(230 + sub, 416)[:256], quality=80, subsampling=sub) for sub in (0, 1, 2)]
    got = m.decode_jpeg(datas)
    for i, d in enumerate(datas):
        assert np.array_equal(got[i], ref_jpeg.decode_reference(d)), i


@pytest.mark.gpu
def test_device_decode_of_damaged_streams_equals_pillow():
    """The device IDCT / upsampling / colour kernels on out-of-range coefficients (net size 64x64 model would be needed
    for tiny frames, so the damaged 40x56 streams are checked through full-size ones: damage applied to 416x416 streams)."""
    import warnings
    _, m = gpu_model()
    rng = np.random.default_rng(33)
    base = [encode(modelgen.synthetic_frame(500 + i, 416), quality=q, subsampling=s_) for i, (q, s_) in enumerate([(60, 2), (85, 0), (40, 1)])]
    batch, want, checked = [], [], 0
    with warnings.catch_warnings():
        warnings.simplefilter('ignore')
        for trial in range(400):
            d = bytearray(base[trial % 3])
            start = d.index(b'\xff\xda')
            for _ in range(int(rng.integers(1, 4))):
                pos = int(rng.integers(start + 14, len(d) - 2)) if rng.random() < 0.8 else int(rng.integers(2, start))
                d[pos] ^= 1 << int(rng.integers(0, 8))
            d = bytes(d)
            if _native.jpeg_probe(d).status != _native.FD_JPEG_OK:
                continue
            try:
                _native.jpeg_coefficients(d)
            except _native.JpegRefused:
                continue
            batch.append(d)
            want.append(ref_jpeg.decode_reference(d))
            if len(batch) == 16:
                got = m.decode_jpeg(batch)
                for i in range(16):
                    assert np.array_equal(got[i], want[i]), (trial, i)
                batch, want = [], []
                checked += 16
    assert checked >= 128  # single bit flips mostly re-synchronise: about three quarters of the streams stay decodable


@pytest.mark.gpu
def test_jpeg_of_another_size_is_letterboxed_like_decoded_frames():
    """allow_resize for encoded payloads: decode at the source size on the device, then the same letterbox as
    fd_preprocess — pixels and detections equal the Pillow-decode + letterbox route bit for bit."""
    from fastdet_b200 import detector as fdet
    onnx, m = gpu_model()
    rng = np.random.default_rng(9)
    # odd sizes with subsampled chroma: the last pixel pair of a row has no second pixel, the last chroma column takes the
    # edge rule, and the bottom 4:2:0 output row's context row lies past the picture; 7x6 has 3 chroma columns
    for (h, w, sub) in [(480, 640, 2), (360, 202, 1), (481, 641, 2), (417, 833, 2), (361, 203, 1), (7, 6, 2), (833, 417, 0)]:
        frames = [np.clip(np.kron(rng.integers(0, 255, (h // 8 + 1, w // 8 + 1, 3)), np.ones((8, 8, 1)))[:h, :w] +
                          rng.normal(0, 6, (h, w, 3)), 0, 255).astype(np.uint8) for _ in range(3)]
        datas = [encode(f, quality=85, subsampling=sub) for f in frames]
        decoded = np.stack([ref_jpeg.decode_reference(d) for d in datas])
        want = m.letterbox(decoded)
        got = m.decode_jpeg(datas, allow_resize=True)
        assert np.array_equal(got, want), (h, w)
        d0, c0 = m.detect(decoded, 0.05, allow_resize=True, max_det=256)
        d1, c1 = m.detect_jpeg(datas, 0.05, max_det=256, allow_resize=True)
        assert np.array_equal(c0, c1)
        for f in range(3):
            assert d0[f, :c0[f]].tobytes() == d1[f, :c1[f]].tobytes()
    with pytest.raises(ValueError, match='invalid image size'):
        m.detect_jpeg(datas, 0.05)  # without allow_resize the reference's size check stands
    with pytest.raises(ValueError, match='invalid image size'):  # one size per batch
        m.detect_jpeg([datas[0], encode(modelgen.synthetic_frame(1, 416), quality=80)], 0.05, allow_resize=True)
    det = fdet.ONNXDetector(onnx, num_classes=80, image_size=(416, 416), max_det=256)
    a = det.perform_jpegs(datas, threshold=0.05, allow_resize=True, source_coords=True)
    b = det.perform_frames(decoded, threshold=0.05, allow_resize=True, source_coords=True)
    assert a == b and det.jpeg_device_frames == 3


@pytest.mark.gpu
def test_detect_jpeg_equals_detect_on_pillow_frames():
    _, m = gpu_model()
    datas = [encode(modelgen.synthetic_frame(300 + i, 416), quality=80, subsampling=2 if i % 2 else 0) for i in range(5)]
    frames = np.stack([ref_jpeg.decode_reference(d) for d in datas])
    d0, c0 = m.detect(frames, 0.05, max_det=256)
    d1, c1 = m.detect_jpeg(datas, 0.05, max_det=256)
    assert np.array_equal(c0, c1) and c0.sum() > 0
    for f in range(len(datas)):
        assert d0[f, :c0[f]].tobytes() == d1[f, :c1[f]].tobytes()
    # pipelined form, alternating slots, JPEG and raw batches interleaved
    m.submit_jpeg(0, datas, 0.05, max_det=256)
    m.submit(1, frames, 0.05, max_det=256)
    a = m.collect(0)
    b = m.collect(1)
    m.submit_jpeg(0, datas[:2], 0.05, max_det=256)
    c = m.collect(0)
    assert np.array_equal(a[1], c0) and np.array_equal(b[1], c0) and np.array_equal(c[1], c0[:2])
    for f in range(len(datas)):
        assert a[0][f, :c0[f]].tobytes() == d0[f, :c0[f]].tobytes()
        assert b[0][f, :c0[f]].tobytes() == d0[f, :c0[f]].tobytes()


@pytest.mark.gpu
def test_refused_batches_launch_nothing_and_detector_takes_the_reference_route():
    from fastdet_b200 import detector as fdet
    onnx, m = gpu_model()
    good = encode(modelgen.synthetic_frame(400, 416), quality=80)
    prog = encode(modelgen.synthetic_frame(401, 416), quality=80, progressive=True)
    with pytest.raises(_native.JpegRefused) as e:
        m.detect_jpeg([good, prog, good], 0.1)
    assert e.value.status.tolist() == [_native.FD_JPEG_OK, _native.FD_JPEG_UNSUPPORTED, _native.FD_JPEG_OK]
    with pytest.raises(ValueError, match='invalid image size'):
        m.detect_jpeg([encode(modelgen.synthetic_frame(402, 320), quality=80)], 0.1)
    det = fdet.ONNXDetector(onnx, num_classes=80, image_size=(416, 416), max_det=256)
    want = det.perform_frames(ref_jpeg.decode_reference(good)[None], threshold=0.05)[0]
    assert det.perform(good, threshold=0.05) == want and det.jpeg_device_frames == 1 and det.jpeg_host_frames == 0
    want_p = det.perform_frames(ref_jpeg.decode_reference(prog)[None], threshold=0.05)[0]
    assert det.perform(prog, threshold=0.05) == want_p and det.jpeg_host_frames == 1
    buf = io.BytesIO()
    Image.fromarray(modelgen.synthetic_frame(400, 416)).save(buf, 'PNG')
    assert det.perform(buf.getvalue(), threshold=0.05) == det.perform_frames(modelgen.synthetic_frame(400, 416)[None], threshold=0.05)[0]
    with pytest.raises(ValueError, match='invalid image size'):
        det.perform(encode(modelgen.synthetic_frame(402, 320), quality=80))
    with pytest.raises(ValueError):  # grey JPEG: the reference's reshape fails (detector.py:133)
        det.perform(encode(modelgen.synthetic_frame(403, 416)[..., 0], quality=80))
    with pytest.raises(Exception) as ei:  # not an image at all: PIL's UnidentifiedImageError, as in the reference
        det.perform(b'not an image')
    assert type(ei.value).__name__ == 'UnidentifiedImageError'
    outs = list(det.perform_stream([[good, good], [good]], threshold=0.05))
    assert outs[1] == [want] and outs[0][0] == outs[0][1]  # same batch size: identical; the pair rode in a batch of two
    assert _same_detections(outs[0][0], want, 0.05)


from tests.compare import same_detections as _same_detections  # noqa: E402  (results that rode in different batch sizes)


@pytest.mark.gpu
def test_bad_payload_in_a_batch_is_isolated_on_device():
    """One entropy-damaged JPEG (valid header, so it is queued for the device path) and one progressive JPEG among good
    ones: perform_jpegs(return_exceptions=True) and BatchingService answer every good payload exactly as perform() does and
    hand the damaged one's exception (what PIL raises for it) to its own caller only."""
    from fastdet_b200 import detector as fdet
    onnx, m = gpu_model()
    det = fdet.ONNXDetector(onnx, num_classes=80, image_size=(416, 416), max_det=256)
    good = [encode(modelgen.synthetic_frame(410 + i, 416), quality=80) for i in range(5)]
    prog = encode(modelgen.synthetic_frame(420, 416), quality=80, progressive=True)
    # cut the entropy data short: the header still parses, libjpeg/PIL raise on the truncated stream
    broken = good[0][:len(good[0]) // 3]
    try:
        np.array(Image.open(io.BytesIO(broken)))
        pil_raises = None
    except Exception as e:  # noqa: BLE001
        pil_raises = type(e)
    assert pil_raises is not None and _native.jpeg_probe(broken).status == _native.FD_JPEG_OK
    want = {d: det.perform(d, threshold=0.05) for d in good + [prog]}
    batch = [good[0], good[1], broken, good[2], prog, good[3], good[4]]
    res = det.perform_jpegs(batch, threshold=0.05, return_exceptions=True)
    for d, r in zip(batch, res):
        if d is broken:
            assert isinstance(r, pil_raises)
        else:
            assert not isinstance(r, BaseException) and _same_detections(r, want[d], 0.05)
    with pytest.raises(pil_raises):
        det.perform_jpegs(batch, threshold=0.05)
    svc = BatchingService(det, max_batch=8, max_delay=0.2)
    out = {}

    def call(i):
        try:
            out[i] = svc.perform(batch[i], threshold=0.05)
        except Exception as e:  # noqa: BLE001
            out[i] = e

    threads = [threading.Thread(target=call, args=(i,)) for i in range(len(batch))]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    svc.close()
    for i, d in enumerate(batch):
        if d is broken:
            assert isinstance(out[i], pil_raises)
        else:
            assert not isinstance(out[i], BaseException) and _same_detections(out[i], want[d], 0.05), i
    assert svc.isolated >= 1
