"""The reference's own inputs and its own caller.

* testdata/{dog,rsu1,rsu2}.jpg (reference README.md:34-55) — committed as tests/golden/ref_images.npz by
  tests/golden/make_golden_ref_images.py: streams a camera / another encoder produced (4:2:2 sampling, their own
  Huffman and quantisation tables), unlike every other JPEG in this suite, which this image's Pillow wrote.
  CPU: the restatement (oracle/ref_jpeg.py) and the library's host half reproduce the pixels the reference's decode
  lines give.  GPU: device decode bit-exact, perform(bytes) through the library's JPEG route == the reference's route
  (PIL pixels), and the detections against the oracle's restatement of perform() on those pixels.
* dropin/detector.py as server.py uses it: imported as `detector` from a server/-shaped directory by a fresh
  interpreter, constructed and called with the arguments server.py passes, its answer packed as the response the
  reference client receives (DummyDetector on the CPU, ONNXDetector on the GPU).
* server/server.py + server/client.py, UNCHANGED, over loopback with this repo's `detector` module in place of the
  reference's (the deployment INTEGRATION.md §1 describes).  Those two files are the original project's, not this
  one's: the tests run when FASTDET_REFERENCE names a checkout of it and are skipped otherwise.
"""
import hashlib
import importlib.util
import io
import json
import os
import shutil
import socket
import struct
import subprocess
import sys
import time

import numpy as np
import pytest
from PIL import Image

from fastdet_b200 import _native, modelgen
from oracle import ref_jpeg

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
REF = os.environ.get("FASTDET_REFERENCE", "")
NEEDS_REF = pytest.mark.skipif(not (REF and os.path.exists(os.path.join(REF, "server", "server.py"))),
                               reason="needs FASTDET_REFERENCE: a checkout of the original project (server/server.py, server/client.py)")
NAMES = ("dog", "rsu1", "rsu2")


def fixtures():
    z = np.load(os.path.join(HERE, "golden", "ref_images.npz"))
    return {n: (z[n + "_jpg"].tobytes(), z[n + "_sha256"].tobytes(), z[n + "_probe"]) for n in NAMES}


def test_reference_images_decode_like_the_reference():
    for name, (data, sha, probe) in fixtures().items():
        px = ref_jpeg.decode_reference(data)  # the reference's own lines (PIL)
        assert px.shape == (416, 416, 3)
        assert hashlib.sha256(px.tobytes()).digest() == sha, f"{name}: this image's Pillow decodes the fixture differently"
        assert np.array_equal(px[::52, ::52], probe)
        assert np.array_equal(ref_jpeg.decode(data), px), f"{name}: numpy restatement differs from Pillow"
        info = _native.jpeg_probe(data)
        assert info.status == _native.FD_JPEG_OK and (info.width, info.height) == (416, 416)
        assert (info.h_samp, info.v_samp) == (2, 1)  # 4:2:2 — a layout Pillow's default encoder never produces
        _, planes = _native.jpeg_coefficients(data)  # the library's Huffman decoder on tables it has not seen elsewhere
        assert np.array_equal(ref_jpeg.reconstruct(ref_jpeg.parse(data), planes), px), name
    dog = fixtures()["dog"][2]
    assert dog[0, 0].tolist() == [116, 134, 76]  # SURVEY 8c probe: input (0.4549, 0.5255, 0.2980)


@pytest.mark.gpu
def test_reference_images_on_device():
    from fastdet_b200 import detector as fdet
    from oracle import ref_graph, ref_post
    from tests.test_gpu_parity import DetectionTally
    data = modelgen.build_onnx("tiny", 80, 416, 1)
    det = fdet.ONNXDetector(data, num_classes=80)
    exe, exe16 = ref_graph.GraphExecutor(data), ref_graph.GraphExecutor(data, dtype="bf16")
    t32, t16 = DetectionTally(80, 0.05), DetectionTally(80, 0.05)
    fx = fixtures()
    pixels = {n: ref_jpeg.decode_reference(fx[n][0]) for n in NAMES}
    got = det.model.decode_jpeg([fx[n][0] for n in NAMES])
    for i, n in enumerate(NAMES):
        assert np.array_equal(got[i], pixels[n]), f"{n}: device JPEG decode differs from PIL"
    for n in NAMES:
        res = det.perform(fx[n][0], threshold=0.05)
        assert res == det.perform_frames(pixels[n][None], threshold=0.05)[0]  # JPEG route == the reference's route
        dets, counts = det.model.detect(pixels[n][None], 0.05)
        x = ref_post.normalise(pixels[n])
        h32, h16 = exe.run(x), exe16.run(x)
        t32.add(h32, dets[0, :counts[0]])
        t32.add_floor(h32, h16)  # photographs drive these random-init nets harder than the synthetic frames: bounds follow the CPU floor
        t16.add(h16, dets[0, :counts[0]])
        t16.add_floor(h32, h16)
    assert det.jpeg_device_frames == len(NAMES) and det.jpeg_host_frames == 0
    t32.check("reference images vs fp32 oracle", min_solid=3)
    t16.check("reference images vs bf16-operand oracle", min_solid=3)


# ------------------------------------------------------------------------------------------ the drop-in module
# The calls server.py makes on its `detector` module (INTEGRATION.md §1), run by a fresh interpreter in a directory laid out
# like the reference's server/ with dropin/detector.py as its detector.py.
_SERVER_CALLS = r"""
import json, sys
from detector import DummyDetector, ONNXDetector                                          # server.py:17
data_path, spec, threshold, dbgout = sys.argv[1], sys.argv[2], int(sys.argv[3]), sys.argv[4] or None
if spec:                                                                                  # "name:classes:path", :355-358
    name, num_classes, path = spec.split(":")
    detector = ONNXDetector(path, mode=None, num_classes=int(num_classes), dbgout=dbgout)
else:                                                                                     # no model argument, :359-360
    detector = DummyDetector(dbgout=dbgout)
with open(data_path, "rb") as fp:
    print(json.dumps(detector.perform(fp.read(), threshold=threshold * 0.01)))           # :232
"""


def _perform_through_dropin(tmp_path, payload, spec="", threshold_percent=10, dbgout=""):
    srv = tmp_path / "server"
    srv.mkdir()
    shutil.copy(os.path.join(ROOT, "dropin", "detector.py"), srv / "detector.py")
    (tmp_path / "payload.jpg").write_bytes(payload)
    env = dict(os.environ, FASTDET_B200_HOME=ROOT)  # where the deployment finds the package (INTEGRATION.md §1)
    r = subprocess.run([sys.executable, "-c", _SERVER_CALLS, str(tmp_path / "payload.jpg"), spec, str(threshold_percent), dbgout],
                       cwd=str(srv), env=env, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=300)
    assert r.returncode == 0, r.stderr[-3000:]
    return [tuple(t) for t in json.loads(r.stdout.strip().splitlines()[-1])]


def test_dropin_module_answers_server_calls_dummy(tmp_path):
    """No model argument: DummyDetector from the drop-in answers with the reference's fixed box, packed as the response
    the reference client receives, and dumps the payload to dbgout as the reference's -o does."""
    from oracle import ref_wire
    dog = fixtures()["dog"][0]
    got = _perform_through_dropin(tmp_path, dog, dbgout=str(tmp_path / "dbgout"))
    assert got == [(16, 1.0, 208.0, 208.0, 166.4, 166.4)]
    assert _unpack(ref_wire.pack_results(got, 7, 0)) == (7, [(16, 255, 208, 208, 166, 166)])
    assert (tmp_path / "dbgout").read_bytes() == dog


@pytest.mark.gpu
def test_dropin_module_answers_server_calls_onnx(tmp_path):
    """`name:classes:model.onnx`: ONNXDetector from the drop-in, built and called as server.py does, returns what the
    package's ONNXDetector.perform returns for the same payload, and packs to the same response."""
    from fastdet_b200 import detector as fdet
    from oracle import ref_wire
    data = modelgen.build_onnx("tiny", 80, 416, 1)
    onnx_path = tmp_path / "tiny.onnx"
    onnx_path.write_bytes(data)
    dog = fixtures()["dog"][0]
    got = _perform_through_dropin(tmp_path, dog, spec=f"tiny:80:{onnx_path}")
    want = fdet.ONNXDetector(data, num_classes=80).perform(dog, threshold=0.1)
    assert want and got == want
    assert ref_wire.pack_results(got, 7, 0) == ref_wire.pack_results(want, 7, 0)


# ------------------------------------------------------------------------------------------ the unchanged caller
def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    return port


def _deploy(tmp_path):
    """What INTEGRATION.md §1 tells a maintainer to do: the reference's server/ directory with detector.py replaced."""
    srv = tmp_path / "server"
    srv.mkdir()
    for f in ("server.py", "client.py"):
        shutil.copy(os.path.join(REF, "server", f), srv / f)
    shutil.copy(os.path.join(ROOT, "dropin", "detector.py"), srv / "detector.py")
    for f in ("server.py", "client.py"):  # unchanged, byte for byte
        with open(srv / f, "rb") as a, open(os.path.join(REF, "server", f), "rb") as b:
            assert a.read() == b.read()
    return srv


def _round_trip(srv, server_args, payload, path, threshold=0.1, wait=60.0):
    port = _free_port()
    env = dict(os.environ, PYTHONPATH=ROOT + os.pathsep + os.environ.get("PYTHONPATH", ""), FASTDET_B200_HOME=ROOT)
    proc = subprocess.Popen([sys.executable, str(srv / "server.py"), "-s", str(port)] + server_args, env=env, cwd=str(srv),
                            stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    try:
        spec = importlib.util.spec_from_file_location("reference_client", str(srv / "client.py"))
        client_mod = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(client_mod)
        deadline = time.time() + wait
        client = None
        while time.time() < deadline:
            try:
                client = client_mod.RTSPClient("127.0.0.1", port, path)
                client.open()
                break
            except (ConnectionRefusedError, OSError):
                client = None
                assert proc.poll() is None, proc.stdout.read()
                time.sleep(0.2)
        assert client is not None, "server did not come up"
        answers = []
        client.process_data = answers.append  # the client's own RTP reassembly hands us the response payload
        client.request(7, threshold, payload)
        while not answers and time.time() < deadline:
            client.idle(0.2)
        assert answers, "no response from the server"
        return _unpack(answers[0])
    finally:
        proc.terminate()
        try:
            proc.wait(5)
        except subprocess.TimeoutExpired:
            proc.kill()


def _unpack(resp):
    tp, reqid, msec, length = struct.unpack(">4sLLL", resp[:16])
    assert tp == b"YOLO" and length == len(resp) - 16 and length % 10 == 0
    return reqid, [struct.unpack(">BBhhhh", resp[16 + i:26 + i]) for i in range(0, length, 10)]


@NEEDS_REF
def test_unchanged_server_and_client_round_trip_dummy(tmp_path):
    """No model argument -> server.py builds DummyDetector from OUR detector module (server.py:17,360) and answers the
    reference client's request with the packed fixed box (detector.py:83-92 -> server.py:234-239)."""
    srv = _deploy(tmp_path)
    dog = fixtures()["dog"][0]
    reqid, recs = _round_trip(srv, [], dog, "detect")
    assert reqid == 7 and recs == [(16, 255, 208, 208, 166, 166)]


@pytest.mark.gpu
@NEEDS_REF
def test_unchanged_server_and_client_round_trip_onnx(tmp_path):
    """`server.py full:80:model.onnx` with our module: the response the reference client receives is the wire packing of
    ONNXDetector.perform on the same payload.  (Runs only where a GPU and the reference checkout are both present.)"""
    from fastdet_b200 import detector as fdet
    from oracle import ref_wire
    srv = _deploy(tmp_path)
    data = modelgen.build_onnx("tiny", 80, 416, 1)
    onnx_path = tmp_path / "tiny.onnx"
    onnx_path.write_bytes(data)
    dog = fixtures()["dog"][0]
    reqid, recs = _round_trip(srv, [f"tiny:80:{onnx_path}"], dog, "tiny", wait=180.0)
    want = fdet.ONNXDetector(data, num_classes=80).perform(dog, threshold=0.1)
    assert reqid == 7 and recs == _unpack(ref_wire.pack_results(want, 7, 0))[1]
