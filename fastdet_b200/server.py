"""server.py — multi-model, multi-GPU detection service in one process (BASELINE config 5).

The reference's ``server/server.py`` builds a dict ``detectors[name] = ONNXDetector(path, ...)`` (:355-358), hands the
SAME dict to every RTSP session (:295, :311-312) and serves each payload with one blocking
``detector.perform(data, threshold)`` (:232).  ``DetectServer`` is that dict on every GPU of the box: each model spec is
replicated per device, a stream (session) is pinned to one device (``stream_id % n_devices``), and ``perform`` keeps the
reference's call shape — blocking, one frame in, that frame's result tuples out — while being callable from any number of
threads at once: concurrent calls for the same (device, model) share micro-batches, two of which are in flight per lane.
The queues, worker threads and batching live in the native library (csrc/server.cc, ``fd_server_*`` in
include/fastdet_b200.h); this class owns the handle and converts records to the reference's tuples.

    srv = DetectServer({"full": (full_onnx_bytes, 80), "rsu": (rsu_onnx_bytes, 9)}, devices=range(8))
    results = srv.perform("full", stream_id, frame_u8_hwc, threshold=0.1)     # [(klass, conf, x, y, w, h), ...]
    srv.detector("full", stream_id).perform(jpeg_bytes, threshold)           # drop-in object for server.py's dict

JPEG payloads (``perform_jpeg_records`` and the drop-in object) take the device decode path of ``fd_detect_jpeg``: each
caller entropy-decodes its payload in its own thread straight into the lane's open micro-batch, and requests with
different thresholds share that batch.  Payloads the device decoder refuses (PNG, progressive, greyscale, damaged
entropy data) are decoded with PIL by the drop-in object, as the reference does.
"""
import ctypes as C
import io

import numpy as np

from . import _native


class DetectServer:
    def __init__(self, models, devices=(0,), image_size=(416, 416), max_batch=64, max_det=256, max_delay_ms=0.0):
        """models: {name: (onnx bytes or path, num_classes)} (the reference's ``name:num_classes:path`` specs)."""
        self.names = list(models)
        self.image_size = tuple(image_size)
        self.devices = [int(d) for d in devices]
        self.max_det = int(max_det)
        self.num_classes = {}
        specs = (_native.FdServerModel * len(self.names))()
        self._keep = []
        for i, name in enumerate(self.names):
            data, nc = models[name]
            if not isinstance(data, (bytes, bytearray)):
                with open(data, "rb") as fp:
                    data = fp.read()
            buf = C.create_string_buffer(bytes(data), len(data))
            self._keep.append(buf)
            specs[i] = _native.FdServerModel(C.cast(buf, C.c_void_p), len(data), int(nc), self.image_size[0], self.image_size[1])
            self.num_classes[name] = int(nc)
        devs = (C.c_int32 * len(self.devices))(*self.devices)
        self._h = C.c_void_p()
        _native._check(_native.lib().fd_server_create(specs, len(self.names), devs, len(self.devices), int(max_batch), self.max_det,
                                                      float(max_delay_ms), C.byref(self._h)))
        self._keep = []  # the library has parsed and uploaded the graphs

    @classmethod
    def fake(cls, n_models=2, n_devices=2, image_size=(8, 8), max_batch=8, max_delay_ms=0.0, latency_us=0):
        """Host-only stand-in backend (no GPU): for tests of the routing and batching logic."""
        self = cls.__new__(cls)
        self.names = [f"m{i}" for i in range(n_models)]
        self.image_size = tuple(image_size)
        self.devices = list(range(n_devices))
        self.max_det = 1
        self.num_classes = {n: 255 for n in self.names}
        self._h = C.c_void_p()
        _native._check(_native.lib().fd_server_create_fake(n_models, n_devices, image_size[0], image_size[1], int(max_batch),
                                                           float(max_delay_ms), int(latency_us), C.byref(self._h)))
        return self

    def close(self):
        if getattr(self, "_h", None) is not None and self._h.value:
            _native.lib().fd_server_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @staticmethod
    def _check(rc):
        if rc == _native.FD_OK:
            return
        msg = (_native.lib().fd_server_last_error() or b"").decode("utf-8", "replace")
        if rc == _native.FD_ERR_SIZE:
            raise ValueError(msg)  # reference: ValueError('invalid image size'), server/detector.py:132
        raise _native.NativeError(rc, msg)

    def perform_records(self, model, stream_id, frame, threshold=0.1):
        """frame: [h, w, 3] u8 RGB.  Returns the frame's fd_det records (structured array)."""
        frame = np.ascontiguousarray(frame, np.uint8)
        if frame.ndim != 3 or frame.shape[2] != 3:
            raise ValueError("invalid image size")
        h, w, _ = frame.shape
        out = np.zeros(self.max_det, _native.DET_DTYPE)
        count = C.c_int32()
        m = model if isinstance(model, int) else self.names.index(model)
        self._check(_native.lib().fd_server_perform(self._h, int(stream_id), m, _native._ptr(frame), w, h, float(threshold),
                                                    _native._ptr(out), self.max_det, C.byref(count)))
        return out[:count.value]

    def perform_jpeg_records(self, model, stream_id, data, threshold=0.1):
        """data: one JPEG payload (bytes).  Returns the frame's fd_det records (structured array).  Raises
        _native.JpegRefused (with the FD_JPEG_* status) for a payload the device decoder does not take or whose entropy data
        is damaged, and ValueError('invalid image size') for a frame that is not the model's size."""
        data = bytes(data)
        out = np.zeros(self.max_det, _native.DET_DTYPE)
        count, status = C.c_int32(), C.c_int32()
        m = model if isinstance(model, int) else self.names.index(model)
        rc = _native.lib().fd_server_perform_jpeg(self._h, int(stream_id), m, data, len(data), float(threshold), _native._ptr(out),
                                                  self.max_det, C.byref(count), C.byref(status))
        if rc == _native.FD_ERR_JPEG:
            msg = (_native.lib().fd_server_last_error() or b"").decode("utf-8", "replace")
            raise _native.JpegRefused(msg, np.array([status.value], np.int32))
        self._check(rc)
        return out[:count.value]

    def perform(self, model, stream_id, frame, threshold=0.1):
        """The reference's result list for one decoded frame: [(klass, conf, x, y, w, h), ...] (detector.py:142-144)."""
        return self.perform_records(model, stream_id, frame, threshold)[["klass", "conf", "x", "y", "w", "h"]].tolist()

    def warm(self, up_to=64):
        """Builds every lane's execution state for batches of up to `up_to` frames now (seconds), so no request ever does."""
        self._check(_native.lib().fd_server_warm(self._h, int(up_to)))

    def lane_stats(self):
        out = {}
        b, f = C.c_int64(), C.c_int64()
        for d in range(len(self.devices)):
            for m, name in enumerate(self.names):
                _native._check(_native.lib().fd_server_lane_stats(self._h, d, m, C.byref(b), C.byref(f)))
                out[(d, name)] = (b.value, f.value)
        return out

    def closed_loop(self, stream_models, frames, threshold=0.1, warmup_seconds=1.0, seconds=10.0):
        """Native load generator: len(stream_models) caller threads (stream i -> model stream_models[i], device slot
        i % n_devices), each sending its next frame as soon as its previous result is back.  frames: [k, h, w, 3] u8."""
        frames = np.ascontiguousarray(frames, np.uint8)
        k, h, w, _ = frames.shape
        idx = [m if isinstance(m, int) else self.names.index(m) for m in stream_models]
        sm = (C.c_int32 * len(idx))(*idx)
        st = _native.FdServeStats()
        self._check(_native.lib().fd_server_closed_loop(self._h, len(idx), sm, _native._ptr(frames), k, w, h, float(threshold),
                                                        float(warmup_seconds), float(seconds), C.byref(st)))
        return {"seconds": st.seconds, "frames": st.frames, "frames_per_second": st.frames_per_second,
                "latency_ms": {"p50": st.latency_ms_p50, "p90": st.latency_ms_p90, "p99": st.latency_ms_p99, "mean": st.latency_ms_mean,
                               "max": st.latency_ms_max},
                "batches": st.batches, "mean_batch": st.mean_batch, "detections": st.detections, "streams": st.streams,
                "frames_per_device": list(st.frames_per_device)[:len(self.devices)],
                "frames_per_model": dict(zip(self.names, list(st.frames_per_model)))}

    def detector(self, model, stream_id=0):
        """An object with the reference detector's surface (image_size, num_classes, perform(data, threshold)) bound to one
        model and one stream: what ``detectors[name]`` holds in server/server.py:355-358."""
        return _BoundDetector(self, model, stream_id)


class _BoundDetector:
    def __init__(self, server, model, stream_id):
        self.server, self.model, self.stream_id = server, model, stream_id
        self.image_size = server.image_size
        self.num_classes = server.num_classes[model if not isinstance(model, int) else server.names[model]]

    def __repr__(self):
        return f"<DetectServer.detector model={self.model}, stream={self.stream_id}, devices={self.server.devices}>"

    def perform(self, data, threshold=0.1):
        """Encoded payload in, like the reference (detector.py:126-146).  A JPEG the device decoder takes rides the lane's JPEG
        micro-batch; anything else is decoded with PIL in the caller's thread, so it gives the reference's result or exception."""
        try:
            recs = self.server.perform_jpeg_records(self.model, self.stream_id, data, threshold)
            return recs[["klass", "conf", "x", "y", "w", "h"]].tolist()
        except _native.JpegRefused:
            pass
        from PIL import Image
        img = Image.open(io.BytesIO(data))
        if img.size != self.image_size:
            raise ValueError("invalid image size")
        (width, height) = img.size
        frame = np.array(img)
        if frame.ndim != 3 or frame.shape[2] != 3:
            raise ValueError(f"cannot reshape array of size {frame.size} into shape (1,{height},{width},3)")
        return self.server.perform(self.model, self.stream_id, frame, threshold)
