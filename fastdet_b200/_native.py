"""ctypes binding of libfastdet_b200.so (include/fastdet_b200.h).

There is deliberately no fallback: if the shared library is missing or a CUDA call fails, the error
propagates.  The only thing this module does without a GPU is load the library and run its host-side
planner (``Model(..., device=-1)``).
"""
from __future__ import annotations

import ctypes as C
import os
from typing import List, Optional, Sequence, Tuple

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("FASTDET_LIB") or os.path.join(_HERE, "libfastdet_b200.so")  # FASTDET_LIB: developer A/B runs

FD_OK, FD_ERR_ARG, FD_ERR_MODEL, FD_ERR_HEADS, FD_ERR_CUDA, FD_ERR_SIZE, FD_ERR_JPEG = 0, -1, -2, -3, -4, -5, -6
FD_JPEG_OK, FD_JPEG_NOT_JPEG, FD_JPEG_CORRUPT, FD_JPEG_UNSUPPORTED, FD_JPEG_SIZE = 0, 1, 2, 3, 4
FD_MAX_HEADS = 4
FD_MAX_SLOTS = 2


class FdDet(C.Structure):
    _fields_ = [("klass", C.c_int32), ("box", C.c_int32), ("conf", C.c_double), ("x", C.c_double),
                ("y", C.c_double), ("w", C.c_double), ("h", C.c_double)]


DET_DTYPE = np.dtype([("klass", "<i4"), ("box", "<i4"), ("conf", "<f8"), ("x", "<f8"), ("y", "<f8"),
                      ("w", "<f8"), ("h", "<f8")])
assert DET_DTYPE.itemsize == C.sizeof(FdDet) == 48


class FdInfo(C.Structure):
    _fields_ = [("abi_version", C.c_int32), ("device", C.c_int32), ("net_w", C.c_int32), ("net_h", C.c_int32),
                ("num_classes", C.c_int32), ("n_heads", C.c_int32),
                ("head_h", C.c_int32 * FD_MAX_HEADS), ("head_w", C.c_int32 * FD_MAX_HEADS),
                ("head_c", C.c_int32 * FD_MAX_HEADS), ("anchors", C.c_float * (FD_MAX_HEADS * 3 * 2)),
                ("boxes_per_frame", C.c_int32), ("n_layers", C.c_int32), ("n_conv", C.c_int32),
                ("launches_per_detect", C.c_int32), ("conv_flops_per_frame", C.c_double),
                ("num_params", C.c_uint64), ("weight_bytes", C.c_uint64)]


class FdLayerDesc(C.Structure):
    _fields_ = [("kind", C.c_int32), ("c", C.c_int32), ("h", C.c_int32), ("w", C.c_int32), ("cin", C.c_int32),
                ("ksize", C.c_int32), ("stride", C.c_int32), ("act", C.c_int32), ("has_residual", C.c_int32),
                ("upsample2x", C.c_int32), ("out_fp32", C.c_int32), ("block_n", C.c_int32), ("flops", C.c_double),
                ("name", C.c_char * 96), ("out_name", C.c_char * 96)]


class FdLayerExec(C.Structure):
    _fields_ = [("kernel", C.c_int32), ("bucket", C.c_int32), ("block_n", C.c_int32), ("split_k", C.c_int32),
                ("grid", C.c_int32), ("num_stages", C.c_int32), ("kb_per_stage", C.c_int32), ("b_resident", C.c_int32),
                ("smem_bytes", C.c_int32), ("chunk_frames", C.c_int32), ("launches", C.c_int32),
                ("reserved", C.c_int32 * 5)]


KERNEL_NAMES = {0: "conv0", 1: "tc_single", 2: "tc_pair", 3: "tc_pair_strip", 4: "tc_swapped", 5: "halo", 6: "maxpool",
                7: "copy", 8: "stem", 9: "fused_next", 10: "block"}


FD_SERVER_MAX_MODELS, FD_SERVER_MAX_DEVICES = 8, 16


class FdServerModel(C.Structure):
    _fields_ = [("onnx_bytes", C.c_void_p), ("len", C.c_size_t), ("num_classes", C.c_int32), ("net_w", C.c_int32),
                ("net_h", C.c_int32)]


class FdServeStats(C.Structure):
    _fields_ = [("seconds", C.c_double), ("frames", C.c_int64), ("frames_per_second", C.c_double),
                ("latency_ms_p50", C.c_double), ("latency_ms_p90", C.c_double), ("latency_ms_p99", C.c_double),
                ("latency_ms_mean", C.c_double), ("latency_ms_max", C.c_double), ("batches", C.c_int64),
                ("mean_batch", C.c_double), ("detections", C.c_int64), ("streams", C.c_int32), ("reserved", C.c_int32),
                ("frames_per_device", C.c_int64 * FD_SERVER_MAX_DEVICES), ("frames_per_model", C.c_int64 * FD_SERVER_MAX_MODELS)]


class FdJpegInfo(C.Structure):
    _fields_ = [("status", C.c_int32), ("width", C.c_int32), ("height", C.c_int32), ("components", C.c_int32),
                ("h_samp", C.c_int32), ("v_samp", C.c_int32), ("restart_interval", C.c_int32),
                ("blocks_w", C.c_int32 * 3), ("blocks_h", C.c_int32 * 3), ("coef_count", C.c_int64),
                ("quant", C.c_uint16 * (3 * 64)), ("reason", C.c_char * 160)]


# every symbol include/fastdet_b200.h declares, with its ctypes signature
_PROTOS = {
    "fd_last_error": (C.c_char_p, []),
    "fd_abi_version": (C.c_int, []),
    "fd_device_count": (C.c_int, []),
    "fd_model_create": (C.c_int, [C.c_void_p, C.c_size_t, C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_void_p)]),
    "fd_model_destroy": (None, [C.c_void_p]),
    "fd_model_info": (C.c_int, [C.c_void_p, C.POINTER(FdInfo)]),
    "fd_layer_info": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(FdLayerDesc)]),
    "fd_layer_exec_info": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.POINTER(FdLayerExec)]),
    "fd_planned_fusions": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(C.c_int32), C.POINTER(C.c_int32)]),
    "fd_set_option": (C.c_int, [C.c_char_p, C.c_int]),
    "fd_get_option": (C.c_int, [C.c_char_p, C.POINTER(C.c_int)]),
    "fd_preprocess": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "fd_forward": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p]),
    "fd_postprocess": (C.c_int, [C.c_void_p, C.c_int, C.c_double, C.c_int, C.c_void_p]),
    "fd_postprocess_thresholds": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_void_p]),
    "fd_fetch": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "fd_detect": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_double, C.c_int,
                            C.c_void_p, C.c_void_p]),
    "fd_submit": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_double, C.c_int]),
    "fd_collect": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]),
    "fd_jpeg_probe": (C.c_int, [C.c_void_p, C.c_size_t, C.POINTER(FdJpegInfo)]),
    "fd_jpeg_coefficients": (C.c_int, [C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, C.POINTER(FdJpegInfo)]),
    "fd_decode_jpeg": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p]),
    "fd_detect_jpeg": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_double, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]),
    "fd_submit_jpeg": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_double, C.c_int, C.c_void_p]),
    "fd_letterbox_geometry": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_int] + [C.POINTER(C.c_int32)] * 4),
    "fd_unmap_letterbox": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int]),
    "fd_pack_wire": (C.c_int, [C.c_void_p, C.c_int, C.c_uint32, C.c_uint32, C.c_int, C.c_void_p, C.c_size_t, C.POINTER(C.c_size_t)]),
    "fd_server_create": (C.c_int, [C.POINTER(FdServerModel), C.c_int, C.POINTER(C.c_int32), C.c_int, C.c_int, C.c_int, C.c_double,
                                   C.POINTER(C.c_void_p)]),
    "fd_server_create_fake": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_double, C.c_int, C.POINTER(C.c_void_p)]),
    "fd_server_destroy": (None, [C.c_void_p]),
    "fd_server_perform": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_double, C.c_void_p, C.c_int,
                                    C.POINTER(C.c_int32)]),
    "fd_server_perform_jpeg": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_size_t, C.c_double, C.c_void_p, C.c_int,
                                         C.POINTER(C.c_int32), C.POINTER(C.c_int32)]),
    "fd_server_warm": (C.c_int, [C.c_void_p, C.c_int]),
    "fd_server_lane_stats": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.POINTER(C.c_int64), C.POINTER(C.c_int64)]),
    "fd_server_closed_loop": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(C.c_int32), C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_double,
                                        C.c_double, C.c_double, C.POINTER(FdServeStats)]),
    "fd_server_last_error": (C.c_char_p, []),
    "fd_heads_fp32": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_int]),
    "fd_set_heads_fp32": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_int]),
    "fd_layer_output_fp32": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_int]),
    "fd_normalise_f32": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]),
    "fd_letterbox_u8": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "fd_time_layers": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_void_p]),
    "fd_time_forward": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.POINTER(C.c_float)]),
}

_lib = None


def lib() -> C.CDLL:
    """Loads the shared library (once).  Raises if it has not been built — never falls back."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(f"{LIB_PATH} is missing: build it with `python -m fastdet_b200.build` "
                              "(fastdet_b200 has no CPU or pure-Python fallback)")
        l = C.CDLL(LIB_PATH)
        for name, (res, args) in _PROTOS.items():
            fn = getattr(l, name)
            fn.restype = res
            fn.argtypes = args
        _lib = l
    return _lib


class NativeError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"fastdet_b200 native error {code}: {msg}")
        self.code = code
        self.msg = msg


class JpegRefused(NativeError):
    """FD_ERR_JPEG: a frame is not a JPEG the device decoder takes; nothing was launched.  ``status`` holds one
    FD_JPEG_* per frame.  The caller decodes those bytes the way the reference does (PIL) instead."""

    def __init__(self, msg: str, status):
        super().__init__(FD_ERR_JPEG, msg)
        self.status = status


def _check(rc: int):
    if rc == FD_OK:
        return
    msg = (lib().fd_last_error() or b"").decode("utf-8", "replace")
    if rc == FD_ERR_SIZE:
        raise ValueError(msg)  # reference: ValueError('invalid image size'), server/detector.py:132
    if rc == FD_ERR_HEADS:
        raise KeyError(int(msg) if msg.lstrip("-").isdigit() else msg)  # reference: ANCHORS[len(outputs)], :136
    raise NativeError(rc, msg)


def _ptr(a: np.ndarray):
    return a.ctypes.data_as(C.c_void_p)


class Model:
    """One loaded network on one device (``device=-1``: plan only, no CUDA)."""

    def __init__(self, onnx_bytes: bytes, num_classes: int, net_wh: Tuple[int, int] = (416, 416), device: int = 0):
        self._h = C.c_void_p()
        buf = C.create_string_buffer(onnx_bytes, len(onnx_bytes))
        _check(lib().fd_model_create(buf, len(onnx_bytes), num_classes, net_wh[0], net_wh[1], device, C.byref(self._h)))
        info = FdInfo()
        _check(lib().fd_model_info(self._h, C.byref(info)))
        self.info = info
        self.net_w, self.net_h = info.net_w, info.net_h
        self.n_heads = info.n_heads
        self.head_shapes = [(info.head_c[i], info.head_h[i], info.head_w[i]) for i in range(info.n_heads)]
        self.device = device

    def close(self):
        if getattr(self, "_h", None) is not None and self._h.value:
            lib().fd_model_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # -- introspection
    def layers(self) -> List[dict]:
        out = []
        d = FdLayerDesc()
        for i in range(self.info.n_layers):
            _check(lib().fd_layer_info(self._h, i, C.byref(d)))
            out.append({k: (getattr(d, k).decode() if isinstance(getattr(d, k), bytes) else getattr(d, k))
                        for k, _ in FdLayerDesc._fields_})
        return out

    def planned_fusions(self, n: int) -> Tuple[bool, int]:
        """(stem, block_layer): whether layers 0 + 1 would run as the fused stem kernel, and the first layer of the pair that
        would run as the fused residual-block kernel (-1: none) at batch n.  Host logic: works on a plan-only model."""
        stem, block = C.c_int32(0), C.c_int32(-1)
        _check(lib().fd_planned_fusions(self._h, n, C.byref(stem), C.byref(block)))
        return bool(stem.value), int(block.value)

    def exec_info(self, n: int) -> List[dict]:
        """Kernel form of every fused layer in the execution state of batch size n (built if needed)."""
        out = []
        d = FdLayerExec()
        for i in range(self.info.n_layers):
            _check(lib().fd_layer_exec_info(self._h, i, n, C.byref(d)))
            row = {k: getattr(d, k) for k, _ in FdLayerExec._fields_ if k != "reserved"}
            row["kernel_name"] = KERNEL_NAMES.get(d.kernel, str(d.kernel))
            out.append(row)
        return out

    # -- staged pipeline (asynchronous on `stream`, a cudaStream_t as int; 0 = the model's own stream)
    def preprocess(self, frames, n: int, src_wh: Tuple[int, int], on_device=False, allow_resize=False, stream=0):
        p = C.c_void_p(frames) if isinstance(frames, int) else _ptr(frames)
        _check(lib().fd_preprocess(self._h, p, n, src_wh[0], src_wh[1], int(on_device), int(allow_resize), C.c_void_p(stream)))

    def forward(self, n: int, stream=0):
        _check(lib().fd_forward(self._h, n, C.c_void_p(stream)))

    def postprocess(self, n: int, threshold: float, max_det: int = 2048, stream=0):
        _check(lib().fd_postprocess(self._h, n, float(threshold), max_det, C.c_void_p(stream)))
        self._max_det = max_det

    def postprocess_thresholds(self, thresholds, max_det: int = 2048, stream=0):
        """postprocess with one threshold per frame: frame f at thresholds[f] (n = len(thresholds))."""
        thr = np.ascontiguousarray(thresholds, np.float64)
        _check(lib().fd_postprocess_thresholds(self._h, thr.size, _ptr(thr), max_det, C.c_void_p(stream)))
        self._max_det = max_det

    def fetch(self, n: int, stream=0):
        dets = np.zeros((n, self._max_det), DET_DTYPE)
        counts = np.zeros(n, np.int32)
        total = np.zeros(n, np.int32)
        _check(lib().fd_fetch(self._h, n, _ptr(dets), _ptr(counts), _ptr(total), C.c_void_p(stream)))
        return dets, counts, total

    def detect(self, frames: np.ndarray, threshold: float, allow_resize=False, max_det: int = 2048, with_total=False):
        """frames: [n, h, w, 3] u8 (host).  Returns (dets[n, max_det] structured, counts[n]) and, with_total, the number of
        detections each frame had before the cut at max_det."""
        if frames.dtype != np.uint8 or frames.ndim != 4 or frames.shape[3] != 3:
            raise ValueError("invalid image size")
        frames = np.ascontiguousarray(frames)
        n, h, w, _ = frames.shape
        dets = np.zeros((n, max_det), DET_DTYPE)
        counts = np.zeros(n, np.int32)
        _check(lib().fd_detect(self._h, _ptr(frames), n, w, h, 0, int(allow_resize), float(threshold), max_det,
                               _ptr(dets), _ptr(counts)))
        if with_total:
            total = np.zeros(n, np.int32)
            _check(lib().fd_fetch(self._h, n, _ptr(dets), _ptr(counts), _ptr(total), None))  # the same records again + the totals
            return dets, counts, total
        return dets, counts

    # -- pipelined serving: two batches in flight, the H2D copy of one overlaps the compute of the other
    def submit(self, slot: int, frames, threshold: float, allow_resize=False, max_det: int = 2048, n=None, src_wh=None,
               on_device=False):
        """frames: [n, h, w, 3] u8 numpy array (ideally backed by pinned memory) or a raw pointer (then give n and
        src_wh).  The caller keeps `frames` alive and unmodified until collect(slot) returns."""
        if isinstance(frames, int):
            p, (w, h) = C.c_void_p(frames), src_wh
        else:
            if frames.dtype != np.uint8 or frames.ndim != 4 or frames.shape[3] != 3 or not frames.flags.c_contiguous:
                raise ValueError("invalid image size")
            n, h, w, _ = frames.shape
            p = _ptr(frames)
        _check(lib().fd_submit(self._h, slot, p, n, w, h, int(on_device), int(allow_resize), float(threshold), max_det))
        if not hasattr(self, "_slot_shape"):
            self._slot_shape = {}
        self._slot_shape[slot] = (n, max_det, frames)

    # -- JPEG in (reference server/detector.py:128-133): Huffman decode on host threads, the rest on the device
    @staticmethod
    def _jpeg_args(datas):
        n = len(datas)
        keep = [d if isinstance(d, bytes) else bytes(d) for d in datas]
        ptrs = (C.c_char_p * n)(*keep)
        lens = (C.c_size_t * n)(*[len(d) for d in keep])
        return n, keep, ptrs, lens, np.zeros(n, np.int32)

    @staticmethod
    def _check_jpeg(rc, status):
        if rc == FD_ERR_JPEG:
            raise JpegRefused((lib().fd_last_error() or b"").decode("utf-8", "replace"), status)
        _check(rc)

    def decode_jpeg(self, datas, want_rgb=True, allow_resize=False):
        """Decodes a list of JPEG byte strings into the input tensor of batch size len(datas); returns the decoded
        frames [n, net_h, net_w, 3] u8 if want_rgb (parity hook), and leaves them on the device for forward(n)."""
        n, keep, ptrs, lens, status = self._jpeg_args(datas)
        rgb = np.empty((n, self.net_h, self.net_w, 3), np.uint8) if want_rgb else None
        rc = lib().fd_decode_jpeg(self._h, ptrs, lens, n, int(allow_resize), _ptr(status), _ptr(rgb) if want_rgb else None)
        self._check_jpeg(rc, status)
        return rgb

    def detect_jpeg(self, datas, threshold: float, max_det: int = 2048, allow_resize=False):
        n, keep, ptrs, lens, status = self._jpeg_args(datas)
        dets = np.zeros((n, max_det), DET_DTYPE)
        counts = np.zeros(n, np.int32)
        rc = lib().fd_detect_jpeg(self._h, ptrs, lens, n, int(allow_resize), float(threshold), max_det, _ptr(dets), _ptr(counts),
                                  _ptr(status))
        self._check_jpeg(rc, status)
        return dets, counts

    def submit_jpeg(self, slot: int, datas, threshold: float, max_det: int = 2048, allow_resize=False):
        n, keep, ptrs, lens, status = self._jpeg_args(datas)
        rc = lib().fd_submit_jpeg(self._h, slot, ptrs, lens, n, int(allow_resize), float(threshold), max_det, _ptr(status))
        self._check_jpeg(rc, status)
        if not hasattr(self, "_slot_shape"):
            self._slot_shape = {}
        self._slot_shape[slot] = (n, max_det, None)  # the coefficients are already in the slot's pinned buffer

    def collect(self, slot: int):
        n, max_det, _keepalive = self._slot_shape.pop(slot)
        dets = np.zeros((n, max_det), DET_DTYPE)
        counts = np.zeros(n, np.int32)
        total = np.zeros(n, np.int32)
        _check(lib().fd_collect(self._h, slot, _ptr(dets), _ptr(counts), _ptr(total)))
        return dets, counts, total

    # -- parity / profiling hooks
    def heads(self, n: int) -> List[np.ndarray]:
        outs = []
        for i, (c, h, w) in enumerate(self.head_shapes):
            a = np.empty((n, c, h, w), np.float32)
            _check(lib().fd_heads_fp32(self._h, i, _ptr(a), n))
            outs.append(a)
        return outs

    def set_heads(self, heads: Sequence[np.ndarray]):
        n = heads[0].shape[0]
        for i, a in enumerate(heads):
            a = np.ascontiguousarray(a, np.float32)
            assert a.shape == (n,) + self.head_shapes[i], (a.shape, self.head_shapes[i])
            _check(lib().fd_set_heads_fp32(self._h, i, _ptr(a), n))
        return n

    def layer_output(self, layer: int, n: int) -> np.ndarray:
        d = FdLayerDesc()
        _check(lib().fd_layer_info(self._h, layer, C.byref(d)))
        a = np.empty((n, d.c, d.h, d.w), np.float32)
        _check(lib().fd_layer_output_fp32(self._h, layer, _ptr(a), n))
        return a

    def normalise(self, frames: np.ndarray) -> np.ndarray:
        frames = np.ascontiguousarray(frames, np.uint8)
        n = frames.shape[0]
        out = np.empty((n, 3, self.net_h, self.net_w), np.float32)
        _check(lib().fd_normalise_f32(self._h, _ptr(frames), n, _ptr(out)))
        return out

    def letterbox(self, frames: np.ndarray) -> np.ndarray:
        frames = np.ascontiguousarray(frames, np.uint8)
        n, h, w, _ = frames.shape
        out = np.empty((n, self.net_h, self.net_w, 3), np.uint8)
        _check(lib().fd_letterbox_u8(self._h, _ptr(frames), n, w, h, _ptr(out)))
        return out

    def time_layers(self, n: int, reps: int = 5) -> np.ndarray:
        ms = np.zeros(self.info.n_layers, np.float32)
        _check(lib().fd_time_layers(self._h, n, reps, _ptr(ms)))
        return ms


    def time_forward(self, n: int, reps: int = 10) -> float:
        """Device ms of one fd_forward at batch n (captured graph, mean over reps back-to-back runs)."""
        ms = C.c_float()
        _check(lib().fd_time_forward(self._h, n, reps, C.byref(ms)))
        return float(ms.value)


def pack_wire(dets: np.ndarray, reqid: int = 0, msec: int = 0, saturate: bool = False) -> bytes:
    """The reference server's response payload (server/server.py:234-239) for one frame's detections (a DET_DTYPE array,
    already cut to its count).  saturate=False raises struct.error where struct.pack would."""
    import struct
    dets = np.ascontiguousarray(dets, DET_DTYPE)
    buf = np.empty(16 + 10 * len(dets), np.uint8)
    n = C.c_size_t()
    rc = lib().fd_pack_wire(_ptr(dets), len(dets), reqid & 0xFFFFFFFF, msec & 0xFFFFFFFF, int(saturate), _ptr(buf), buf.size, C.byref(n))
    if rc == FD_ERR_ARG and not saturate:
        raise struct.error((lib().fd_last_error() or b"").decode("utf-8", "replace"))
    _check(rc)
    return buf[:n.value].tobytes()


def letterbox_geometry(src_wh, net_wh):
    """(new_w, new_h, off_x, off_y) of the allow_resize letterbox."""
    v = [C.c_int32() for _ in range(4)]
    _check(lib().fd_letterbox_geometry(src_wh[0], src_wh[1], net_wh[0], net_wh[1], *[C.byref(x) for x in v]))
    return tuple(x.value for x in v)


def unmap_letterbox(dets: np.ndarray, src_wh, net_wh) -> np.ndarray:
    """Detections of a letterboxed frame (DET_DTYPE array cut to its count) -> pixels of the source frame."""
    out = np.ascontiguousarray(dets, DET_DTYPE).copy()
    _check(lib().fd_unmap_letterbox(_ptr(out), len(out), src_wh[0], src_wh[1], net_wh[0], net_wh[1]))
    return out


def jpeg_probe(data: bytes) -> FdJpegInfo:
    """Header parse of one JPEG (host only)."""
    info = FdJpegInfo()
    _check(lib().fd_jpeg_probe(C.c_char_p(data), len(data), C.byref(info)))
    return info


def jpeg_coefficients(data: bytes):
    """Entropy-decodes one JPEG on the host: returns (info, [coefficients of component c as int16 [bh, bw, 8, 8]]).
    Raises JpegRefused for streams the device decoder does not take."""
    info = jpeg_probe(data)
    if info.status != FD_JPEG_OK:
        raise JpegRefused(info.reason.decode("utf-8", "replace"), np.array([info.status], np.int32))
    coefs = np.empty(info.coef_count, np.int16)
    rc = lib().fd_jpeg_coefficients(C.c_char_p(data), len(data), _ptr(coefs), coefs.size, C.byref(info))
    if rc == FD_ERR_JPEG:
        raise JpegRefused((lib().fd_last_error() or b"").decode("utf-8", "replace"), np.array([info.status], np.int32))
    _check(rc)
    planes, o = [], 0
    for c in range(3):
        k = info.blocks_w[c] * info.blocks_h[c] * 64
        planes.append(coefs[o:o + k].reshape(info.blocks_h[c], info.blocks_w[c], 8, 8))
        o += k
    return info, planes


def set_option(name: str, value: int) -> None:
    """Plan-time option (csrc/options.h); takes effect for execution state built afterwards."""
    _check(lib().fd_set_option(name.encode(), int(value)))


def get_option(name: str) -> int:
    v = C.c_int()
    _check(lib().fd_get_option(name.encode(), C.byref(v)))
    return v.value


class option:
    """with option("strip", 2): ... — sets an option for the block and restores the previous value."""

    def __init__(self, name, value):
        self.name, self.value = name, value

    def __enter__(self):
        self.old = get_option(self.name)
        set_option(self.name, self.value)
        return self

    def __exit__(self, *exc):
        set_option(self.name, self.old)
        return False


def device_count() -> int:
    return int(lib().fd_device_count())
