"""Every layer's output against a float64 prediction from that layer's OWN GPU inputs, at every batch bucket (-m gpu).

The checks of tests/test_gpu_parity.py compare against the fp32 oracle's own chain, whose input to layer i already differs from
the GPU's by the bf16 noise of every earlier layer, so they have to be statistical (RMS per layer, 2e-2 of max|ref| at the
heads) and miss a local bug: one wrong pixel of a 52x52 layer at batch 8 moves the RMS ratio by about 1e-2.  Here the oracle is
teacher-forced (oracle/ref_graph.GraphExecutor.run_forced): every fused layer is evaluated in float64 on the bf16 tensors the
GPU's layer actually read (fetched with Model.layer_output), and each output element is held to the rounding model of
tests/compare.py — half a bf16 step plus U*(K+4)*S of fp32 summation — which any dropped product, shifted tile, unwritten
partial tile, wrong pad read or doubled split-K part exceeds.

The matrix runs each batch-size bucket (power of two, execution state is built per bucket) and the paths that only some
buckets take; test_matrix_covers_every_kernel_form asserts, through fd_layer_exec_info, that the rows together still run every
kernel form, so a planner change that moves a form out of the matrix fails there.  Rows on non-square nets (416x256 and its
transpose, 640x384, 320x192, 96x160) catch what a square map hides — a swapped height and width, a row pitch or a tile count
taken from the wrong axis — and test_nonsquare_rows_cover_every_kernel_form asserts that they alone run every form.  Each row
prints one line per layer:
index, name, kernel form, block_n, split_k, K, the worst ratio of |g - r| to the bound, the share of elements that differ from
r rounded to the output type, and the worst fp32 accumulation error in units of U*S (the model allows K + 4)."""
import numpy as np
import pytest
import torch

from fastdet_b200 import _native, modelgen
from oracle import onnx_min, ref_graph, ref_post
from tests.compare import check_layer
from tests.test_gpu_parity import frames_for

pytestmark = pytest.mark.gpu

THR = 0.1

# id: (arch, classes, net (w, h), options, batch, path, checked frames (None: all))
ROWS = {
    "full416-n1": ("full", 80, (416, 416), {}, 1, "forward", None),     # 64-wide latency tiles; split-K on 13x13 (+ residual) and 26x26
    "full416-n2": ("full", 80, (416, 416), {}, 2, "forward", None),     # split-K into 3 parts
    "full416-n3": ("full", 80, (416, 416), {}, 3, "forward", None),     # bucket 4 with a stale frame
    "full416-n8": ("full", 80, (416, 416), {}, 8, "forward", [0, 1, 4, 7]),      # 128-wide latency tiles; 52x52 strips
    "full416-n13": ("full", 80, (416, 416), {}, 13, "forward", [0, 1, 7, 12]),   # bucket 16: the CTA pair in im2col form on 13x13 3x3
    "full416-n20": ("full", 80, (416, 416), {}, 20, "detect", [0, 7, 8, 16, 19]),  # bucket 32: copy-overlapped quarter front
    "full416-n64": ("full", 80, (416, 416), {}, 64, "forward", [0, 1, 32, 63]),  # the benchmarked configuration
    "full416-strip-n2": ("full", 80, (416, 416), {"strip": 2}, 2, "forward", None),  # strips at widths 27 / 14
    "full608-n1": ("full", 80, (608, 608), {}, 1, "forward", None),
    "full608-n4": ("full", 80, (608, 608), {}, 4, "forward", [0, 3]),   # 76x76 strips
    "full608-n32": ("full", 80, (608, 608), {}, 32, "forward", [0, 31]),  # a per-GPU shard of the 2-GPU 608 configuration
    "rsu416-n64": ("rsu", 9, (416, 416), {}, 64, "forward", [0, 63]),   # 42-channel heads in 44-wide rows
    "tiny416-n1": ("tiny", 80, (416, 416), {}, 1, "forward", None),     # conv0_ws and halo with fused pool, stand-alone maxpool
    "tiny416-n5": ("tiny", 80, (416, 416), {}, 5, "forward", [0, 4]),
    # Non-square and off-grid nets: on a square map a kernel that swaps height and width, takes a row pitch or a tile count
    # from the wrong axis, or decomposes a pixel index in the wrong order still gives the right answer.
    "full416x256-n1": ("full", 80, (416, 256), {}, 1, "forward", None),   # split-K on 13x8 and 26x16, latency tiles, stem/block on 208x128
    "full256x416-n3": ("full", 80, (256, 416), {}, 3, "forward", [0, 2]),  # the same net transposed: an axis swap fails one of the two
    "full640x384-n8": ("full", 80, (640, 384), {}, 8, "forward", [0, 7]),  # 80x48 maps in the strip form, 20x12 heads
    "full416x256-n20": ("full", 80, (416, 256), {}, 20, "detect", [0, 8, 16, 19]),  # quarter-batch front and copy pieces, non-square
    "rsu320x192-n64": ("rsu", 9, (320, 192), {}, 64, "forward", [0, 63]),  # the batch-64 plan on a 6x10 grid; 42-channel heads
    "tiny416x256-n5": ("tiny", 80, (416, 256), {}, 5, "forward", [0, 4]),  # conv0_ws / halo with fused pool, stride-1 maxpool on 8x13
    "full96x160-n2": ("full", 80, (96, 160), {}, 2, "forward", None),     # too small for the stem: conv0 on the full graph, heads 3 wide and 5 tall
}
SEED = {"full": 2, "rsu": 3, "tiny": 1}

_models = {}


@pytest.fixture(scope="module", autouse=True)
def _release_models():
    """The models of this module hold device buffers for every bucket they ran: free them before the next module runs."""
    yield
    for _, m in _models.values():
        m.close()
    _models.clear()


def _model(arch, nc, wh, opts):
    """One Model per (graph, net, options); options apply to execution state built while they are set, so every use of a
    model with options runs inside the same option block.  A non-square net runs the graph generated at 416 (the planner
    builds every layer from the net's (w, h), whatever input shape the graph declares)."""
    key = (arch, nc, wh, tuple(sorted(opts.items())))
    if key not in _models:
        data = modelgen.build_onnx(arch, nc, wh[0] if wh[0] == wh[1] else 416, SEED[arch])
        _models[key] = (data, _native.Model(data, nc, wh, device=0))
    return _models[key]


class _options:
    def __init__(self, opts):
        self.blocks = [_native.option(k, v) for k, v in opts.items()]

    def __enter__(self):
        for b in self.blocks:
            b.__enter__()

    def __exit__(self, *exc):
        for b in reversed(self.blocks):
            b.__exit__(*exc)
        return False


def _pooled(data):
    """Output names of the layers that end in a MaxPool (a fused pool when the layer is a convolution)."""
    return {n.outputs[0] for n in onnx_min.load(data).nodes if n.op == "MaxPool"}


def _form(l, e, pooled):
    return e["kernel_name"] + ("+pool" if l["kind"] != 2 and l["out_name"] in pooled else "")


def _records(m, n):
    m.postprocess(n, THR, max_det=512)
    dets, counts, _ = m.fetch(n)
    return [dets[f, :counts[f]].copy() for f in range(n)]


def _front_layers(L, pooled, net_h):
    """Layers fd_detect runs quarter batch by quarter batch behind the pieces of its frame copy (build_overlap_plan in
    capi.cu): those in front of the second down-sampling layer."""
    downs, prev_h = 0, net_h
    for i, l in enumerate(L):
        if l["stride"] == 2 or l["out_name"] in pooled or l["h"] < prev_h:
            downs += 1
            if downs == 2:
                return set(range(i))
        prev_h = l["h"]
    return set()


def _run_path(m, frames, path):
    """Runs the batch through `path`; returns the detection records of the "detect" path (None for "forward")."""
    n, wh = frames.shape[0], (frames.shape[2], frames.shape[1])
    if path == "forward":
        m.preprocess(frames, n, wh)
        m.forward(n)
        return None
    # "detect": the synchronous call (frame copy in pieces overlapped with the first layers, quarter batch by quarter batch).
    # The bucket's buffers first hold a pass over OTHER frames, so a quarter, a piece of the copy or a partial last quarter
    # that the call leaves unwritten shows up as a wrong layer instead of as the right value left behind
    other = frames_for(n, wh, first_seed=900)
    m.preprocess(other, n, wh)
    m.forward(n)
    dets, counts = m.detect(frames, THR, max_det=512)
    return [dets[f, :counts[f]].copy() for f in range(n)]


def check_layers_exact(data, m, frames, picks, label, front=frozenset()):
    """Runs the teacher-forced oracle on frames `picks` of the batch the model last ran and applies the rounding model to every
    layer.  Returns {kernel form: (worst ratio, flip share, worst accumulation error / (U*S), elements)}.
    front: layers that ran as quarter-batch launches (fd_detect); fd_layer_exec_info describes the whole-batch launches, so
    their printed form, block_n and split_k are marked as such ("q")."""
    n = frames.shape[0]
    L = m.layers()
    info = m.exec_info(n)
    outs = {}
    for i, l in enumerate(L):  # one layer at a time, only the checked frames kept (conv1 of 64 frames at 608 is 3 GB in fp32)
        a = m.layer_output(i, n)
        sel = np.ascontiguousarray(a[picks])
        del a
        outs[l["out_name"]] = sel if l["out_fp32"] else torch.from_numpy(sel).to(torch.bfloat16)
    index = {l["out_name"]: i for i, l in enumerate(L)}
    pooled = _pooled(data)
    exe = ref_graph.GraphExecutor(data, dtype="bf16")
    worst = {}
    failures = []
    for j, f in enumerate(picks):
        x = ref_post.normalise(frames[f])
        over = {k: (v[j:j + 1] if isinstance(v, np.ndarray) else v[j:j + 1].float().numpy()) for k, v in outs.items()}

        def on_value(name, rec, f=f, j=j):
            i = index[name]
            l, e = L[i], info[i]
            form = e["kernel_name"]
            ok, st = check_layer(over[name], rec, out_fp32=bool(l["out_fp32"]),
                                 halo_residual=form == "halo" and bool(l["has_residual"]), relaxed=form in ("stem", "block"))
            w = worst.setdefault(i, [0.0, 0, 0, 0.0])
            w[0] = max(w[0], st["ratio"])
            w[1] += st["flips"] * st["n"]
            w[2] += st["n"]
            w[3] = max(w[3], st["acc"])
            if not ok:
                failures.append((i, l["name"], form, f, st))

        exe.run_forced(x, over, on_value=on_value)
    missing = [i for i in range(len(L)) if i not in worst]
    assert not missing, ("layers the oracle never produced", missing)
    by_form = {}
    print(f"\n{label}: bucket {info[0]['bucket']}, frames {list(picks)}"
          + (f"; layers {sorted(front)} ran as quarter-batch launches (q: form of the whole-batch set shown)" if front else ""))
    for i in range(len(L)):
        l, e = L[i], info[i]
        ratio, flips, cnt, acc = worst[i]
        form = _form(l, e, pooled)
        K = l["cin"] * l["ksize"] ** 2
        print(f"  {i:3d}{'q' if i in front else ' '}{l['name']:<10} {form:<14} bn={e['block_n']:<4} sk={e['split_k']:<2} K={K:<5} "
              f"worst/bound={ratio:.3f} flips={flips / cnt:.4f} acc/(U*S)={acc:.2f}")
        b = by_form.setdefault(form, [0.0, 0, 0, 0.0])
        b[0] = max(b[0], ratio)
        b[1] += flips
        b[2] += cnt
        b[3] = max(b[3], acc)
    for form, (ratio, flips, cnt, acc) in sorted(by_form.items()):
        print(f"  form {form:<14} worst/bound={ratio:.3f} flips={flips / cnt:.4f} acc/(U*S)={acc:.2f} elements={cnt}")
    assert not failures, failures[:5]
    return by_form


@pytest.mark.parametrize("row", list(ROWS))
def test_layers_exact(row):
    arch, nc, wh, opts, n, path, picks = ROWS[row]
    picks = list(range(n)) if picks is None else picks
    frames = frames_for(n, wh, first_seed=700)
    with _options(opts):
        data, m = _model(arch, nc, wh, opts)
        records = _run_path(m, frames, path)
        front = _front_layers(m.layers(), _pooled(data), wh[1]) if path == "detect" else frozenset()
        check_layers_exact(data, m, frames, picks, row, front)
        if records is not None:  # the staged path on the same frames returns the very same records
            m.preprocess(frames, n, wh)
            m.forward(n)
            staged = _records(m, n)
            for f in range(n):
                assert np.array_equal(records[f], staged[f]), f


REQUIRED_FORMS = {"fused_next", "stem", "block", "halo", "halo+pool", "conv0+pool", "maxpool", "tc_pair", "tc_pair_strip", "tc_swapped"}


def _forms(rows):
    """Kernel forms the rows run: (forms, block_n of the single-CTA launches, whether each split-K layer has a residual)."""
    seen, single_bn, split = set(), set(), set()
    for row, (arch, nc, wh, opts, n, path, picks) in rows.items():
        with _options(opts):
            data, m = _model(arch, nc, wh, opts)
            L, pooled = m.layers(), _pooled(data)
            for i, e in enumerate(m.exec_info(n)):
                name = e["kernel_name"]
                seen.add(_form(L[i], e, pooled))
                if name == "tc_single":
                    single_bn.add(e["block_n"])
                if e["split_k"] > 1:
                    split.add(bool(L[i]["has_residual"]))
    return seen, single_bn, split


def test_matrix_covers_every_kernel_form():
    """The rows of ROWS together run every kernel form: the fused stem and block, halo with and without a fused pool, conv0
    (YOLOv3-tiny's, with its fused pool; YOLOv3's first layer runs inside the stem), the stand-alone maxpool, conv_tc
    single-CTA with block_n 64 and 128, the CTA pair in im2col and strip form, the swapped form, and split-K on a layer with a
    residual and on one without."""
    seen, single_bn, split = _forms(ROWS)
    assert REQUIRED_FORMS <= seen, sorted(REQUIRED_FORMS - seen)
    assert {64, 128} <= single_bn, single_bn
    assert split == {True, False}, split


def test_nonsquare_rows_cover_every_kernel_form():
    """The rows whose net has w != h on their own run every kernel form, so each form meets a map where a swapped height
    and width would show."""
    seen, single_bn, split = _forms({k: r for k, r in ROWS.items() if r[2][0] != r[2][1]})
    assert REQUIRED_FORMS <= seen, sorted(REQUIRED_FORMS - seen)
    assert {64, 128} <= single_bn, single_bn
    assert split == {True, False}, split
