"""The per-layer rounding model (tests/compare.py: layer_bound / check_layer) on the CPU: it accepts every fp32 summation
order a conv kernel may use and rejects the local bugs a new tiling or kernel form tends to bring, each on its own; and
the teacher-forced oracle (GraphExecutor.run_forced) that supplies its reference reproduces the plain float64 oracle.

The layer: 3x3 conv, 32 -> 64 channels over a 15x15 map (225 output positions: one full 128-row tile and a partial
one), bf16 inputs in [-1, 1), bf16 weights in [-2^-6, 2^-6), fp32 bias in [-0.5, 0.5), LeakyReLU(0.1) and a bf16 residual;
K = 288.  A dropped product moves a sum by less than 2^-6, inside the old per-element tolerance of 2e-2 + 1e-2 |v|."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from fastdet_b200 import modelgen
from oracle import ref_graph, ref_post
from tests.compare import U, check_layer

H = W = 15
CIN, COUT, KS = 32, 64, 3
K = CIN * KS * KS
TILE_M, BLOCK_K = 128, 64


def _bf16(a):
    return torch.from_numpy(np.ascontiguousarray(a, np.float32)).to(torch.bfloat16).to(torch.float32).numpy()


@pytest.fixture(scope="module")
def layer():
    rng = np.random.default_rng(7)
    x = _bf16(rng.uniform(-1, 1, (CIN, H, W)))
    w = _bf16(rng.uniform(-2.0 ** -6, 2.0 ** -6, (COUT, CIN, KS, KS)))  # every product below 2^-6: a dropped one is small
    b = rng.uniform(-0.5, 0.5, COUT).astype(np.float32)
    res = _bf16(rng.uniform(-1, 1, (COUT, H, W)))
    # im2col in the kernels' K order (tap-major, channel-minor): X[m, (r*3 + s)*CIN + c]
    xp = np.pad(x, ((0, 0), (1, 1), (1, 1)))
    cols = np.zeros((H * W, K), np.float32)
    for r in range(KS):
        for s in range(KS):
            cols[:, (r * KS + s) * CIN:(r * KS + s + 1) * CIN] = xp[:, r:r + H, s:s + W].reshape(CIN, -1).T
    wk = np.ascontiguousarray(w.transpose(0, 2, 3, 1).reshape(COUT, K).T)  # [K, COUT]
    # the reference: exact sum (float64), bias, activation, residual; S = sum |x w| + |b| + |res|
    acc = torch.from_numpy(cols).double() @ torch.from_numpy(wk).double() + torch.from_numpy(b).double()
    branch = F.leaky_relu(acc, float(np.float32(0.1)))
    resm = torch.from_numpy(res.reshape(COUT, -1).T.copy()).double()
    r = (branch + resm).numpy()
    Sb = (torch.from_numpy(np.abs(cols)).double() @ torch.from_numpy(np.abs(wk)).double() + torch.from_numpy(np.abs(b)).double()).numpy()
    rec = {"r": r, "S": Sb + np.abs(resm.numpy()), "K": K, "m": np.abs(r), "pool": False, "branch": branch.numpy(), "S_branch": Sb}
    return {"cols": cols, "wk": wk, "b": b, "res": resm.numpy().astype(np.float32), "rec": rec}


def _epilogue(acc32, L, bias=None):
    """fp32 bias + LeakyReLU + residual, one rounding to bf16 (what conv_tc's epilogue does)."""
    v = acc32 + (L["b"] if bias is None else bias)
    v = np.where(v > 0, v, v * np.float32(0.1)).astype(np.float32)
    return _bf16(v + L["res"])


def _tiled(cols, L, parts=1, double_part=None):
    """The tcgen05 kernels' order: per 128-row tile, K in 64-wide blocks accumulated into fp32; with `parts`, the K blocks
    are split into that many contiguous parts (split-K), each summed on its own and the parts added in part order.
    double_part: this part is added twice in the first tile (a split-K part counted twice)."""
    wk = L["wk"]
    kbs = [slice(k, min(k + BLOCK_K, K)) for k in range(0, K, BLOCK_K)]
    bounds = np.linspace(0, len(kbs), parts + 1).round().astype(int)
    out = np.zeros((cols.shape[0], COUT), np.float32)
    for m0 in range(0, cols.shape[0], TILE_M):
        tile = slice(m0, m0 + TILE_M)
        total = np.zeros((min(TILE_M, cols.shape[0] - m0), COUT), np.float32)
        for p in range(parts):
            part = np.zeros_like(total)
            for kb in kbs[bounds[p]:bounds[p + 1]]:
                part = (part + cols[tile, kb] @ wk[kb]).astype(np.float32)
            total = (total + part).astype(np.float32)
            if p == double_part and m0 == 0:
                total = (total + part).astype(np.float32)
        out[tile] = total
    return out


def _ok(g, L):
    return check_layer(g, L["rec"])[0]


# ------------------------------------------------------------------ what a correct kernel may do
def test_summation_orders_pass(layer):
    L = layer
    cols, wk = L["cols"], L["wk"]
    fwd = np.zeros((cols.shape[0], COUT), np.float32)
    for k in range(K):  # one product at a time, K ascending
        fwd = (fwd + cols[:, k:k + 1] * wk[k:k + 1]).astype(np.float32)
    rev = np.zeros_like(fwd)
    for k in reversed(range(K)):  # and descending
        rev = (rev + cols[:, k:k + 1] * wk[k:k + 1]).astype(np.float32)
    for acc in (fwd, rev, _tiled(cols, L), _tiled(cols, L, parts=3)):
        ok, st = check_layer(_epilogue(acc, L), L["rec"])
        assert ok, st
        assert st["acc"] <= K + 4
    # the fp32 output rule: no rounding allowance
    v = (fwd + L["b"]).astype(np.float32)
    acc = (torch.from_numpy(cols).double() @ torch.from_numpy(wk).double()).numpy() + L["b"]
    S = L["rec"]["S_branch"]
    ok, st = check_layer(v, {"r": acc, "S": S, "K": K, "m": np.abs(acc), "pool": False}, out_fp32=True)
    assert ok and st["flips"] > 0, st
    # conv_halo's residual form: the branch rounded to bf16 first, then a bf16 add rounded once
    br = (fwd + L["b"]).astype(np.float32)
    br = _bf16(np.where(br > 0, br, br * np.float32(0.1)))
    g = _bf16(br + L["res"])
    assert check_layer(g, L["rec"], halo_residual=True)[0]


def test_teacher_forced_oracle_reproduces_the_float64_oracle():
    """Fed its own bf16 values, run_forced predicts every stored activation of the plain dtype="bf16", accumulate=float64
    run bit for bit once rounded, and its heads exactly."""
    for arch, nc, size in (("tiny", 3, 96), ("full", 4, 64)):
        data = modelgen.build_onnx(arch, nc, size, seed=5)
        exe = ref_graph.GraphExecutor(data, dtype="bf16", accumulate=torch.float64)
        x = ref_post.normalise(modelgen.synthetic_frame(200, size))
        plain = exe.run(x, all_values=True)
        names = sorted(exe.round_after) + list(exe.graph.outputs)
        recs = exe.run_forced(x, {k: plain[k] for k in names})
        assert sorted(recs) == sorted(names)
        for k in names:
            r = recs[k]["r"]
            got = _bf16(r.numpy()) if k in exe.round_after else r.float().numpy()
            assert np.array_equal(got, plain[k]), k
        # S: the magnitude of a convolution's sums bounds |r| and carries the residual
        for k, rec in recs.items():
            if rec["S"] is not None:
                assert (rec["S"] >= rec["r"].abs() * (1 - 1e-6)).all() and rec["K"] > 0, k


# ------------------------------------------------------------------ bugs the bound must catch, each on its own
def _bug(layer, which):
    L = layer
    cols = L["cols"].copy()
    if which == "dropped channel":  # channel 5 of tap (1, 2) left out of the first 128-row tile
        cols[:TILE_M, 5 * CIN + 5] = 0
        return _epilogue(_tiled(cols, L), L)
    if which == "rows shifted":  # the second tile's rows written one pixel late
        g = _epilogue(_tiled(cols, L), L)
        g[TILE_M + 1:] = g[TILE_M:-1].copy()
        return g
    if which == "last tile unwritten":  # the partial last tile (rows 128..224) never stored: the buffer keeps zeros
        g = _epilogue(_tiled(cols, L), L)
        g[TILE_M:] = 0
        return g
    if which == "strip pad column":  # row 6's last pixel: the right-hand taps read the next row's first pixel, not the pad
        m = 6 * W + (W - 1)
        for r in range(KS):
            tap = r * KS + 2                  # reads input (6 + r - 1, W): the pad column
            src = (6 + r) * W                 # input (6 + r, 0) is what the centre tap (4) of output pixel (6 + r, 0) reads
            cols[m, tap * CIN:(tap + 1) * CIN] = L["cols"][src, 4 * CIN:5 * CIN]
        return _epilogue(_tiled(cols, L), L)
    if which == "residual twice":  # one pixel
        acc = _tiled(cols, L)
        g = _epilogue(acc, L)
        v = acc[100] + L["b"]
        v = np.where(v > 0, v, v * np.float32(0.1)).astype(np.float32)
        g[100] = _bf16(v + L["res"][100] + L["res"][100])
        return g
    if which == "split-K part twice":  # part 1 of 3 added twice on the first tile
        return _epilogue(_tiled(cols, L, parts=3, double_part=1), L)
    if which == "bias off 1 %":  # the channel with the largest bias
        b = L["b"].copy()
        c = int(np.argmax(np.abs(b)))
        b[c] *= np.float32(1.01)
        return _epilogue(_tiled(cols, L), L, bias=b)
    raise KeyError(which)


BUGS = ["dropped channel", "rows shifted", "last tile unwritten", "strip pad column", "residual twice", "split-K part twice",
        "bias off 1 %"]


@pytest.mark.parametrize("which", BUGS)
def test_local_bug_fails(layer, which):
    g = _bug(layer, which)
    ok, st = check_layer(g, layer["rec"])
    assert not ok, (which, st)
    # the same output with the bug undone passes: the failure is the bug's, not the simulation's
    assert _ok(_epilogue(_tiled(layer["cols"], layer), layer), layer)

