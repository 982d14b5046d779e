"""Shared comparison helper for result lists that came through different batch sizes.

A frame's tuples do not depend on the batch it rode in beyond the fp32 re-association the kernel forms of different
batch sizes imply (split-K parts, DESIGN.md §4): same boxes and classes, scores within the spec's 1e-2.  Boxes are matched
by class and position (within 1.5 px), not by rounded coordinates — a coordinate that sits on x.5 must not split a match.

The second half states, once, the rounding model a fused conv layer's output is held to when the oracle is fed the layer's
own inputs (layer_bound / check_layer)."""
import numpy as np
import torch


def same_detections(got, want, threshold, max_unmatched=2, dconf=1e-2, dpix=1.5):
    """got / want: reference-style tuples (klass, conf, x, y, w, h).  Solid boxes only (conf >= threshold + 1e-2): a
    near-threshold one may come or go.  Returns True when all but max_unmatched solid boxes of either side have a partner."""
    g = [t for t in got if t[1] >= threshold + 1e-2]
    w = [t for t in want if t[1] >= threshold + 1e-2]

    def partner(t, pool):
        for u in pool:
            if u[0] == t[0] and abs(u[2] - t[2]) <= dpix and abs(u[3] - t[3]) <= dpix and abs(u[1] - t[1]) <= dconf:
                return True
        return False

    miss_g = sum(not partner(t, want) for t in g)
    miss_w = sum(not partner(t, got) for t in w)
    return miss_g <= max_unmatched and miss_w <= max_unmatched


# ------------------------------------------------------------------ the rounding model of one fused conv layer

U = 2.0 ** -23
"""Error of one fp32 addition, relative to the running magnitude: 2^-23 rather than round-to-nearest's 2^-24, so that an
accumulator that truncates instead of rounding (how tcgen05 adds bf16 products in fp32 is not documented) still meets it.
Measured (tests/test_gpu_layers_exact.py, every row, NVIDIA B200 at its 1000 W power limit): the worst accumulation error,
|g - r| less the rounding allowance, in units of U*S, was 4.40 for tc_single, 3.99 tc_pair, 4.44 tc_pair_strip, 1.47
tc_swapped, 0.96 halo, 0.62 halo+pool, 1.09 block, 0.69 for the unfused kernels the parity hook runs (fused_next), 0.08
conv0+pool; the rule allows K + 4 >= 31 (K = 27 for conv0).  The fused stem's conv2 reaches 401 on the < 0.1 % of its
elements that differ by a step of the recomputed input (RELAXED_EXTRA allows 2^16)."""

RELAXED_SHARE = 0.999
"""Share of elements that must meet the strict bound in a layer that reads a tensor the fused kernel never writes out."""
RELAXED_EXTRA = 2.0 ** -7
"""... and the extra allowance, times S, every element of such a layer gets (one bf16 step of each input of the sum)."""


def bf16_ulp(v):
    """Spacing of bf16 numbers at |v| (bf16 keeps 8 significant bits; below 2^-126 the subnormal spacing 2^-133)."""
    v = np.maximum(np.abs(np.asarray(v, np.float64)), 2.0 ** -126)
    return np.ldexp(1.0, np.frexp(v)[1] - 8)


def layer_bound(g, rec, out_fp32=False, halo_residual=False):
    """Bound on |g - r| for each element of one fused conv layer's output g, given the teacher-forced record `rec` of
    oracle/ref_graph.GraphExecutor.run_forced (computed from the layer's own bf16 inputs).

    Derivation.  The inputs and the weights are bf16, so every product is exact in fp32; K = cin*k*k of them are summed
    with the bias in fp32, in some order.  Each fp32 addition errs by at most U times the magnitude of the running sum,
    which never exceeds S = sum |x*w| + |b|; with the activation (one multiply) and the residual add, at most K + 4
    roundings touch a value, so the fp32 result x differs from the exact r by at most A = U*(K+4)*(S + |res|) (the
    record's S already includes |res|).  The kernel then rounds x to bf16 once: half a bf16 step at |x|, and |x| lies
    between |r| and |g| unless it crossed a power of two, where the step of |g| is the larger one.  Hence
        bf16 output:   |g - r| <= ulp(max(|g|, |r|)) / 2 + A
        fp32 output:   |g - r| <= A
    conv_halo with a residual rounds the branch (the activation's value) to bf16 before its bf16x2 add: + ulp(|branch| + A)/2.
    A fused MaxPool(2, 2) takes the maximum of rounded values; |max g_i - max r_i| is at most the error of the element
    that wins on either side, so the bound is the largest in the window: S is max-pooled, |r| replaced by the window's
    largest |r_i| (+ A, for a winner whose fp32 value crossed a power of two).
    A value computed exactly from the layer's inputs (stand-alone MaxPool, a copy) has bound 0."""
    S = rec["S"]
    if S is None:
        return np.zeros(np.shape(g))
    A = U * (rec["K"] + 4) * np.asarray(S, np.float64)
    if out_fp32:
        return A
    m = np.asarray(rec["m"], np.float64)
    if rec.get("pool"):
        m = m + A
    b = 0.5 * bf16_ulp(np.maximum(np.abs(np.asarray(g, np.float64)), m)) + A
    if halo_residual and "branch" in rec:
        b = b + 0.5 * bf16_ulp(np.abs(np.asarray(rec["branch"], np.float64)) + A)
    return b


def check_layer(g, rec, out_fp32=False, halo_residual=False, relaxed=False):
    """Applies layer_bound.  Returns (ok, stats); stats: worst |g-r|/bound ('ratio', over the elements that must meet the
    strict bound), the share of elements that meet it ('share'), the share of elements that differ from r rounded to the
    output type ('flips'), and the worst accumulation error in units of U*S ('acc': |g-r| less the rounding allowance,
    over U*S — the rule allows K + 4).
    relaxed (the fused stem's conv2 and the fused block's conv4, whose input the parity hook recomputes with the unfused
    kernel, so one-step rounding differences of that input are possible): >= RELAXED_SHARE of the elements meet the strict
    bound and all meet it plus RELAXED_EXTRA * S, which holds if every element of the recomputed input is within one bf16
    step of the fused kernel's internal value (each product then moves by at most 2^-7 |x*w|)."""
    g = np.asarray(g, np.float64)
    r = np.asarray(rec["r"], np.float64)
    err = np.abs(g - r)
    b = layer_bound(g, rec, out_fp32, halo_residual)
    rounded = r.astype(np.float32)
    if not out_fp32:
        rounded = torch.from_numpy(r).to(torch.float32).to(torch.bfloat16).to(torch.float32).numpy()
    stats = {"flips": float(np.mean(g != rounded)), "n": int(g.size)}
    within = err <= b
    stats["share"] = float(np.mean(within))
    with np.errstate(divide="ignore", invalid="ignore"):
        ratio = np.where(b > 0, err / b, np.where(err > 0, np.inf, 0.0))
        if rec["S"] is not None:
            S = np.asarray(rec["S"], np.float64)
            rnd = np.zeros_like(b) if out_fp32 else b - U * (rec["K"] + 4) * S
            acc = np.where(S > 0, np.maximum(err - rnd, 0.0) / (U * S), 0.0)
            stats["acc"] = float(acc.max()) if acc.size else 0.0
        else:
            stats["acc"] = 0.0
    stats["ratio"] = float(ratio.max()) if ratio.size else 0.0
    if relaxed:
        loose = b + RELAXED_EXTRA * np.asarray(rec.get("S_branch", rec["S"]), np.float64)
        stats["loose_ratio"] = float((err / loose).max()) if err.size else 0.0
        ok = stats["share"] >= RELAXED_SHARE and bool((err <= loose).all())
    else:
        ok = bool(within.all())
    return ok, stats
