"""The rounding model of tests/compare.py for a fused convolution whose activation is Mish.

tests/mish_oracle.py tags the teacher-forced record of every value a Mish is fused into with rec["act"] = "mish".  For
such a record the fp32 error of the pre-activation, U (K + 4) S, grows by at most MISH_SLOPE through the Mish, and the
device's formula adds its own error, relative to the Mish's value (the branch value before a residual Add, or |g|, |r|):
    bf16 output:   |g - r| <= ulp(max(|g|, |r|)) / 2 + MISH_SLOPE * U (K + 4) S + MISH_C * U * max(|g|, |r|, |branch|)
check_layer applies it by handing compare.check_layer the record with S replaced by the S that makes its U (K + 4) S equal
to the last two terms; a record without the tag goes to compare.check_layer unchanged."""
import numpy as np

from tests import compare
from tests.compare import U

MISH_SLOPE = 1.09
"""max |mish'(x)| = 1.0885 (at x = 1.19): how much an error of the fp32 pre-activation can grow through Mish."""
MISH_C = 6.0
"""Relative error, in units of U, of the device's Mish (fastdet_b200/csrc/act.cuh) against the exact Mish of its fp32 input:
ex2.approx (PTX ISA: 2 ulp) 2, n = e (e + 2) 1, d = n + 2 1/2, the Newton reciprocal 3/2, the products x * (n * r) 1.  The
rounding of x * log2(e) changes x by a relative 2^-24: one more rounding of the pre-activation, inside the K + 4."""


def mish_record(g, rec):
    """rec with S such that U (K + 4) S = MISH_SLOPE * U (K + 4) S + MISH_C * U * max(|g|, |r|, |branch|)."""
    if rec.get("act") != "mish" or rec["S"] is None:
        return rec
    m = np.maximum(np.abs(np.asarray(g, np.float64)), np.asarray(rec["m"], np.float64))
    if "branch" in rec:
        m = np.maximum(m, np.abs(np.asarray(rec["branch"], np.float64)))
    S = MISH_SLOPE * np.asarray(rec["S"], np.float64) + MISH_C * m / (rec["K"] + 4)
    return dict(rec, S=S)


def check_layer(g, rec, out_fp32=False, halo_residual=False, relaxed=False):
    """compare.check_layer with the Mish form of the bound for records tagged Mish (stats['acc'] is then in units of U
    times the effective S)."""
    return compare.check_layer(g, mish_record(g, rec), out_fp32, halo_residual, relaxed)
