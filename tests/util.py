"""Shared helpers for the parity tests (test infrastructure)."""
import os
import random

import numpy as np

from qrack_b200 import qscript

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")

# north_star tolerances: max |delta amplitude| vs QEngineCPU on identical circuits
AMP_TOL = {32: 1e-6, 64: 1e-12}
# scalar queries (probabilities, norms) are fp reductions with unspecified order.  The oracle restatement sums |amp|^2
# into ONE fp32 accumulator (the reference does that per worker thread, state.cpp:1751-1810), which by itself drifts by up
# to ~6e-6 at 2^10..2^13 terms (measured: 0.647028148 vs 0.647021766 exact for an 11-qubit state), while the CUDA
# reductions accumulate in double.  The amplitude bar (AMP_TOL) is the parity criterion; this one only has to absorb the
# oracle's own summation drift.
PROB_TOL = {32: 5e-6, 64: 1e-12}


def golden_names():
    return sorted(f[:-3] for f in os.listdir(GOLDEN) if f.endswith(".qs"))


def load_golden(name, prec):
    text = open(os.path.join(GOLDEN, name + ".qs")).read()
    z = np.load(os.path.join(GOLDEN, "%s.f%d.npz" % (name, prec)))
    regs = {int(k[3:]): z[k] for k in z.files if k.startswith("reg")}
    results = qscript.parse_results(str(z["results"]))
    return text, regs, results


def load_reference(name):
    """Stored outputs of the compiled reference (tests/golden/reference, written by make_golden.py): the script "text" and
    either a seeded sample of register 0's final amplitudes ("idx", "amp") or the query results ("results", and "results_f64"
    from the fp64 build for fp32 cases)."""
    z = np.load(os.path.join(GOLDEN, "reference", name + ".npz"))
    return {k: (str(z[k]) if z[k].dtype.kind == "U" else z[k]) for k in z.files}


def assert_sample_close(state, ref, prec, what=""):
    """register 0's state against the reference's stored amplitude sample"""
    assert state.size > int(ref["idx"].max()), (what, state.size)
    d = float(np.abs(state[ref["idx"]].astype(np.complex128) - ref["amp"].astype(np.complex128)).max())
    assert d <= AMP_TOL[prec], "%s: max |delta amp| over %d sampled amplitudes = %.3e > %.1e" % (what, ref["idx"].size, d, AMP_TOL[prec])


def ref_harness(prec):
    p = os.path.join(ROOT, "oracle", "_ref", "ref_harness_f%d" % prec)
    return p if os.path.exists(p) else None


def make_factory(cls, prec, **kw):
    def make(n, perm):
        return cls(n, perm, random.Random(1), 1.0 + 0j, False, False, precision=prec, **kw)
    return make


def run_engine(text, cls, prec, **kw):
    regs, results = qscript.run(text, make_factory(cls, prec, **kw))
    return {k: v.GetQuantumState() for k, v in regs.items()}, results


def assert_states_close(got, want, prec, what=""):
    assert set(got.keys()) == set(want.keys()), (what, got.keys(), want.keys())
    for k in want:
        assert got[k].shape == want[k].shape, (what, k, got[k].shape, want[k].shape)
        d = float(np.abs(got[k].astype(np.complex128) - want[k].astype(np.complex128)).max()) if want[k].size else 0.0
        assert d <= AMP_TOL[prec], "%s reg %d: max |delta amp| = %.3e > %.1e" % (what, k, d, AMP_TOL[prec])


def assert_results_close(got, want, prec, what=""):
    assert len(got) == len(want), (what, len(got), len(want))
    for i, ((gn, gv), (wn, wv)) in enumerate(zip(got, want)):
        assert gn == wn, (what, i, gn, wn)
        for a, b in zip(gv, wv):
            assert abs(a - b) <= PROB_TOL[prec], "%s result %d (%s): %r vs %r" % (what, i, gn, a, b)
