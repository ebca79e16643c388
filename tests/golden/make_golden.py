"""Generate the committed golden fixtures from the UNMODIFIED reference (oracle/_ref/ref_harness_f{32,64}, i.e.
Qrack::QEngineCPU compiled from the reference sources by oracle/Makefile, REF=<reference checkout>):

    make -C oracle ref && python tests/golden/make_golden.py
    python tests/golden/make_golden.py reference [case ...]     # only the sampled outputs under reference/

Each fixture = <name>.qs (the script) + <name>.f32.npz / <name>.f64.npz (final state of every register and the
query results, as produced by the reference).  Scripts are deterministic (seeded python RNG).
"""
import math
import os
import random
import subprocess
import sys
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
from qrack_b200 import qscript  # noqa: E402


def misc_gates(n=8, seed=3):
    rng = random.Random(seed)
    L = ["qubits %d" % n]
    for q in range(n):
        L.append("H %d" % q)

    def rq(k=1):
        return rng.sample(range(n), k)

    def cx():
        a = rng.uniform(0, 2 * math.pi)
        return "%.17g %.17g" % (math.cos(a), math.sin(a))

    def unitary():
        th, ph, la = (rng.uniform(-math.pi, math.pi) for _ in range(3))
        c, s = math.cos(th / 2), math.sin(th / 2)
        m = [c, -s * complex(math.cos(la), math.sin(la)), s * complex(math.cos(ph), math.sin(ph)),
             c * complex(math.cos(ph + la), math.sin(ph + la))]
        return " ".join("%.17g %.17g" % (complex(z).real, complex(z).imag) for z in m)

    for rep in range(3):
        for g in ("X", "Y", "Z", "S", "IS", "T", "IT", "SqrtX", "H"):
            L.append("%s %d" % (g, rq()[0]))
        for g in ("CNOT", "AntiCNOT", "CZ", "CY", "Swap", "ISwap", "SqrtSwap"):
            a, b = rq(2)
            L.append("%s %d %d" % (g, a, b))
        a, b, c = rq(3)
        L.append("CCNOT %d %d %d" % (a, b, c))
        a, b = rq(2)
        L.append("FSim %.17g %.17g %d %d" % (rng.uniform(-3, 3), rng.uniform(-3, 3), a, b))
        a, b, c, d = rq(4)
        L.append("CSwap 2 %d %d %d %d" % (a, b, c, d))
        L.append("AntiCSwap 1 %d %d %d" % (a, c, d))
        L.append("U %d %.17g %.17g %.17g" % (rq()[0], rng.uniform(-3, 3), rng.uniform(-3, 3), rng.uniform(-3, 3)))
        L.append("AI %d %.17g %.17g" % (rq()[0], rng.uniform(-3, 3), rng.uniform(-3, 3)))
        L.append("IAI %d %.17g %.17g" % (rq()[0], rng.uniform(-3, 3), rng.uniform(-3, 3)))
        L.append("Phase %d %s %s" % (rq()[0], cx(), cx()))
        L.append("Invert %d %s %s" % (rq()[0], cx(), cx()))
        L.append("Mtrx %d %s" % (rq()[0], unitary()))
        a, b, c = rq(3)
        L.append("MCMtrx 2 %d %d %d %s" % (a, b, c, unitary()))
        L.append("MACMtrx 2 %d %d %d %s" % (b, c, a, unitary()))
        L.append("UCMtrx 2 %d %d %d %d %s" % (a, c, b, rng.randrange(4), unitary()))
        L.append("MCPhase 1 %d %d %s %s" % (a, b, cx(), cx()))
        L.append("MACPhase 2 %d %d %d %s %s" % (a, b, c, cx(), cx()))
        L.append("MCInvert 2 %d %d %d %s %s" % (c, b, a, cx(), cx()))
        L.append("MACInvert 1 %d %d %s %s" % (c, a, cx(), cx()))
        L.append("PhaseRootN %d %d" % (rng.randrange(1, 6), rq()[0]))
        a, b = rq(2)
        L.append("CPhaseRootN %d %d %d" % (rng.randrange(1, 6), a, b))
        L.append("XMask %d" % rng.randrange(1, 1 << n))
        L.append("ZMask %d" % rng.randrange(1, 1 << n))
        L.append("PhaseParity %.17g %d" % (rng.uniform(-3, 3), rng.randrange(1, 1 << n)))
        L.append("PhaseRootNMask %d %d" % (rng.randrange(1, 5), rng.randrange(1, 1 << n)))
        L.append("ZeroPhaseFlip %d %d" % (1, n - 2))
        L.append("INC %d 1 %d" % (rng.randrange(1, 30), n - 2))
        L.append("DEC %d 0 %d" % (rng.randrange(1, 30), n - 1))
    for q in range(n):
        L.append("Prob %d" % q)
    L.append("ProbAll 5")
    L.append("ProbReg 2 3 5")
    L.append("ProbMask 37 33")
    L.append("ProbParity 77")
    L.append("CProb 1 4")
    L.append("ACProb 2 6")
    L.append("GetAmplitude 9")
    L.append("Norm")
    return "\n".join(L) + "\n"


def structure(seed=9):
    """Compose / Decompose / Dispose / Allocate / ForceM on separable blocks (SURVEY C1d)."""
    rng = random.Random(seed)
    L = ["qubits 5", "reg 1 3 5", "reg 2 2 0"]

    def local_layer(reg, n):
        for q in range(n):
            L.append("@%d U %d %.17g %.17g %.17g" % (reg, q, rng.uniform(-3, 3), rng.uniform(-3, 3), rng.uniform(-3, 3)))
        for a, b in qscript.random_matching(rng, n):
            L.append("@%d CNOT %d %d" % (reg, a, b))

    for _ in range(3):
        local_layer(0, 5)
        local_layer(1, 3)
        local_layer(2, 2)
    L.append("Compose 1")          # reg0: 8 qubits = [0..4]=A, [5..7]=B
    L.append("Compose 2 2")        # insert C at 2: [0,1]=A, [2,3]=C, [4..6]=A, [7..9]=B
    for q in range(10):
        L.append("Prob %d" % q)
    L.append("ProbMask 771 513")
    # gates inside the blocks only, keeps separability
    L.append("U 2 0.3 0.2 0.1")
    L.append("CNOT 2 3")
    L.append("CNOT 7 9")
    L.append("T 8")
    L.append("Decompose 7 3 3")    # B out into reg 3
    L.append("Decompose 2 2 4")    # C out into reg 4
    L.append("@3 Prob 0")
    L.append("@3 Prob 2")
    L.append("@4 Prob 1")
    L.append("Allocate 1 2")       # two fresh |0> qubits at 1
    L.append("X 1")
    L.append("Dispose 1 1 1")      # drop the |1> qubit by permutation
    L.append("Dispose 1 1")        # drop the |0> qubit by marginal
    L.append("ForceM 0 1")
    L.append("Prob 0")
    L.append("H 0")
    L.append("ForceMReg 1 2 1")
    L.append("ProbReg 1 2 1")
    L.append("Norm")
    L.append("@3 H 0")
    L.append("@3 ForceM 0 0")
    L.append("@3 Norm")
    return "\n".join(L) + "\n"


def qft_roundtrip(n=10, seed=4):
    rng = random.Random(seed)
    L = ["qubits %d" % n, "SetPermutation %d" % rng.getrandbits(n)]
    for q in range(n):
        if rng.random() < 0.5:
            L.append("H %d" % q)
    L.append("QFT 0 %d" % n)
    L.append("T 3")
    L.append("IQFT 1 %d" % (n - 2))
    for q in range(n):
        L.append("Prob %d" % q)
    return "\n".join(L) + "\n"


def _u_layer(L, rng, qubits):
    for q in qubits:
        L.append("U %d %.17g %.17g %.17g" % (q, rng.uniform(-3, 3), rng.uniform(-3, 3), rng.uniform(-3, 3)))


def alu_add(seed=21):
    """QAlu adders (SURVEY §8f N3).  Register 0..4, carries 5..8 (each used once, so every M(carry) is deterministic),
    overflow flag 9 (in superposition), controls 10, 11."""
    rng = random.Random(seed)
    L = ["qubits 12"]
    _u_layer(L, rng, [0, 1, 2, 3, 4, 9, 10, 11])
    L += ["CNOT 0 3", "CNOT 10 2", "CNOT 4 11"]
    L += ["INC 7 0 5", "DEC 3 1 4", "CINC 2 10 11 5 0 5", "CDEC 1 11 9 1 4", "ROL 2 0 5", "ROR 1 0 5"]
    L += ["PhaseFlipIfLess 13 0 5", "CPhaseFlipIfLess 21 0 5 10"]
    L += ["INCS 11 0 5 9", "DECS 6 0 5 9"]
    L += ["INCC 9 0 5 5", "X 6", "DECC 5 0 5 6", "INCSC 13 0 5 9 7", "X 8", "DECSCc 4 0 5 8"]
    for q in range(12):
        L.append("Prob %d" % q)
    L += ["GetAmplitude 77", "Norm"]
    return "\n".join(L) + "\n"


def alu_mul(seed=22):
    """MUL/DIV and the ModNOut family.  in 0..3, out/carry A 4..7, out B 8..11, controls 12, 13."""
    rng = random.Random(seed)
    L = ["qubits 14"]
    _u_layer(L, rng, [0, 1, 2, 3, 12, 13])
    L += ["CNOT 1 12", "CNOT 13 2"]
    L += ["MUL 5 0 4 4", "Prob 5", "DIV 5 0 4 4", "CMUL 2 12 13 3 0 4 4", "Prob 4", "CDIV 2 12 13 3 0 4 4"]
    L += ["MULModNOut 3 13 0 4 4", "Prob 6", "IMULModNOut 3 13 0 4 4", "POWModNOut 2 11 0 4 4"]
    L += ["CMULModNOut 2 12 13 5 7 0 8 4", "Prob 9", "CIMULModNOut 2 12 13 5 7 0 8 4", "CPOWModNOut 1 12 3 13 0 8 4"]
    for q in range(14):
        L.append("Prob %d" % q)
    L += ["GetAmplitude 1234", "Norm"]
    return "\n".join(L) + "\n"


def alu_idx(seed=23):
    """IndexedLDA / ADC / SBC and Hash.  index 0..2, value 3..6, ADC carry 7, hash register 8..10, SBC carry 11."""
    rng = random.Random(seed)
    L = ["qubits 12"]
    _u_layer(L, rng, [0, 1, 2, 8, 9, 10])
    L += ["CNOT 0 9"]
    tab = lambda: bytes(rng.randrange(16) for _ in range(8)).hex()
    perm = list(range(8))
    rng.shuffle(perm)
    L += ["IndexedLDA 0 3 3 4 %s" % tab(), "Prob 4", "IndexedADC 0 3 3 4 7 %s" % tab(), "X 11",
          "IndexedSBC 0 3 3 4 11 %s" % tab(), "Hash 8 3 %s" % bytes(perm).hex()]
    for q in range(12):
        L.append("Prob %d" % q)
    L += ["GetAmplitude 99", "Norm"]
    return "\n".join(L) + "\n"


SCRIPTS = {
    "htcnot_10q": qscript.random_htcnot(10, 12, seed=20250921, timed=False),
    "htcnot_12q": qscript.random_htcnot(12, 20, seed=12, timed=False),
    "u3_9q": qscript.random_u3_cnot(9, 6, seed=7),
    "qv_9q": qscript.quantum_volume(9, seed=33, timed=False),
    "qft_10q": qft_roundtrip(10),
    "misc_8q": misc_gates(8),
    "structure": structure(),
    "grover_8q": qscript.grover(8, 4, target=3, timed=False),
    "alu_add_12q": alu_add(),
    "alu_mul_14q": alu_mul(),
    "alu_idx_12q": alu_idx(),
}


def _harness(prec, text, td, *args):
    """Run `text` on the compiled reference, outputs inside td."""
    path = os.path.join(td, "c.qs")
    with open(path, "w") as f:
        f.write(text)
    subprocess.run([os.path.join(ROOT, "oracle", "_ref", "ref_harness_f%d" % prec), path] + list(args), check=True)


# Reference outputs kept under reference/ for the tests that compare with the reference on circuits too large for a
# full-state fixture.  A state keeps a seeded sample of SAMPLE amplitudes of register 0 (the whole state when it is smaller).
SAMPLE = 1024


def state_case(text, prec, engine="cpu"):
    dt = np.complex64 if prec == 32 else np.complex128
    with tempfile.TemporaryDirectory() as td:
        _harness(prec, text, td, "--dump", os.path.join(td, "s"), "--engine", engine)
        st = np.fromfile(os.path.join(td, "s.0.bin"), dtype=dt)
    idx = np.arange(st.size) if st.size <= SAMPLE else np.sort(np.random.default_rng(1).choice(st.size, SAMPLE, replace=False))
    return {"text": text, "idx": idx.astype(np.int64), "amp": st[idx]}


def results_case(text, prec):
    """Query results of the fp`prec` reference; for fp32 also those of the fp64 build on the same circuit ("results_f64"):
    the fp32 reference sums each Prob in fp32 per worker thread with a dynamic work split, so its own Prob wanders by up to
    ~1e-4 from run to run at these sizes, and the tests take the probabilities from the fp64 build."""
    out = {"text": text}
    for p in ((32, 64) if prec == 32 else (64,)):
        with tempfile.TemporaryDirectory() as td:
            _harness(p, text, td, "--results", os.path.join(td, "r.txt"))
            out["results" if p == prec else "results_f64"] = open(os.path.join(td, "r.txt")).read()
    return out


def full_size_text(n, kind):
    """tests/test_parity_gpu.py::test_full_size_parity_against_the_compiled_reference: 30-qubit fp32 depth-2 H/T/CNOT or
    29-qubit fp64 QFT prefix, then every per-qubit Prob and 64 sampled amplitudes."""
    rng = random.Random(77)
    if kind == "htcnot":
        text = qscript.random_htcnot(n, 2, seed=31, timed=False)
    else:
        # H on a random half of the qubits, then the first 3 target qubits of QFT(0, n): 3 H + 84 controlled phases on all qubits
        lines = ["qubits %d" % n] + ["H %d" % q for q in range(n) if rng.random() < 0.5]
        for i in range(3):
            hb = n - 1 - i
            lines.append("H %d" % hb)
            for j in range(hb):
                lines.append("CPhaseRootN %d %d %d" % (hb - j + 1, j, hb))
        text = "\n".join(lines) + "\n"
    idx = sorted(rng.randrange(1 << n) for _ in range(64))
    return text + "".join("Prob %d\n" % q for q in range(n)) + "".join("GetAmplitude %d\n" % i for i in idx)


def sharded_26q_text(kind):
    """tests/test_sharded_gpu.py::test_sharded_26q_against_the_compiled_reference: all per-qubit Prob, 48 sampled amplitudes."""
    n = 26
    rng = random.Random(5)
    text = {"htcnot": lambda: qscript.random_htcnot(n, 6, seed=12, timed=False),
            "qv": lambda: qscript.quantum_volume(n, depth=4, seed=13, timed=False),
            "grover": lambda: "\n".join(l for l in qscript.grover(n, 1, target=3, timed=False).splitlines() if not l.startswith("ProbAll")) + "\n"}[kind]()
    idx = sorted(rng.randrange(1 << n) for _ in range(48)) + [3]
    return text + "".join("Prob %d\n" % q for q in range(n)) + "".join("GetAmplitude %d\n" % i for i in idx)


C1_16Q = qscript.random_htcnot(16, 40, seed=20250921, timed=False)   # BASELINE configs[0] at reduced width
C1_20Q = qscript.random_htcnot(20, 40, seed=20250921, timed=False)   # BASELINE configs[0]
REFERENCE_CASES = {
    "c1_16q_f32": lambda: state_case(C1_16Q, 32),
    "c1_16q_f64": lambda: state_case(C1_16Q, 64),
    # QPager over QEngineCPU with forced small pages (2^7 amplitudes)
    "pager_10q_f32": lambda: state_case(qscript.random_htcnot(10, 6, seed=3, timed=False), 32, engine="pager:7"),
    "c1_20q_f32": lambda: state_case(C1_20Q, 32),
    "c1_20q_f64": lambda: state_case(C1_20Q, 64),
    "full_30q_htcnot_f32": lambda: results_case(full_size_text(30, "htcnot"), 32),
    "full_29q_qft_f64": lambda: results_case(full_size_text(29, "qft"), 64),
    "sharded_26q_htcnot_f32": lambda: results_case(sharded_26q_text("htcnot"), 32),
    "sharded_26q_qv_f32": lambda: results_case(sharded_26q_text("qv"), 32),
    "sharded_26q_grover_f32": lambda: results_case(sharded_26q_text("grover"), 32),
}


def main_reference(names):
    os.makedirs(os.path.join(HERE, "reference"), exist_ok=True)
    for name in names or REFERENCE_CASES:
        np.savez_compressed(os.path.join(HERE, "reference", name + ".npz"), **REFERENCE_CASES[name]())
        print("wrote reference/%s.npz" % name)


def main():
    for name, text in SCRIPTS.items():
        path = os.path.join(HERE, name + ".qs")
        with open(path, "w") as f:
            f.write(text)
        for prec, dt in ((32, np.complex64), (64, np.complex128)):
            harness = os.path.join(ROOT, "oracle", "_ref", "ref_harness_f%d" % prec)
            with tempfile.TemporaryDirectory() as td:
                subprocess.run([harness, path, "--dump", os.path.join(td, "s"), "--results", os.path.join(td, "r.txt")],
                               check=True)
                arrays = {}
                for fn in sorted(os.listdir(td)):
                    if fn.startswith("s.") and fn.endswith(".bin"):
                        arrays["reg%s" % fn.split(".")[1]] = np.fromfile(os.path.join(td, fn), dtype=dt)
                res = open(os.path.join(td, "r.txt")).read()
            arrays["results"] = np.array(res)
            np.savez_compressed(os.path.join(HERE, "%s.f%d.npz" % (name, prec)), **arrays)
        print("wrote", name)


if __name__ == "__main__":
    if sys.argv[1:2] == ["reference"]:
        main_reference(sys.argv[2:])
    else:
        main()
