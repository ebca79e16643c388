"""bench.py's JSON contract, exercised without a GPU: the N=1 main path runs end to end against a stand-in engine (the
oracle restatement with the CUDA backend's stats/timer hooks stubbed), and the reference arm runs for real on host cores.
Guards the keys the driver reads (metric/value/unit/..., roofline, cpu_baseline, e2e, gpu_launches, clocks)."""
import json
import os
import subprocess
import sys

import pytest

import util

SHIM = r'''
import sys, random, time
sys.path.insert(0, %r)
import bench
from oracle.restate_engine import QEngineRestate
class Fake(QEngineRestate):
    def __init__(self, n, perm, rng, phase, a, b, deviceId=0, precision=32):
        super().__init__(n, perm, rng, phase, a, b, precision=precision)
        be = self.be
        st = {'kernel_launches': 0, 'fused_sweeps': 0, 'fused_gates': 0, 'bytes_swept': 0, 'gates_submitted': 0, 'single_launches': 0}
        t = [0.0]
        be.set_fusion = lambda f: None
        def flush():
            st['kernel_launches'] += 1; st['fused_sweeps'] += 1; st['bytes_swept'] += 2 * (1 << n) * 8
        be.flush = flush
        be.stats = lambda: dict(st)
        be.reset_stats = lambda: [st.__setitem__(k, 0) for k in st]
        be.timer_begin = lambda: t.__setitem__(0, time.perf_counter())
        def tend():
            flush(); return (time.perf_counter() - t[0]) * 1e3
        be.timer_end = tend
import qrack_b200
qrack_b200.QEngineCUDA = Fake
sys.argv = ['bench.py', '--qubits', '9', '--steps', '2', '--warmup', '3', '--skip-cpu-baseline']
bench.main()
'''


def _last_json(out):
    return json.loads([l for l in out.splitlines() if l.startswith("{")][-1])


def test_b200_arm_json_contract():
    r = subprocess.run([sys.executable, "-c", SHIM % util.ROOT], capture_output=True, text=True, timeout=600, cwd=util.ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    j = _last_json(r.stdout)
    for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
              "dtype", "data", "config", "gpu_launches", "e2e", "roofline", "clocks"):
        assert k in j, k
    assert j["n_gpus"] == 1 and j["steps"] == 2 and j["warmup"] >= 3 and j["unit"] == "gates/s" and j["dtype"] == "f32"
    assert j["vs_baseline"] is None and "workload" in j["config"] and "model" not in j["config"]
    for k in ("bound", "achieved", "peak", "unit", "frac", "traffic", "algorithmic_gbs", "algorithmic_frac", "fused_single_qubit_sweep"):
        assert k in j["roofline"], k
    for k in ("value", "unit", "h2d_bytes_per_step", "d2h_bytes_per_step"):
        assert k in j["e2e"], k
    assert j["gpu_launches"] > 0
    # self-checks computed in the run: norm, marginals, mirror-circuit return
    assert j["check"]["ok"] is True and abs(j["check"]["norm_minus_1"]) < 1e-4 and abs(j["check"]["mirror_return_prob"] - 1) < 1e-3


@pytest.mark.parametrize("workload,extra", [("grover", ["--depth", "2"]), ("qft", ["--precision", "64"]), ("qv", ["--depth", "3"])])
def test_b200_arm_other_baseline_workloads(workload, extra):
    shim = (SHIM % util.ROOT).replace("'--skip-cpu-baseline']", "'--skip-cpu-baseline', '--workload', %r] + %r" % (workload, extra))
    r = subprocess.run([sys.executable, "-c", shim], capture_output=True, text=True, timeout=600, cwd=util.ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    j = _last_json(r.stdout)
    assert j["check"]["ok"] is True, j["check"]
    if workload == "grover":
        assert abs(j["check"]["grover_success_prob"] - j["check"]["grover_law_sin2((2k+1)asin(2^-n/2))"]) < 1e-4


def test_reference_arm_runs_on_host_cores():
    # the compiled reference when oracle/_ref was built (it needs the reference sources), otherwise the oracle port
    kind = "port" if util.ref_harness(32) is None else "reference"
    r = subprocess.run([sys.executable, os.path.join(util.ROOT, "bench.py"), "--impl", "reference", "--qubits", "16", "--steps", "2",
                        "--warmup", "1"], capture_output=True, text=True, timeout=600, cwd=util.ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    j = _last_json(r.stdout)
    assert j["impl"] == "reference" and j["unit"] == "gates/s" and j["value"] > 0
    assert j["cpu_baseline"]["kind"] == kind and j["cpu_baseline"]["cores"] >= 1
    assert j["e2e"]["h2d_bytes_per_step"] == 0 and j["e2e"]["d2h_bytes_per_step"] == 0
    # the sample is a fixed prefix of the circuit (>= one full layer incl. CNOTs), whatever --steps is, and `config` is the b200 arm's
    assert j["reference_sample"]["ops_total"] >= 60 and len(j["reference_sample"]["segment_seconds"]) == 2
    r5 = subprocess.run([sys.executable, os.path.join(util.ROOT, "bench.py"), "--impl", "reference", "--qubits", "16", "--steps", "20",
                         "--warmup", "0"], capture_output=True, text=True, timeout=600, cwd=util.ROOT)
    j5 = _last_json(r5.stdout)
    assert j5["reference_sample"]["ops_total"] == 60 and j5["config"] == j["config"]
    assert set(j["config"]) == {"workload", "l2_policy", "fusion", "parallelism"}
    # other ranks of a torchrun launch do no work
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    r = subprocess.run([sys.executable, os.path.join(util.ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--qubits", "16"],
                       capture_output=True, text=True, timeout=120, cwd=util.ROOT, env=env)
    assert r.returncode == 0 and not r.stdout.strip()


def test_dump_outputs_are_the_same_from_run_to_run(tmp_path):
    """--dump-outputs DIR: the last timed step's state sample and the per-qubit probabilities, in the engine's precision, identical
    for two runs with the same arguments."""
    import numpy as np
    outs = []
    for run in ("a", "b"):
        d = tmp_path / run
        shim = (SHIM % util.ROOT).replace("'--skip-cpu-baseline']", "'--skip-cpu-baseline', '--dump-outputs', %r]" % str(d))
        r = subprocess.run([sys.executable, "-c", shim], capture_output=True, text=True, timeout=600, cwd=util.ROOT)
        assert r.returncode == 0, r.stderr[-2000:]
        outs.append({f.name: np.load(str(f)) for f in d.iterdir()})
    a, b = outs
    assert set(a) == {"state_sample.npy", "qubit_probs.npy"}
    assert a["state_sample.npy"].dtype == np.float32 and a["state_sample.npy"].shape == (1 << 9, 2)
    assert a["qubit_probs.npy"].dtype == np.float64 and a["qubit_probs.npy"].shape == (9,)
    for k in a:
        assert np.array_equal(a[k], b[k]), k
    # the state sample is the state: its marginals are the probabilities the end-to-end arm read
    st = a["state_sample.npy"].astype(np.float64)
    p = st[:, 0] ** 2 + st[:, 1] ** 2
    idx = np.arange(p.size)
    assert np.allclose([p[(idx >> q) & 1 == 1].sum() for q in range(9)], a["qubit_probs.npy"], atol=1e-5)


def test_state_sample_pages_are_fixed_and_exact():
    import numpy as np
    import bench

    class Engine:
        def __init__(self, n):
            self.st = (np.arange(1 << n) * (1 + 2j)).astype(np.complex128)

        def GetAmplitudePage(self, offset, length):
            return self.st[offset:offset + length]

    n = 22
    a, b = bench.state_sample(Engine(n), n), bench.state_sample(Engine(n), n)
    assert a.dtype == np.float64 and a.shape == (1 << 20, 2) and np.array_equal(a, b)
    pos = a[:, 0].astype(np.int64)              # amplitude i holds i + 2i j
    assert np.array_equal(a[:, 1], 2 * a[:, 0]) and np.all(np.diff(pos) > 0)
    assert np.all(pos.reshape(-1, 1 << 12) % (1 << 12) == np.arange(1 << 12))   # whole pages
    assert pos.max() >= (1 << 21)                                                # spread over the state
