#!/usr/bin/env python
"""bench.py — gates/sec on BASELINE.json's workloads + Apply2x2 HBM roofline (contract: see DESIGN.md §Measurement).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--workload htcnot|qft|qv|grover]
                  [--qubits n] [--depth d] [--precision 32|64] [--dump-outputs DIR]

A "step" = one replay of the whole seeded circuit on a state vector that is already resident in HBM.  Default workload =
BASELINE configs[1]: 30 qubits, H/T/CNOT depth 40, 1800 gates, fp32.  Other BASELINE configs: `--workload qft --precision 64`
(configs[2]), `--workload qv --gpus 8` (configs[3]: 33 q, depth 33), `--workload grover --qubits 31 --gpus 8` (configs[4]: 34 q).
`value` = gates/s over exactly K timed steps (CUDA events on the engine's own stream, max over ranks); `e2e` = the same
metric through the public QEngineCUDA API with host-side gate submission, state (re)initialisation and a device->host read
of per-qubit probabilities inside the timed region.  `check` = self-checks computed in the run after the timed regions
(norm, mirror-circuit return probability, Grover success law): a throughput number over an unverified state is not a result.
`--impl reference` times the compiled reference QEngineCPU (oracle/_ref) — or the oracle port when that binary did not
travel — on a bounded, fixed sample of the same workload on the host cores.
`--dump-outputs DIR` (1 GPU) writes what the last timed steps computed, for comparing two builds output for output:
DIR/state_sample.npy = a fixed sample of the final state (see state_sample), DIR/qubit_probs.npy = Prob(q) of every qubit.
"""
import argparse
import json
import math
import os
import random
import statistics
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

from qrack_b200 import qscript  # noqa: E402

METRIC = "gates/sec at 30q random circuit; Apply2x2 HBM GB/s vs roofline"
REF_SAMPLE_GATES = 60  # reference arm / cpu_baseline: the first 60 gates (one full layer incl. its CNOTs + 15), whatever --steps is
GROVER_TARGET = 3


# ---------------------------------------------------------------------------------------------------------------------
# workloads
# ---------------------------------------------------------------------------------------------------------------------
def build_workload(name, n, depth, seed, prec):
    """-> (script text without TIC/TOC and queries, gate count as the metric counts it, description)"""
    if name == "qft":
        text = qscript.qft(n, seed=11, timed=False)
        calls = gate_calls(text)
        gates = sum(1 for c in calls if c[0] == "H") + n + n * (n - 1) // 2  # init H's + QFT's own H and CPhaseRootN gates
        desc = "%d-qubit QFT (%d H + %d controlled-phase), fp%d amplitudes" % (n, n, n * (n - 1) // 2, prec)
    elif name == "qv":
        d = n if depth is None else depth
        text = qscript.quantum_volume(n, depth=d, seed=33, timed=False)
        gates = qscript.count_gate_ops(text)
        desc = "%d-qubit quantum-volume layers (AI + CNOT matching, depth %d, %d gates), fp%d" % (n, d, gates, prec)
    elif name == "grover":
        it = 3 if depth is None else depth
        text = "\n".join(l for l in qscript.grover(n, it, target=GROVER_TARGET, timed=False).splitlines() if not l.startswith("ProbAll")) + "\n"
        gates = qscript.count_gate_ops(text)
        desc = "%d-qubit Grover search (H^n; %d x {DEC, ZeroPhaseFlip, INC, H^n, ZeroPhaseFlip, H^n}; %d ops), fp%d" % (n, it, gates, prec)
    else:
        d = 40 if depth is None else depth
        text = qscript.random_htcnot(n, d, seed=seed, timed=False)
        gates = qscript.count_gate_ops(text)
        desc = "%d-qubit random circuit (H/T/CNOT, depth %d, %d gates), fp%d amplitudes" % (n, d, gates, prec)
    return text, gates, desc


_INVERSE = {"H": "H", "X": "X", "Y": "Y", "Z": "Z", "CNOT": "CNOT", "CZ": "CZ", "CCNOT": "CCNOT", "Swap": "Swap",
            "T": "IT", "IT": "T", "S": "IS", "IS": "S", "AI": "IAI", "IAI": "AI", "QFT": "IQFT", "IQFT": "QFT",
            "INC": "DEC", "DEC": "INC", "ZeroPhaseFlip": "ZeroPhaseFlip"}


def inverse_text(text):
    """The mirror circuit: ops reversed, each replaced by its inverse (only the op families the workloads use)."""
    out = []
    for _, t in reversed(qscript.parse(text)):
        if t[0] in ("qubits", "TIC", "TOC") or t[0] in qscript.QUERY_OPS:
            continue
        out.append(" ".join([_INVERSE[t[0]]] + list(t[1:])))
    return "\n".join(out) + "\n"


def gate_calls(text):
    """Pre-parse the script into (method name, args) so the timed loop is only API calls."""
    calls = []
    for _, t in qscript.parse(text):
        if t[0] in ("qubits", "TIC", "TOC") or t[0] in qscript.QUERY_OPS:
            continue
        calls.append((t[0], tuple((float(x) if ("." in x or "e" in x or "inf" in x or "nan" in x) else int(x)) for x in t[1:])))
    return calls


def algorithmic_bytes(calls, n, amp_bytes):
    """SURVEY.md §8(d): B(gate) = 2 * 2^(n-c) * S, c = number of control qubits (register-wide ops: one full sweep)."""
    tot = 0
    for name, args in calls:
        c = 1 if name in ("CNOT", "CZ", "CY", "AntiCNOT", "Swap", "CPhaseRootN") else 0
        if name == "QFT":
            ln = args[1]
            tot += ln * 2 * (1 << n) * amp_bytes + (ln * (ln - 1) // 2) * 2 * (1 << (n - 1)) * amp_bytes
            continue
        tot += 2 * (1 << (n - c)) * amp_bytes
    return tot


# ---------------------------------------------------------------------------------------------------------------------
# roofline helpers
# ---------------------------------------------------------------------------------------------------------------------
def committed_traffic(kernel_bytes_per_launch):
    """dram__bytes_read+write per launch of the fused sweep from the newest committed `ncu --set full` summary under
    profiles/ (a 28-qubit capture), scaled to this run's state size.  NOT measured in this run — labelled as such."""
    for fn in ("r2_final_fused_ncu_full.json", "r2_fused_ncu_full.json", "r1_fused_v9_ncu_full.json"):
        p = os.path.join(ROOT, "profiles", fn)
        try:
            j = json.load(open(p))
            l = j["launches"][0]
            per28 = (float(l["dram__bytes_read.sum"]) + float(l["dram__bytes_write.sum"])) * 1e9
            return per28 / (2.0 * (1 << 28) * 8) * kernel_bytes_per_launch, "profiles/%s (28-qubit ncu capture scaled by state size; not measured in this run)" % fn
        except Exception:
            continue
    return None, None


def fused_single_qubit_sweep_probe(q, n, amp_bytes, peak, reps=5, warm=2):
    """The north-star's own roofline target, measured live: ONE fused sweep of single-qubit gates (H on qubits 0 and 1)
    over the resident 2^n state; physical bytes 2 * 2^n * S / CUDA-event time on the engine's stream.  Never fatal."""
    try:
        def layer():
            q.H(0)
            q.H(1)
            q.be.flush()
        for _ in range(warm):
            layer()
        q.Finish()
        s0 = q.be.stats()
        q.be.timer_begin()
        for _ in range(reps):
            layer()
        ms = q.be.timer_end() / reps
        s1 = q.be.stats()
        sweeps = (s1["fused_sweeps"] - s0["fused_sweeps"]) / float(reps)
        if ms <= 0 or sweeps != 1.0:
            return {"gates": 2, "ms": ms, "sweeps": sweeps, "physical_gbs": None, "frac": None}
        gbs = 2.0 * (1 << n) * amp_bytes / (ms * 1e-3) / 1e9
        return {"gates": 2, "ms": ms, "sweeps": sweeps, "physical_gbs": gbs, "frac": gbs / peak}
    except Exception as e:  # diagnostic only: the headline numbers above are already taken
        return {"error": repr(e)[:200]}


def state_sample(q, n, page=1 << 12, pages=1 << 8):
    """A fixed sample of the state, the same for every run at this n: the whole state up to page * pages amplitudes, else
    `pages` pages of `page` amplitudes at seeded offsets.  -> float array (amplitudes, 2) of (real, imaginary) in the engine's
    precision: 8 MiB (fp32) / 16 MiB (fp64) at most."""
    import numpy as np
    if (1 << n) <= page * pages:
        spans = [(0, 1 << n)]
    else:
        spans = [(p * page, page) for p in sorted(random.Random(0).sample(range((1 << n) // page), pages))]
    amps = np.concatenate([q.GetAmplitudePage(o, k) for o, k in spans])
    return np.stack([amps.real, amps.imag], axis=-1)


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler(threading.Thread):
    """nvidia-smi clocks + throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        super().__init__(daemon=True)
        self.gpu = gpu_index
        self.rows = []
        self.stop_flag = False

    def run(self):
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([x.strip() for x in out.split(",")])
            except Exception:
                pass
            time.sleep(0.2)

    def summary(self):
        sm = [float(r[1]) for r in self.rows if len(r) > 2 and r[1].replace(".", "").isdigit()]
        mx = [float(r[2]) for r in self.rows if len(r) > 2 and r[2].replace(".", "").isdigit()]
        reasons = set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            for k, nm in enumerate(names):
                if len(r) > 5 + k and r[5 + k].lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(self.rows)}


# ---------------------------------------------------------------------------------------------------------------------
# the reference's CPU path on the host cores (cpu_baseline leg and --impl reference)
# ---------------------------------------------------------------------------------------------------------------------
def cpu_reference_sample(text, n, prec, per_step, steps, desc, threads=None):
    """Time the compiled reference (oracle/_ref/ref_harness) on the FIRST steps*per_step ops of the workload, as `steps`
    consecutive TIC..TOC segments of one process (the state carries over, so the sample is one contiguous prefix of the
    circuit — the same prefix whatever `steps` is, as long as steps*per_step is)."""
    harness = os.path.join(ROOT, "oracle", "_ref", "ref_harness_f%d" % prec)
    lines = [l for l in text.splitlines() if l.strip()]
    head, ops = lines[0], lines[1:]
    total = min(len(ops), per_step * steps)
    per_step = max(1, total // steps)
    total = per_step * steps
    if os.path.exists(harness):
        sample = [head]
        for s in range(steps):
            sample += ["TIC"] + ops[s * per_step:(s + 1) * per_step] + ["TOC"]
        with tempfile.TemporaryDirectory() as td:
            sp = os.path.join(td, "s.qs")
            open(sp, "w").write("\n".join(sample) + "\n")
            cmd = [harness, sp, "--time"] + (["--threads", str(threads)] if threads else [])
            out = subprocess.run(cmd, capture_output=True, text=True, check=True).stdout
        j = json.loads(out.strip().splitlines()[-1])
        segs = j.get("segments") or [[j["ops"], j["seconds"]]]
        return {"value": j["ops"] / j["seconds"], "unit": "gates/s", "cores": j["threads"], "kind": "reference",
                "sample": "first %d ops of the %s on QEngineCPU (fp%d), %d segments, %.1f s" % (j["ops"], desc, prec, len(segs), j["seconds"]),
                "seconds": j["seconds"], "gates": j["ops"], "segments": segs}
    # oracle port (single-threaded C restatement)
    from oracle.restate_engine import QEngineRestate
    q = QEngineRestate(n, 0, random.Random(1), 1.0 + 0j, False, False, precision=prec)
    calls = gate_calls("\n".join([head] + ops[:total]) + "\n")
    segs = []
    for s in range(steps):
        t0 = time.perf_counter()
        for name, a in calls[s * per_step:(s + 1) * per_step]:
            getattr(q, name)(*a)
        segs.append([per_step, time.perf_counter() - t0])
    dt = sum(x[1] for x in segs)
    return {"value": total / dt, "unit": "gates/s", "cores": 1, "kind": "port",
            "sample": "first %d ops of the %s on the oracle C restatement (fp%d), %.1f s" % (total, desc, prec, dt),
            "seconds": dt, "gates": total, "segments": segs}


def dist_setup(n_gpus):
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        import torch
        import torch.distributed as dist
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
        return rank, world, local, dist
    return rank, world, local, None


def make_config(desc, n, amp_bytes, world, exchange, fusion):
    """Identical in both arms (the driver compares the two lines' `config`)."""
    return {"workload": desc,
            "l2_policy": "state vector (%.1f GiB) is far larger than the 126 MB L2" % ((1 << n) * amp_bytes / 2 ** 30),
            "fusion": fusion,
            "parallelism": "1 GPU" if world == 1 else
            "1 state vector sharded over %d GPUs (top %d qubits = rank), qubit exchange: %s" %
            (world, world.bit_length() - 1, "fused NVLink peer-store kernel" if exchange == "p2p" else "NCCL all_to_all_single + local swap sweeps")}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--qubits", type=int, default=30, help="qubits PER GPU SHARD: the state has qubits + log2(gpus) qubits")
    ap.add_argument("--depth", type=int, default=None, help="htcnot: layers (40); qv: layers (= qubits); grover: iterations (3)")
    ap.add_argument("--precision", type=int, default=32)
    ap.add_argument("--seed", type=int, default=20250921)
    ap.add_argument("--fusion", type=int, default=1)
    ap.add_argument("--cpu-sample-gates", type=int, default=REF_SAMPLE_GATES)
    ap.add_argument("--skip-cpu-baseline", action="store_true")
    ap.add_argument("--skip-check", action="store_true")
    ap.add_argument("--exchange", default="p2p", choices=["p2p", "nccl"],
                    help="N>1: qubit exchange by the fused NVLink peer-store kernel (default) or NCCL all_to_all + local swaps")
    ap.add_argument("--workload", default="htcnot", choices=["htcnot", "qft", "qv", "grover"],
                    help="htcnot = BASELINE configs[1] (default, the headline); qft = configs[2]; qv = configs[3]; grover = configs[4]")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the last timed steps to DIR/<name>.npy (1 GPU, --impl b200)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "b200" or args.gpus > 1):
        ap.error("--dump-outputs needs --impl b200 on 1 GPU")
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup

    world_req = max(1, args.gpus)
    shard_bits = world_req.bit_length() - 1 if world_req > 1 else 0
    prec = args.precision
    amp_bytes = 8 if prec == 32 else 16
    dtype = "f32" if prec == 32 else "f64"
    # weak scaling: 2^qubits amplitudes per GPU => qubits + log2 N in all, in BOTH arms
    n = args.qubits + shard_bits
    text, gates, desc = build_workload(args.workload, n, args.depth, args.seed, prec)
    if shard_bits:
        desc += ", 2^%d amplitudes per GPU" % args.qubits
    calls = gate_calls(text)
    config = make_config(desc, n, amp_bytes, world_req, args.exchange, args.fusion)

    if args.impl == "reference":
        rank = int(os.environ.get("RANK", "0"))
        if rank != 0:
            return
        steps = max(args.steps, 1)
        # a FIXED prefix of the circuit (one full layer with its CNOTs and more), independent of --steps; it shrinks with the
        # state size at N>1 so that the run still ends within minutes (each op costs 2x per extra qubit)
        budget = max(steps, args.cpu_sample_gates >> shard_bits)
        per_step = max(1, -(-budget // steps))
        if args.warmup > 0:
            wtext, _, wdesc = build_workload(args.workload, min(n, 22), args.depth, args.seed, prec)
            cpu_reference_sample(wtext, min(n, 22), prec, per_step, 1, wdesc)
        cb = cpu_reference_sample(text, n, prec, per_step, steps, desc)
        v = cb["value"]
        line = {"impl": "reference", "metric": METRIC, "value": v, "unit": "gates/s", "n_gpus": args.gpus, "steps": steps,
                "warmup": args.warmup, "ms_per_step": 1e3 * cb["seconds"] / steps, "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": dtype, "data": "synthetic", "config": config,
                "cpu_baseline": {k: cb[k] for k in ("value", "unit", "cores", "kind", "sample")},
                "reference_sample": {"ops_per_step": per_step, "ops_total": cb["gates"], "engine": "QEngineCPU (reference, host cores)",
                                     "segment_seconds": [round(s[1], 4) for s in cb["segments"]]},
                "e2e": {"value": v, "unit": "gates/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        print(json.dumps(line))
        return

    rank, world, local, dist = dist_setup(args.gpus)
    from qrack_b200 import QEngineCUDA

    sharded = world > 1
    if sharded:
        # ONE state vector of n = qubits + log2(N) qubits sharded over the N GPUs
        import torch
        from qrack_b200.sharded import QEngineSharded, cuda_engine_factory
        if world != world_req:
            raise SystemExit("bench.py: --gpus %d but WORLD_SIZE=%d" % (args.gpus, world))
        os.environ["B200SV_FUSED"] = os.environ.get("B200SV_FUSED", "")
        q = QEngineSharded(n, 0, random.Random(1), 1.0 + 0j, precision=prec, dist=dist, world=world, rank=rank,
                           device=torch.device("cuda", local), make_engine=cuda_engine_factory(local, prec),
                           p2p=(args.exchange == "p2p"))
    else:
        q = QEngineCUDA(n, 0, random.Random(1), 1.0 + 0j, False, False, deviceId=local, precision=prec)
        q.be.set_fusion(args.fusion)

    def replay(cs=calls):
        for name, a in cs:
            getattr(q, name)(*a)

    def barrier():
        if dist is not None:
            import torch
            dist.barrier()
            torch.cuda.synchronize()

    def get_stats():
        return q.be.shard.stats() if sharded else q.be.stats()

    # ---- device-timed arm: state resident in HBM, CUDA events on the stream the kernels run on --------------------
    for _ in range(args.warmup):
        q.SetPermutation(0, 1.0 + 0j)
        replay()
        q.Finish()
    sampler = ClockSampler(local)
    sampler.start()
    ms_steps = []
    ex0 = q.be.exchanges if sharded else 0
    car0 = getattr(q.be, "carried_ops", 0) if sharded else 0
    stats0 = get_stats()
    if not sharded:
        q.be.reset_stats()
        stats0 = {k: 0 for k in stats0}
    barrier()
    for _ in range(args.steps):
        q.SetPermutation(0, 1.0 + 0j)
        q.Finish()
        if sharded:
            import torch
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()          # the local engines run on torch's current stream (b200sv_set_stream), like NCCL
            replay()
            q.be.flush()
            q.be.loc.be.flush()
            e1.record()
            e1.synchronize()
            ms_steps.append(e0.elapsed_time(e1))
        else:
            q.be.timer_begin()
            replay()
            ms_steps.append(q.be.timer_end())
    barrier()
    stats1 = get_stats()
    stats = {k: stats1[k] - stats0.get(k, 0) for k in stats1}
    exchanges = (q.be.exchanges - ex0) if sharded else 0
    carried = (getattr(q.be, "carried_ops", 0) - car0) if sharded else 0
    dumped_state = state_sample(q, n) if args.dump_outputs else None
    # ---- end-to-end arm: public API, host submission + init + result read inside the timed region -----------
    h2d = gates * (8 * 8 + 8 * 4)  # per gate: 8 doubles of matrix + offsets/powers words crossing the C ABI
    d2h = n * 8
    e2e_steps = []
    probs = None
    for _ in range(args.steps):
        t0 = time.perf_counter()
        q.SetPermutation(0, 1.0 + 0j)
        replay()
        probs = [q.Prob(b) for b in range(n)]
        e2e_steps.append(time.perf_counter() - t0)
    barrier()
    # the same end-to-end step with whole-circuit submission (QCircuit.Run -> b200sv_apply_gates: one ABI call per step)
    e2e_batched = None
    if not sharded:
        try:
            from qrack_b200 import QCircuit
            circ = QCircuit(n, prec)
            for name, a in calls:
                getattr(circ, name)(*a)
            circ.packed()
            tb = []
            for _ in range(args.steps):
                t0 = time.perf_counter()
                q.SetPermutation(0, 1.0 + 0j)
                circ.Run(q)
                probs_b = [q.Prob(b) for b in range(n)]
                tb.append(time.perf_counter() - t0)
            agree = max(abs(x - y) for x, y in zip(probs, probs_b))
            e2e_batched = {"value": gates * args.steps / sum(tb), "unit": "gates/s", "abi_calls_per_step": 1,
                           "recorded_apply2x2_forms": circ.GetGateCount(), "max_prob_diff_vs_per_gate_path": agree}
        except NotImplementedError as e:
            e2e_batched = {"unavailable": str(e)[:160]}
    sampler.stop_flag = True
    sampler.join(timeout=2)

    # ---- self-checks on the state the timed steps produced (outside every timed region) --------------------------------
    check = None
    if not args.skip_check:
        check = {}
        tol = 2e-4 if prec == 32 else 1e-9
        q.UpdateRunningNorm()
        nrm = float(q.GetRunningNorm())
        check["norm_minus_1"] = nrm - 1.0
        ok = abs(nrm - 1.0) <= tol
        check["marginals_in_unit_interval"] = bool(all(-1e-6 <= p <= 1.0 + 1e-6 for p in probs))
        ok = ok and check["marginals_in_unit_interval"]
        if args.workload == "grover":
            it = 3 if args.depth is None else args.depth
            got = float(q.ProbAll(GROVER_TARGET))
            law = math.sin((2 * it + 1) * math.asin(2.0 ** (-n / 2.0))) ** 2
            check["grover_success_prob"] = got
            check["grover_law_sin2((2k+1)asin(2^-n/2))"] = law
            ok = ok and abs(got - law) <= max(1e-3 * law, 1e-12)
        # mirror circuit: U then U^-1 from |0..0> must return to |0..0>
        inv_calls = gate_calls(inverse_text(text))
        q.SetPermutation(0, 1.0 + 0j)
        replay()
        replay(inv_calls)
        amp0 = q.GetAmplitude(0)
        ret = float(abs(amp0) ** 2)
        check["mirror_return_prob"] = ret
        ok = ok and abs(ret - 1.0) <= (5e-3 if prec == 32 else 1e-9)
        check["ok"] = bool(ok)
        barrier()

    ms_total = sum(ms_steps)
    e2e_total = sum(e2e_steps)
    if dist is not None:
        import torch
        t = torch.tensor([ms_total, e2e_total], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_total, e2e_total = t.tolist()
    total_gates = gates * args.steps  # one circuit on one (possibly sharded) state vector: whole-job gate count
    value = total_gates / (ms_total / 1e3)
    e2e_value = total_gates / e2e_total

    if rank == 0:
        peak, peak_src = peaks()
        launches = stats["kernel_launches"]
        swept = stats["bytes_swept"]  # rank 0's local kernels; the roofline entry is per GPU
        kernel_ms = ms_total / max(1, launches) * 1.0
        achieved = (swept / 1e9) / (ms_total / 1e3) if ms_total > 0 else 0.0
        alg = algorithmic_bytes(calls, n, amp_bytes) * args.steps
        traffic, traffic_src = (committed_traffic(swept / max(1, launches)) if stats["fused_sweeps"] else (None, None))
        line = {
            "metric": METRIC, "value": value, "unit": "gates/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_total / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": dtype, "data": "synthetic",
            "config": config,
            "gpu_launches": int(launches),
            "e2e": {"value": e2e_value, "unit": "gates/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "includes": "SetPermutation + host gate submission through the C ABI + Prob(q) for every qubit"},
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src,
                         "kernel": "fused sweep" if stats["fused_sweeps"] else "k_apply2x2",
                         "bytes_per_launch": swept / max(1, launches), "ms_per_launch": kernel_ms,
                         "algorithmic_gbs": (alg / 1e9) / (ms_total / 1e3),
                         "algorithmic_frac": (alg / 1e9) / (ms_total / 1e3) / peak,
                         "note": "achieved/frac = PHYSICAL bytes of the launch (2 * 2^n * S) / duration (per GPU); algorithmic_* "
                                 "credits sum_W 2*2^(n-c)*S per fused gate (SURVEY 8d) and is not a roofline fraction",
                         "fused_sweeps": int(stats["fused_sweeps"]),
                         "fused_gates": int(stats["fused_gates"])},
            "clocks": sampler.summary(),
        }
        if sharded:
            page_bytes = (1 << args.qubits) * amp_bytes
            line["sharding"] = {"exchanges_per_step": exchanges / max(1, args.steps),
                                "nvlink_bytes_out_per_gpu_per_step": exchanges / max(1, args.steps) * page_bytes * (world - 1) / world,
                                "sweeps_per_step": stats["fused_sweeps"] / max(1, args.steps),
                                # exchanges carried by the first sweep of the next window (b200sv_exchange_pull) instead of a pass of their own
                                "pull_sweeps_per_step": stats.get("pull_sweeps", 0) / max(1, args.steps),
                                "exchange_mode": "pull (fused into the next sweep)" if stats.get("pull_sweeps", 0) else "push kernel",
                                # lowered ops the local engine handed back instead of running them in a nearly empty last sweep of a window
                                # (b200sv_flush_carry); they ran at the head of the next window
                                "ops_carried_across_exchanges_per_step": carried / max(1, args.steps)}
        if check is not None:
            line["check"] = check
        if e2e_batched is not None:
            line["e2e_batched"] = e2e_batched
        if world == 1 and stats["fused_sweeps"]:
            line["roofline"]["fused_single_qubit_sweep"] = fused_single_qubit_sweep_probe(q, n, amp_bytes, peak)
        if world == 1 and not args.skip_cpu_baseline:
            cb = cpu_reference_sample(text, n, prec, args.cpu_sample_gates, 1, desc)
            line["cpu_baseline"] = {k: cb[k] for k in ("value", "unit", "cores", "kind", "sample")}
        if args.dump_outputs:
            import numpy as np
            os.makedirs(args.dump_outputs, exist_ok=True)
            np.save(os.path.join(args.dump_outputs, "state_sample.npy"), dumped_state)
            np.save(os.path.join(args.dump_outputs, "qubit_probs.npy"), np.asarray(probs, dtype=np.float64))
        print(json.dumps(line))
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
