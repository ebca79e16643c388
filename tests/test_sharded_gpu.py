"""Multi-GPU parity (needs >= 2 CUDA devices; skipped otherwise): QEngineSharded over QEngineCUDA local engines + NCCL
all-to-all must reproduce the single-engine oracle state."""
import os
import random

import numpy as np
import pytest

from oracle.restate_engine import QEngineRestate
from qrack_b200 import qscript

import util
from test_sharded_cpu import _free_port

pytestmark = pytest.mark.gpu


def _ngpu():
    try:
        import torch
        return torch.cuda.device_count()
    except Exception:
        return 0


def _worker(rank, world, port, text, prec, out_path, mode):
    import torch
    import torch.distributed as dist
    p2p = mode != "nccl"
    os.environ["B200SV_SHARD_PULL"] = "1" if mode in ("pull", "pull_carry") else "0"
    os.environ["B200SV_SHARD_VIRT"] = "1" if mode == "pull_carry" else "0"   # rank bits as virtual qubits + tail carry across exchanges
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    try:
        from qrack_b200.sharded import QEngineSharded, cuda_engine_factory

        def make(n, perm):
            return QEngineSharded(n, perm, random.Random(1), 1.0 + 0j, precision=prec, dist=dist, world=world, rank=rank,
                                  device=torch.device("cuda", rank), make_engine=cuda_engine_factory(rank, prec), p2p=p2p)
        regs, results = qscript.run(text, make)
        st = regs[0].GetQuantumState()
        if rank == 0:
            np.savez(out_path, state=st, exchanges=regs[0].be.exchanges, pull_sweeps=regs[0].be.shard.stats().get("pull_sweeps", 0),
                     carried=regs[0].be.carried_ops)
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("mode", ["nccl", "push", "pull", "pull_carry"],
                         ids=["nccl_all_to_all", "p2p_scatter_kernel", "p2p_pull_fused_into_sweep", "p2p_pull_and_tail_carry"])
@pytest.mark.parametrize("prec", [32, 64])
def test_sharded_nccl_matches_oracle(prec, mode, tmp_path):
    world = 2 if _ngpu() < 4 else 4
    if _ngpu() < 2:
        pytest.skip("needs >= 2 GPUs")
    import torch.multiprocessing as mp
    text = qscript.random_htcnot(18, 12, seed=8, timed=False)
    want, _ = util.run_engine(text, QEngineRestate, prec)
    out = str(tmp_path / "o.npz")
    for attempt in range(3):  # the rendezvous port can be taken between probing and binding
        try:
            mp.spawn(_worker, args=(world, _free_port(), text, prec, out, mode), nprocs=world, join=True)
            break
        except Exception as e:
            if "EADDRINUSE" not in str(e) or attempt == 2:
                raise
    z = np.load(out)
    d = float(np.abs(z["state"].astype(np.complex128) - want[0].astype(np.complex128)).max())
    assert d <= util.AMP_TOL[prec], (d, "ops carried across exchanges: %d" % int(z["carried"]))
    assert int(z["exchanges"]) >= 1
    if mode != "pull_carry":
        assert int(z["carried"]) == 0         # gates are specialised per rank on these routes: nothing may cross an exchange
    if mode in ("pull", "pull_carry"):
        assert int(z["pull_sweeps"]) >= 1     # the re-page really rode on a fused sweep (b200sv_exchange_pull)
    else:
        assert int(z["pull_sweeps"]) == 0


def _worker_queries(rank, world, port, text, prec, out_path):
    import torch
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    try:
        from qrack_b200.sharded import QEngineSharded, cuda_engine_factory

        def make(n, perm):
            return QEngineSharded(n, perm, random.Random(1), 1.0 + 0j, precision=prec, dist=dist, world=world, rank=rank,
                                  device=torch.device("cuda", rank), make_engine=cuda_engine_factory(rank, prec), p2p=True)
        regs, results = qscript.run(text, make)
        q = regs[0]
        q.UpdateRunningNorm()
        nrm = q.GetRunningNorm()
        perm = q.MAll()                       # on-device sampling across the shards, then collapse
        amp = q.GetAmplitude(perm)
        if rank == 0:
            np.savez(out_path, results=np.array([v for _, vals in results for v in vals], dtype=np.float64), norm=nrm, perm=perm,
                     amp=abs(amp), exchanges=q.be.exchanges)
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("kind", ["htcnot", "qv", "grover"])
def test_sharded_26q_against_the_compiled_reference(kind, tmp_path):
    """BASELINE.md §3 'Parity': the sharded path at 26 qubits over every GPU of the box (8 ranks on the 8-GPU box) against the
    compiled reference QEngineCPU: all per-qubit Prob, 48 sampled amplitudes (1e-6), the norm, and a sharded MAll.  The circuits and
    the reference's results are stored in tests/golden/reference (make_golden.py sharded_26q_text)."""
    ng = _ngpu()
    if ng < 2:
        pytest.skip("needs >= 2 GPUs")
    world = 8 if ng >= 8 else (4 if ng >= 4 else 2)
    n = 26
    ref = util.load_reference("sharded_26q_%s_f32" % kind)
    text = ref["text"]
    want = np.array([v for _, vals in qscript.parse_results(ref["results"]) for v in vals], dtype=np.float64)
    # the fp32 reference sums each Prob (2^25 terms) in fp32 per worker thread with a dynamic work split: its own value wanders by
    # ~1e-4 from run to run.  The per-qubit probabilities are therefore taken from the fp64 build of the reference (same circuit).
    want_p = np.array([v for _, vals in qscript.parse_results(ref["results_f64"]) for v in vals], dtype=np.float64)[:n]
    import torch.multiprocessing as mp
    out = str(tmp_path / "o.npz")
    for attempt in range(3):
        try:
            mp.spawn(_worker_queries, args=(world, _free_port(), text, 32, out), nprocs=world, join=True)
            break
        except Exception as e:
            if "EADDRINUSE" not in str(e) or attempt == 2:
                raise
    z = np.load(out)
    got = z["results"]
    assert got.shape == want.shape
    assert np.abs(got[n:] - want[n:]).max() <= util.AMP_TOL[32], np.abs(got[n:] - want[n:]).max()   # amplitudes (re, im pairs): the parity bar
    # Prob (ours: fp32 state, double accumulation) against the fp64 reference: what is left is the fp32 state's own rounding
    assert np.abs(got[:n] - want_p).max() <= 2e-5, np.abs(got[:n] - want_p).max()
    assert abs(float(z["norm"]) - 1.0) < 1e-4 and float(z["amp"]) > 0.999
