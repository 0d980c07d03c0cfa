"""The peer-memory multi-GPU path (kombgpu_comm_* / kombgpu_dist_*: partitioned build, device-driven peel over
mailboxes, sharded CORE-A) against the CPU oracle.

On a one-GPU box the ranks run in EMULATION: threads of one process, all on device 0; exchanges are done by the
host threads and the peel runs every rank's share inside one cooperative grid (kernels of different ranks must
never wait for one another on one GPU).  Same data path — routing, offsets, mailboxes, sub-round protocol — minus
the spin on a peer's flag.  With >= 2 GPUs the same cases also run with one GPU per rank, as threads (peer
access) and as processes (cudaIpc, bootstrap over torch.distributed / NCCL)."""
import os
import pickle
import socket
import sys
from pathlib import Path

import numpy as np
import pytest

ROOT = Path(__file__).resolve().parents[1]
pytestmark = pytest.mark.gpu

CASES = {
    "hits_small": (3000, 9000, 3, "hits"),
    "hits_mid": (40000, 120000, 5, "hits"),
    "rmat": (150000, 1500000, 7, "pairs"),
    "ramp": (0, 0, 0, "ramp"),
    "hubs": (0, 0, 0, "hubs"),
    "empty": (10, 0, 0, "hits"),
}


def _whole(case):
    """(kind, n, a, b): the whole input of a case (hits: read keys / unitigs; else u / v)."""
    from komb_b200 import synth
    n, reads, seed, kind = CASES[case]
    if kind == "hits":
        if reads == 0:
            return "hits", n, np.zeros(0, np.uint32), np.zeros(0, np.uint32)
        m1, m2 = synth.metagenome_hits(n, reads, seed=seed)
        return "hits", n, np.concatenate([m1.read_key, m2.read_key]), np.concatenate([m1.unitig, m2.unitig])
    if kind == "pairs":
        u, v = synth.rmat_edges(18, reads, n_vertices=n, seed=seed)
        return "pairs", n, u, v
    if kind == "ramp":       # hundreds of dependent levels, ids scrambled so every rank owns a share of every level
        u, v = synth.ramp_edges(300, 5)
        n = 300 * 5 + 37
        return "pairs", n, synth.scramble_ids(u, n), synth.scramble_ids(v, n)
    rng = np.random.default_rng(3)   # hubs: rows far above the slice length, a wide level-1 frontier, a dense core
    n = 200_000
    us = [np.zeros(60_000, np.uint32), np.full(9_000, 1, np.uint32)]
    vs = [np.arange(1000, 61_000, dtype=np.uint32), np.arange(100_000, 109_000, dtype=np.uint32)]
    iu, iv = np.triu_indices(50, k=1)
    us.append(iu.astype(np.uint32)); vs.append(iv.astype(np.uint32))
    us.append(rng.integers(0, n, 400_000).astype(np.uint32)); vs.append(rng.integers(0, n, 400_000).astype(np.uint32))
    u, v = np.concatenate(us), np.concatenate(vs)
    return "pairs", n, synth.scramble_ids(u, n), synth.scramble_ids(v, n)


def _share(case, rank, world):
    kind, n, a, b = _whole(case)
    if kind == "hits":     # a read's hits stay on one rank: split by read range
        reads = int(a.max()) + 1 if a.size else 0
        lo, hi = reads * rank // world, reads * (rank + 1) // world
        sel = (a >= lo) & (a < hi)
        return kind, n, a[sel], b[sel]
    sl = slice(len(a) * rank // world, len(a) * (rank + 1) // world)
    return kind, n, a[sl], b[sl]


def _expected(oracle, case):
    kind, n, a, b = _whole(case)
    edges = oracle.build_edges(a, b)[0] if kind == "hits" else oracle.simplify(a, b)
    deg, core = oracle.coreness(n, edges)
    return n, edges, deg, core


def _rank_body(comm, case, key_mode):
    import torch
    from komb_b200.peer import DistGraph
    kind, n, a, b = _share(case, comm.rank, comm.world)
    dev = torch.device("cuda", comm.ctx.device)
    ta = torch.from_numpy(a.view(np.int32).copy()).to(dev)
    tb = torch.from_numpy(b.view(np.int32).copy()).to(dev)
    torch.cuda.synchronize(dev)
    build = DistGraph.from_hits if kind == "hits" else DistGraph.from_pairs
    with build(comm, ta, tb, n) as g:
        g.coreness()
        g.corea(key_mode)
        r = g.results()
        u, v, mult = g.edges(with_mult=True)
        st = g.stats()
        mc, ms = g.summary()
    return {"v_lo": r["v_lo"], "deg": r["degree"], "core": r["coreness"], "score": r["score"], "u": u, "v": v, "mult": mult,
            "stats": st, "max_core": mc, "max_score": ms, "same_device": comm.same_device}


def _check(oracle, parts, case, key_mode):
    n, edges, deg, core = _expected(oracle, case)
    parts = sorted(parts, key=lambda p: p["stats"]["v_lo"] if p["stats"]["n_local"] else 1 << 40)
    assert np.array_equal(np.concatenate([p["deg"] for p in parts]), deg)
    assert np.array_equal(np.concatenate([p["core"] for p in parts]), core)                     # coreness bit-exact
    got_edges = oracle.pack_edges(np.concatenate([p["u"] for p in parts]), np.concatenate([p["v"] for p in parts]))
    assert np.array_equal(got_edges, edges)               # the ranks' slices concatenate to the canonical sorted edge list
    score = np.concatenate([p["score"] for p in parts])
    oracle.check_corea(score, core, deg, key_mode)            # exact ranks, identical ranking
    rd, rk = oracle.corea_ranks(core, deg, key_mode)
    exp_max = float(np.abs(np.log(rd) - np.log(rk)).max()) if n else 0.0
    for p in parts:
        assert p["stats"]["n_edges_global"] == edges.shape[0]
        assert p["max_core"] == (int(core.max()) if n else 0)
        assert abs(p["max_score"] - exp_max) <= oracle.COREA_ATOL
    return parts


@pytest.mark.parametrize("peel", ["async", "log", "replicated", "auto"])
@pytest.mark.parametrize("world", [1, 2, 3])
@pytest.mark.parametrize("case", ["hits_small", "hits_mid", "rmat", "ramp", "hubs", "empty"])
def test_peer_path_emulated_ranks(oracle_mod, monkeypatch, case, world, peel):
    """peel: the asynchronous peel (apeel.cu: remote atomics on the owners' degrees, discoveries pushed into the owners'
    pools, ranks meet once per level), the log-based one (ppeel.cu: ranks meet once per cascade generation), the
    replicated one (rpeel.cu: every rank pulls the others' rows and peels the whole graph), or the library's choice."""
    from komb_b200.peer import run_local
    monkeypatch.setenv("KOMBGPU_DIST_PEEL", peel)
    key_mode = oracle_mod.KEY_EXACT64 if case in ("rmat", "ramp") else oracle_mod.KEY_REF32
    parts = run_local(world, lambda comm: _rank_body(comm, case, key_mode))
    parts = _check(oracle_mod, parts, case, key_mode)
    if world > 1:
        assert all(p["same_device"] for p in parts)
        kinds = {p["stats"]["peel_async"] for p in parts}
        assert kinds == {{"log": 0, "async": 1, "replicated": 2, "auto": 2}[peel]}      # small graphs: auto replicates
        if case in ("hits_mid", "rmat", "hubs") and peel in ("async", "log"):
            assert sum(p["stats"]["n_messages_sent"] for p in parts) == sum(p["stats"]["n_messages_recv"] for p in parts) > 0
    if case == "hits_small":      # multiplicities survive the routing: their sum is the number of pairs emitted
        assert sum(int(p["mult"].sum()) for p in parts) == sum(p["stats"]["n_pairs_local"] for p in parts)


def test_peer_path_bad_input_fails_on_every_rank():
    """An out-of-range unitig id on ONE rank is reported by every rank (nobody is left waiting in an exchange)."""
    import torch
    import komb_b200
    from komb_b200.peer import DistGraph, run_local

    def body(comm):
        u = torch.tensor([0, 1, 2 if comm.rank else 99], dtype=torch.int32, device="cuda")
        v = torch.tensor([1, 2, 3], dtype=torch.int32, device="cuda")
        try:
            DistGraph.from_pairs(comm, u, v, 10)
        except komb_b200.KombGpuError as e:
            return e.code
        return 0
    assert run_local(2, body) == [-1, -1]


@pytest.mark.parametrize("world", [2, 3])
def test_peer_path_bad_corea_mode_fails_on_every_rank(oracle_mod, world):
    """A CORE-A key mode that only rank 1 gets wrong is KOMBGPU_EINVAL on every rank; then CORE-A runs again on the same
    graph and gives the exact scores (the communicator and its symmetric heap are usable after the failure)."""
    import torch
    import komb_b200
    from komb_b200._lib import EINVAL
    from komb_b200.peer import DistGraph, run_local
    key = oracle_mod.KEY_REF32

    def body(comm):
        _, n, a, b = _share("hits_small", comm.rank, comm.world)
        dev = torch.device("cuda", comm.ctx.device)
        ta = torch.from_numpy(a.view(np.int32).copy()).to(dev)
        tb = torch.from_numpy(b.view(np.int32).copy()).to(dev)
        torch.cuda.synchronize(dev)
        with DistGraph.from_hits(comm, ta, tb, n) as g:
            g.coreness()
            code = 0
            try:
                g.corea(7 if comm.rank == 1 else key)
            except komb_b200.KombGpuError as e:
                code = e.code
            g.corea(key)
            return code, g.results()

    out = run_local(world, body)
    assert [code for code, _ in out] == [EINVAL] * world
    _, _, deg, core = _expected(oracle_mod, "hits_small")
    parts = sorted((r for _, r in out), key=lambda r: r["v_lo"])
    assert np.array_equal(np.concatenate([r["degree"] for r in parts]), deg)
    assert np.array_equal(np.concatenate([r["coreness"] for r in parts]), core)
    oracle_mod.check_corea(np.concatenate([r["score"] for r in parts]), core, deg, key)


@pytest.mark.parametrize("peel", ["async", "log", "replicated"])
@pytest.mark.parametrize("case", ["hits_mid", "rmat", "ramp", "hubs"])
def test_peer_path_one_gpu_per_rank_threads(oracle_mod, monkeypatch, case, peel):
    """Real peer access: one GPU per rank, ranks are threads of this process (what a C++ host like komb2 does)."""
    import torch
    from komb_b200.peer import run_local
    monkeypatch.setenv("KOMBGPU_DIST_PEEL", peel)
    n_dev = torch.cuda.device_count()
    if n_dev < 2:
        pytest.skip("needs >= 2 GPUs")
    world = min(n_dev, 4)
    key_mode = oracle_mod.KEY_EXACT64 if case in ("rmat", "ramp") else oracle_mod.KEY_REF32
    parts = run_local(world, lambda comm: _rank_body(comm, case, key_mode), devices=list(range(world)))
    parts = _check(oracle_mod, parts, case, key_mode)
    assert not any(p["same_device"] for p in parts)


def _proc_worker(rank, world, port, out_dir, case, key_mode):
    sys.path.insert(0, str(ROOT))
    import torch
    import torch.distributed as dist
    import komb_b200
    from komb_b200.peer import Comm
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    ctx = komb_b200.Context(rank)
    comm = Comm.from_torch(ctx)
    out = _rank_body(comm, case, key_mode)
    with open(Path(out_dir) / f"rank{rank}.pkl", "wb") as f:
        pickle.dump(out, f)
    dist.barrier()
    comm.close()
    ctx.close()
    dist.destroy_process_group()


@pytest.mark.parametrize("peel", ["async", "log", "replicated"])
@pytest.mark.parametrize("case", ["hits_mid", "rmat"])
def test_peer_path_one_process_per_gpu_nccl_bootstrap(tmp_path, oracle_mod, monkeypatch, case, peel):
    """The bench's arrangement: one process per GPU, symmetric heap mapped with cudaIpc, bootstrap all-gather
    over torch.distributed with the NCCL backend."""
    import torch
    import torch.multiprocessing as mp
    n_dev = torch.cuda.device_count()
    if n_dev < 2:
        pytest.skip("needs >= 2 GPUs")
    world = 2
    monkeypatch.setenv("KOMBGPU_DIST_PEEL", peel)      # inherited by the spawned ranks
    key_mode = oracle_mod.KEY_EXACT64 if case == "rmat" else oracle_mod.KEY_REF32
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    mp.spawn(_proc_worker, args=(world, port, str(tmp_path), case, key_mode), nprocs=world, join=True)
    parts = [pickle.load(open(tmp_path / f"rank{r}.pkl", "rb")) for r in range(world)]
    _check(oracle_mod, parts, case, key_mode)
