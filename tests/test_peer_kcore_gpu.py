"""The consumers of the finished coreness on the partitioned graph (kombgpu_dist_max_core_truss,
kombgpu_dist_densest_core): every rank's answer must equal the single-GPU Graph's on the whole input, bit for bit, and
the CPU oracle's (oracle.max_core_truss, oracle.densest_core).

On a one-GPU box the ranks are emulated (threads of one process, all on device 0, exchanges done by the host
threads); with >= 2 GPUs the same comparisons also run with one GPU per rank."""
import functools
import threading

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

CASES = ["hits_mid", "rmat", "ramp", "hubs", "empty", "k7_planted", "triangle_free", "core_on_rank0", "k4_rank_without_vertices"]
TRUSS_KEYS = ("n_core_vertices", "n_core_edges", "max_trussness", "u", "v", "trussness", "truss_vertices")


@functools.lru_cache(maxsize=None)
def _whole(case):
    """(kind, n, a, b): the whole input of a case (hits: read keys / unitigs; else u / v)."""
    from komb_b200 import synth
    rng = np.random.default_rng(17)
    if case == "hits_mid":
        m1, m2 = synth.metagenome_hits(40000, 120000, seed=5)
        return "hits", 40000, np.concatenate([m1.read_key, m2.read_key]), np.concatenate([m1.unitig, m2.unitig])
    if case == "rmat":
        u, v = synth.rmat_edges(18, 1500000, n_vertices=150000, seed=7)
        return "pairs", 150000, u, v
    if case == "ramp":       # hundreds of dependent levels, ids scrambled so every rank owns a share of every level
        u, v = synth.ramp_edges(300, 5)
        n = 300 * 5 + 37
        return "pairs", n, synth.scramble_ids(u, n), synth.scramble_ids(v, n)
    if case == "hubs":       # two hubs, a K_50 and a random background
        n = 200_000
        iu, iv = np.triu_indices(50, k=1)
        u = np.concatenate([np.zeros(60_000), np.full(9_000, 1), iu, rng.integers(0, n, 400_000)]).astype(np.uint32)
        v = np.concatenate([np.arange(1000, 61_000), np.arange(100_000, 109_000), iv, rng.integers(0, n, 400_000)]).astype(np.uint32)
        return "pairs", n, synth.scramble_ids(u, n), synth.scramble_ids(v, n)
    if case == "empty":
        return "pairs", 10, np.zeros(0, np.uint32), np.zeros(0, np.uint32)
    if case in ("k7_planted", "core_on_rank0"):
        # a K_7 in a sparse background (coreness <= 3 there): the maximal core is the K_7, trussness 7 on every edge.
        # k7_planted scatters its ids over the ranks; core_on_rank0 keeps them in [0, 7), so only rank 0 owns any of it
        n = 6000
        iu, iv = np.triu_indices(7, k=1)
        u = np.concatenate([iu, rng.integers(0, n, 4000)]).astype(np.uint32)
        v = np.concatenate([iv, rng.integers(0, n, 4000)]).astype(np.uint32)
        if case == "k7_planted":
            u, v = synth.scramble_ids(u, n), synth.scramble_ids(v, n)
        return "pairs", n, u, v
    if case == "triangle_free":   # K_{5,5} (coreness 5, no triangle) over a random forest: trussness 2 everywhere
        n = 3000
        a, b = np.meshgrid(np.arange(5), np.arange(5, 10))
        child = np.arange(10, n)
        u = np.concatenate([a.ravel(), child]).astype(np.uint32)
        v = np.concatenate([b.ravel(), rng.integers(0, child)]).astype(np.uint32)
        return "pairs", n, synth.scramble_ids(u, n), synth.scramble_ids(v, n)
    if case == "k4_rank_without_vertices":   # n = 4: with 3 ranks the last one owns no unitig at all
        iu, iv = np.triu_indices(4, k=1)
        return "pairs", 4, iu.astype(np.uint32), iv.astype(np.uint32)
    raise KeyError(case)


def _share(case, rank, world):
    kind, n, a, b = _whole(case)
    if kind == "hits":     # a read's hits stay on one rank: split by read range
        reads = int(a.max()) + 1 if a.size else 0
        sel = (a >= reads * rank // world) & (a < reads * (rank + 1) // world)
        return kind, n, a[sel], b[sel]
    sl = slice(len(a) * rank // world, len(a) * (rank + 1) // world)
    return kind, n, a[sl], b[sl]


@functools.lru_cache(maxsize=None)
def _expected(oracle, case):
    """The single-GPU Graph's answers on the whole input, checked against the oracle once per case."""
    import komb_b200
    kind, n, a, b = _whole(case)
    ctx = komb_b200.Context(0)
    try:
        with (ctx.build_graph(a, b, n) if kind == "hits" else ctx.graph_from_edges(a, b, n)) as g:
            core = g.coreness()
            truss, dense = g.max_core_truss(), g.densest_core()
    finally:
        ctx.close()
    edges = oracle.build_edges(a, b)[0] if kind == "hits" else oracle.simplify(a, b)
    exp_core = oracle.coreness(n, edges)[1]
    assert np.array_equal(core, exp_core)
    _assert_truss_equal(truss, oracle.max_core_truss(n, edges, exp_core))
    assert dense == oracle.densest_core(exp_core, edges)
    return truss, dense


def _assert_truss_equal(got, exp):
    for key in TRUSS_KEYS:
        if isinstance(exp[key], np.ndarray):
            assert got[key].dtype == exp[key].dtype and np.array_equal(got[key], exp[key]), key
        else:
            assert got[key] == exp[key], key


def _rank_body(comm, case):
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
        truss = g.max_core_truss()
        again = g.max_core_truss()      # cached: no second exchange
        dense = g.densest_core()
        st = g.stats()
    return {"truss": truss, "again": again, "dense": dense, "n_local": st["n_local"], "peel": st["peel_async"]}


def _check(oracle, case, parts):
    truss, dense = _expected(oracle, case)
    for p in parts:
        _assert_truss_equal(p["truss"], truss)
        _assert_truss_equal(p["again"], truss)
        assert p["dense"] == dense


@pytest.mark.parametrize("world", [1, 2, 3])
@pytest.mark.parametrize("case", CASES)
def test_dist_kcore_consumers_emulated_ranks(oracle_mod, monkeypatch, case, world):
    from komb_b200.peer import run_local
    monkeypatch.delenv("KOMBGPU_DIST_PEEL", raising=False)
    parts = run_local(world, lambda comm: _rank_body(comm, case))
    _check(oracle_mod, case, parts)
    truss, _ = _expected(oracle_mod, case)
    if case in ("k7_planted", "core_on_rank0"):
        assert truss["max_trussness"] == 7 and truss["n_core_edges"] == 21 and set(truss["trussness"].tolist()) == {7}
    if case == "triangle_free":
        assert truss["n_core_edges"] == 25 and set(truss["trussness"].tolist()) == {2}
    if case == "k4_rank_without_vertices":
        assert truss["max_trussness"] == 4
        if world == 3:
            assert parts[2]["n_local"] == 0


@pytest.mark.parametrize("peel", ["async", "log", "replicated"])
def test_dist_kcore_consumers_any_build_layout(oracle_mod, monkeypatch, peel):
    """The build lays the adjacency out for the peel it prepares for; the consumers read only the edge list and the
    coreness, so the layout must not show in the result."""
    from komb_b200.peer import run_local
    monkeypatch.setenv("KOMBGPU_DIST_PEEL", peel)
    parts = run_local(3, lambda comm: _rank_body(comm, "hubs"))
    assert {p["peel"] for p in parts} == {{"log": 0, "async": 1, "replicated": 2}[peel]}
    _check(oracle_mod, "hubs", parts)


def test_dist_kcore_consumers_need_the_coreness():
    """Before the coreness every rank gets KOMBGPU_ESTATE from both calls and from the getters, and none waits."""
    import torch
    import komb_b200
    from komb_b200._lib import ESTATE
    from komb_b200.peer import DistGraph, run_local

    def body(comm):
        _, n, a, b = _share("k7_planted", comm.rank, comm.world)
        ta, tb = torch.from_numpy(a.view(np.int32).copy()).cuda(), torch.from_numpy(b.view(np.int32).copy()).cuda()
        codes = []
        with DistGraph.from_pairs(comm, ta, tb, n) as g:
            for call in (g.max_core_truss, g.densest_core, g.truss_timing):
                try:
                    call()
                    codes.append(0)
                except komb_b200.KombGpuError as e:
                    codes.append(e.code)
        return codes

    out = {}
    t = threading.Thread(target=lambda: out.setdefault("codes", run_local(3, body)), daemon=True)
    t.start()
    t.join(timeout=300)
    assert not t.is_alive(), "a rank is still waiting"
    assert out["codes"] == [[ESTATE] * 3] * 3


@pytest.mark.parametrize("case", ["hits_mid", "rmat", "hubs", "core_on_rank0"])
def test_dist_kcore_consumers_one_gpu_per_rank(oracle_mod, monkeypatch, case):
    """Real peer access: one GPU per rank, ranks are threads of this process."""
    import torch
    from komb_b200.peer import run_local
    n_dev = torch.cuda.device_count()
    if n_dev < 2:
        pytest.skip("needs >= 2 GPUs")
    monkeypatch.delenv("KOMBGPU_DIST_PEEL", raising=False)
    world = min(n_dev, 4)
    parts = run_local(world, lambda comm: _rank_body(comm, case), devices=list(range(world)))
    _check(oracle_mod, case, parts)
