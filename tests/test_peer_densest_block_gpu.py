"""The densest block on the partitioned graph (kombgpu_dist_densest_block): every rank's sizes, weight sum, density
and passes must equal the single-GPU Graph.densest_block on the whole input bit for bit, the ranks' member slices
concatenated in rank order must equal its member mask, and both must equal the CPU oracle's
(oracle.densest_block_bulk).  Weights are dyadic, so every partial sum is exact in double whatever the order of the
additions; the graph's own CORE-A scores are held to the bar of the single-GPU test (sizes and passes equal, density
within rounding).

On a one-GPU box the ranks are emulated (threads of one process, all on device 0, exchanges done by the host
threads); with >= 2 GPUs the same comparisons also run with one GPU per rank."""
import functools
import threading

import numpy as np
import pytest

from test_peer_kcore_gpu import CASES, _share, _whole

pytestmark = pytest.mark.gpu

BLOCK_KEYS = ("n_vertices", "n_edges", "weight_sum", "density", "passes")
MODES = ((False, 0.5), (False, 0.0), (True, 0.5), (True, 0.05))   # (weighted, eps)


def _input(case):
    """(kind, n, a, b): the nine shapes of test_peer_kcore_gpu plus a K_40 whose ids are scattered over the ranks."""
    if case != "k40_scattered":
        return _whole(case)
    from komb_b200 import synth
    rng = np.random.default_rng(29)
    n = 30_000
    iu, iv = np.triu_indices(40, k=1)
    u = np.concatenate([iu + 100, rng.integers(0, n, 60_000)]).astype(np.uint32)
    v = np.concatenate([iv + 100, rng.integers(0, n, 60_000)]).astype(np.uint32)
    return "pairs", n, synth.scramble_ids(u, n), synth.scramble_ids(v, n)


def _part(case, rank, world):
    if case != "k40_scattered":
        return _share(case, rank, world)
    kind, n, a, b = _input(case)
    sl = slice(len(a) * rank // world, len(a) * (rank + 1) // world)
    return kind, n, a[sl], b[sl]


@functools.lru_cache(maxsize=None)
def _weight(case):
    n = _input(case)[1]
    return np.random.default_rng(101).integers(0, 8192, n).astype(np.float64) / 1024.0


def _mode_weight(case, weighted):
    return _weight(case) if weighted else None


@functools.lru_cache(maxsize=None)
def _expected(oracle, case):
    """The single-GPU Graph's answers on the whole input, one per weight mode, then with its CORE-A scores; the weight
    modes are checked against the oracle once per case."""
    import komb_b200
    kind, n, a, b = _input(case)
    ctx = komb_b200.Context(0)
    try:
        with (ctx.build_graph(a, b, n) if kind == "hits" else ctx.graph_from_edges(a, b, n)) as g:
            modes = [g.densest_block(weight=_mode_weight(case, wt), eps=eps) for wt, eps in MODES]
            g.analyse()
            scores = g.densest_block(use_scores=True, eps=0.5)
    finally:
        ctx.close()
    edges = oracle.build_edges(a, b)[0] if kind == "hits" else oracle.simplify(a, b)
    for (wt, eps), got in zip(MODES, modes):
        exp = oracle.densest_block_bulk(n, edges, _mode_weight(case, wt), eps)
        assert np.array_equal(got["member"], exp["member"])
        assert {k: got[k] for k in BLOCK_KEYS} == {k: exp[k] for k in BLOCK_KEYS}
    return modes, scores


def _rank_body(comm, case):
    """Every weight mode right after the build, the CORE-A scores after analyse(), then every weight mode again in
    the reverse order: each call starts afresh."""
    import torch
    from komb_b200.peer import DistGraph
    kind, n, a, b = _part(case, comm.rank, comm.world)
    dev = torch.device("cuda", comm.ctx.device)
    ta = torch.from_numpy(a.view(np.int32).copy()).to(dev)
    tb = torch.from_numpy(b.view(np.int32).copy()).to(dev)
    torch.cuda.synchronize(dev)
    build = DistGraph.from_hits if kind == "hits" else DistGraph.from_pairs
    with build(comm, ta, tb, n) as g:
        st = g.stats()
        lo, hi = st["v_lo"], st["v_lo"] + st["n_local"]

        def call(weighted, eps):
            w = _weight(case)[lo:hi] if weighted else None
            return g.densest_block(weight=w, eps=eps)

        fresh = [call(*m) for m in MODES]
        g.analyse()
        scores = g.densest_block(use_scores=True, eps=0.5)
        again = [call(*m) for m in reversed(MODES)][::-1]
        st = g.stats()
    return {"fresh": fresh, "scores": scores, "again": again, "n_local": st["n_local"], "v_lo": st["v_lo"],
            "peel": st["peel_async"]}


def _assert_block_equal(parts, exp):
    for p in parts:
        assert {k: p[k] for k in BLOCK_KEYS} == {k: exp[k] for k in BLOCK_KEYS}
    member = np.concatenate([p["member"] for p in parts])
    assert member.dtype == bool and np.array_equal(member, exp["member"])


def _check(oracle, case, parts):
    modes, scores = _expected(oracle, case)
    for i, exp in enumerate(modes):
        _assert_block_equal([p["fresh"][i] for p in parts], exp)
        _assert_block_equal([p["again"][i] for p in parts], exp)
    for p in parts:
        got = p["scores"]
        assert (got["n_vertices"], got["n_edges"], got["passes"]) == (scores["n_vertices"], scores["n_edges"], scores["passes"])
        np.testing.assert_allclose(got["density"], scores["density"], rtol=1e-12)
    # every rank holds the same scalars, bit for bit, also with the scores
    assert len({(p["scores"]["density"], p["scores"]["weight_sum"]) for p in parts}) == 1
    assert np.concatenate([p["scores"]["member"] for p in parts]).sum() == scores["n_vertices"]


@pytest.mark.parametrize("world", [1, 2, 3])
@pytest.mark.parametrize("case", CASES + ["k40_scattered"])
def test_dist_densest_block_emulated_ranks(oracle_mod, monkeypatch, case, world):
    from komb_b200.peer import run_local
    monkeypatch.delenv("KOMBGPU_DIST_PEEL", raising=False)
    parts = run_local(world, lambda comm: _rank_body(comm, case))
    _check(oracle_mod, case, parts)
    if case == "k40_scattered":   # the planted K_40 (density 19.5) is the densest block, whichever ranks own its ids
        n = _input(case)[1]
        from komb_b200 import synth
        k40 = synth.scramble_ids(np.arange(100, 140, dtype=np.uint32), n)
        member = np.concatenate([p["fresh"][0]["member"] for p in parts])
        assert parts[0]["fresh"][0]["density"] >= 19.5 and member[k40].all()
        if world == 3:   # every rank owns a share of it
            assert {int(x) // (n // 3) for x in k40} == {0, 1, 2}
    if case == "k4_rank_without_vertices" and world == 3:
        assert parts[2]["n_local"] == 0


@pytest.mark.parametrize("peel", ["async", "log", "replicated"])
def test_dist_densest_block_any_build_layout(oracle_mod, monkeypatch, peel):
    """The update step reads the adjacency in the layout the build left: grouped by neighbour (log) or as rows (async,
    replicated; a replicated build keeps its hubs' long rows).  The layout must not show in the result."""
    from komb_b200.peer import run_local
    monkeypatch.setenv("KOMBGPU_DIST_PEEL", peel)
    parts = run_local(3, lambda comm: _rank_body(comm, "hubs"))
    assert {p["peel"] for p in parts} == {{"log": 0, "async": 1, "replicated": 2}[peel]}
    _check(oracle_mod, "hubs", parts)


def test_dist_densest_block_errors_reach_every_rank(oracle_mod):
    """Bad arguments on some ranks give an error on every rank, none of them waits, and the graph stays usable."""
    import torch
    import komb_b200
    from komb_b200._lib import EINVAL, ESTATE
    from komb_b200.peer import DistGraph, run_local
    case = "k7_planted"

    def body(comm):
        _, n, a, b = _part(case, comm.rank, comm.world)
        ta, tb = torch.from_numpy(a.view(np.int32).copy()).cuda(), torch.from_numpy(b.view(np.int32).copy()).cuda()
        codes = []
        with DistGraph.from_pairs(comm, ta, tb, n) as g:
            st = g.stats()
            ok = np.ones(st["n_local"], np.float64)
            bad_neg, bad_nan = ok.copy(), ok.copy()
            bad_neg[0], bad_nan[0] = -1.0, np.nan
            mine = comm.rank == 1
            calls = [dict(use_scores=True),                                   # before CORE-A
                     dict(weight=bad_neg if mine else ok),                    # a negative weight on rank 1 only
                     dict(weight=bad_nan if mine else ok),                    # a NaN weight on rank 1 only
                     dict(weight=ok, use_scores=True),                        # weights and scores together
                     dict(eps=0.5 + 0.125 * comm.rank),                       # eps differs between the ranks
                     dict(eps=-1.0 if comm.rank == 0 else 0.5)]               # eps out of range on rank 0 only
            for kw in calls:
                try:
                    g.densest_block(**kw)
                    codes.append(0)
                except komb_b200.KombGpuError as e:
                    codes.append(e.code)
            after = g.densest_block(weight=_weight(case)[st["v_lo"]:st["v_lo"] + st["n_local"]], eps=0.05)
        return codes, after

    out = {}
    t = threading.Thread(target=lambda: out.setdefault("res", run_local(3, body)), daemon=True)
    t.start()
    t.join(timeout=300)
    assert not t.is_alive(), "a rank is still waiting"
    codes = [r[0] for r in out["res"]]
    assert [c[0] for c in codes] == [ESTATE] * 3
    for i in (1, 2):
        assert codes[1][i] == EINVAL and codes[0][i] != 0 and codes[2][i] != 0
    assert [c[3] for c in codes] == [EINVAL] * 3
    assert [c[4] for c in codes] == [EINVAL] * 3
    assert codes[0][5] == EINVAL and codes[1][5] != 0 and codes[2][5] != 0
    modes, _ = _expected(oracle_mod, case)
    _assert_block_equal([r[1] for r in out["res"]], modes[3])


@pytest.mark.parametrize("case", ["hits_mid", "rmat", "hubs"])
def test_dist_densest_block_one_gpu_per_rank(oracle_mod, monkeypatch, case):
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
