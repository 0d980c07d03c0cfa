"""CORE-A on the device held to the oracle's exact ranks (oracle.check_corea: 6e-14 absolute, rank-pair ties
bit-identical) on every key path: the 2-D histogram (shared and global counters), the packed sort, the wide two-pass
exact64 sort, ref32 keys that wrap, degrees >= n, and the sharded ranks of kombgpu_dist_corea.

Each host-array case sits at one edge of a branch in corea.cu and runs in both key modes, with the histogram path
allowed and with KOMBGPU_COREA_SORT forcing the sort.  G_wrap is one graph whose keys reach every hard corner at
once: ref32 keys that wrap onto each other and below zero, and an exact64 key space of 33 bits."""
import ctypes
from functools import lru_cache

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

MODES = {"ref32": 0, "exact64": 1}


@pytest.fixture(scope="module")
def ctx():
    import komb_b200
    c = komb_b200.Context(0)
    yield c
    c.close()


def _realistic(rng, n):
    """Degrees below n, coreness <= degree."""
    deg = rng.integers(0, n, n) if n > 1 else np.zeros(n, np.int64)
    return rng.integers(0, deg + 1), deg


def _case(name):
    rng = np.random.default_rng(list(name.encode()))
    if name.startswith("n_"):
        return _realistic(rng, int(name[2:]))
    if name == "bins_12288":            # (95 + 1) x (127 + 1) pair bins: the most the shared-memory counters hold
        n = 50_000
        core, deg = rng.integers(0, 96, n), rng.integers(0, 128, n)
        core[0], deg[0] = 95, 127
    elif name == "bins_12289":          # one bin more: global counters
        n = 50_000
        core, deg = np.zeros(n, np.int64), rng.integers(0, 12289, n)
        deg[0] = 12288
    elif name == "bins_2^22":           # 1024 x 4096 bins: the largest histogram
        n = 200_000
        core, deg = rng.integers(0, 1024, n), rng.integers(0, 4096, n)
        core[0], deg[0] = 1023, 4095
    elif name == "bins_2^22+1":         # 5 x 838861 bins: the sort
        n = 1_000_000
        core, deg = rng.integers(0, 5, n), rng.integers(0, 838861, n)
        core[0], deg[0] = 4, 838860
    elif name in ("key_2^31-1", "key_2^31"):   # max coreness * n + max degree: the last ref32 key that does not wrap / the first that does
        n = 2_097_151                          # 1024 * n = 2^31 - 1024
        top = 1023 if name == "key_2^31-1" else 1024
        core, deg = rng.integers(0, 1025, n), rng.integers(0, top + 1, n)
        core[:3], deg[:3] = 1024, top
    elif name in ("deg_4095", "deg_4096"):     # the largest degree counted in shared memory / the first in global memory
        n = 10_000
        core, deg = rng.integers(0, 21, n), rng.integers(0, 4000, n)
        deg[:10] = 4095
        if name == "deg_4096":
            deg[10:20] = 4096
    elif name == "one_class":
        core, deg = np.full(1000, 3), np.full(1000, 5)
    elif name == "all_distinct":
        i = np.arange(4096)
        core, deg = i // 64, i % 64
    elif name == "deg_ge_n_example":   # exact64: keys [5, 4, 1, 2], not the pair order (0, 5) < (1, 0)
        core, deg = np.array([0, 1, 0, 0]), np.array([5, 0, 1, 2])
    elif name == "deg_ge_n_random":
        n = 1000
        core, deg = rng.integers(0, 51, n), rng.integers(0, 5001, n)
        core[:5], deg[:5] = 0, n + 3        # the same exact64 key as (1, 3)
        core[5:10], deg[5:10] = 1, 3
    elif name == "deg_ge_n_wide":        # normalised pair needs 26 + 10 bits: the wide exact64 sort with degrees >= n
        n = 1000
        core, deg = rng.integers(0, 2 ** 25, n), rng.integers(0, 2 ** 20, n)
        core[:4], deg[:4] = 5, 3 * n + 7    # the same exact64 key as (8, 7)
        core[4:8], deg[4:8] = 8, 7
    elif name == "wide":                 # 22 + 17 bits: the wide exact64 sort; ref32 wraps everywhere
        n = 100_000
        core, deg = rng.integers(0, 2 ** 22, n), rng.integers(0, n, n)
    elif name == "ref32_wrap_ties":      # 2049 * 2^21 + 50 wraps to 1 * 2^21 + 50: one ref32 class of two pairs
        n = 2 ** 21
        core = rng.integers(0, 10, n)
        deg = core + rng.integers(0, 90, n)
        core[:1000], deg[:1000] = 2049, 50
        core[1000:2000], deg[1000:2000] = 1, 50
        core[2000:2100], deg[2000:2100] = 1099, 1099
    else:
        raise KeyError(name)
    return core, deg


HOST_CASES = ["bins_12288", "bins_12289", "bins_2^22", "bins_2^22+1", "key_2^31-1", "key_2^31", "deg_4095", "deg_4096",
              "n_1", "n_2", "n_31", "n_33", "n_4095", "n_4097", "n_8191", "n_8193", f"n_{2 ** 20 + 1}",
              "one_class", "all_distinct", "deg_ge_n_example", "deg_ge_n_random", "deg_ge_n_wide", "wide", "ref32_wrap_ties"]


def _exp_max(oracle_mod, core, deg, mode):
    rd, rk = oracle_mod.corea_ranks(core, deg, mode)
    return float(np.abs(np.log(rd) - np.log(rk)).max()) if core.size else 0.0


@lru_cache(maxsize=None)
def _host_case(name):
    core, deg = _case(name)
    return core.astype(np.int32), deg.astype(np.int32)


def _corea_dev(ctx, core, deg, mode):
    """kombgpu_corea_dev on device copies of the arrays: (scores, max score)."""
    import torch
    from komb_b200 import _lib
    n = core.shape[0]
    tc, td = torch.from_numpy(core).cuda(), torch.from_numpy(deg).cuda()
    ts = torch.empty(n, dtype=torch.float64, device="cuda")
    mx = ctypes.c_double()
    ctx._check(_lib.load().kombgpu_corea_dev(ctx._h, ctypes.c_void_p(tc.data_ptr()), ctypes.c_void_p(td.data_ptr()), n, mode,
                                             ctypes.c_void_p(ts.data_ptr()), ctypes.byref(mx)))
    return ts.cpu().numpy(), mx.value


@pytest.mark.parametrize("mode", list(MODES))
@pytest.mark.parametrize("case", HOST_CASES)
def test_host_arrays_exact(ctx, oracle_mod, monkeypatch, case, mode):
    """kombgpu_corea and kombgpu_corea_dev, histogram allowed and sort forced: exact ranks, the same doubles on every
    path, and the maximum."""
    core, deg = _host_case(case)
    m = MODES[mode]
    monkeypatch.delenv("KOMBGPU_COREA_SORT", raising=False)
    a = ctx.corea(core, deg, m)
    oracle_mod.check_corea(a, core, deg, m, ranking=False)
    a_dev, a_max = _corea_dev(ctx, core, deg, m)
    assert np.array_equal(a_dev, a) and a_max == a.max()
    assert abs(a_max - _exp_max(oracle_mod, core, deg, m)) <= oracle_mod.COREA_ATOL
    monkeypatch.setenv("KOMBGPU_COREA_SORT", "1")
    b = ctx.corea(core, deg, m)
    assert np.array_equal(b, a)


# ---- G_wrap: one graph with wrapping ref32 keys and a 33-bit exact64 key space -------------------------------------
N_WRAP = 2 ** 21


@lru_cache(maxsize=None)
def _g_wrap():
    """(u, v) of G_wrap on N_WRAP vertices:
    K_2050 on 0..2049, and 100 leaves on vertex 0 (coreness 2049, degree 2149: ref32 key 2^21 + 2149 after the wrap);
    a star of 2149 leaves (centre: coreness 1, degree 2149, the same ref32 key);
    K_1100 (coreness 1099: ref32 keys below zero);
    a hub of 2^20 leaves (degree 2^20: 21 + 12 bits of exact64 key, the wide sort).  About 3.8 M edges."""
    parts = []
    iu, iv = np.triu_indices(2050, k=1)
    parts.append((iu, iv))
    nxt = 2050
    parts.append((np.zeros(100, np.int64), np.arange(nxt, nxt + 100))); nxt += 100
    parts.append((np.full(2149, nxt), np.arange(nxt + 1, nxt + 2150))); nxt += 2150
    iu, iv = np.triu_indices(1100, k=1)
    parts.append((iu + nxt, iv + nxt)); nxt += 1100
    parts.append((np.full(2 ** 20, nxt), np.arange(nxt + 1, nxt + 1 + 2 ** 20))); nxt += 1 + 2 ** 20
    assert nxt <= N_WRAP
    u = np.concatenate([p[0] for p in parts]).astype(np.uint32)
    v = np.concatenate([p[1] for p in parts]).astype(np.uint32)
    return u, v


@lru_cache(maxsize=None)
def _g_wrap_expected(oracle_mod):
    u, v = _g_wrap()
    edges = oracle_mod.simplify(u, v)
    deg, core = oracle_mod.coreness(N_WRAP, edges)
    return edges, deg, core


def test_g_wrap_keys(oracle_mod):
    """G_wrap has what it is built for."""
    edges, deg, core = _g_wrap_expected(oracle_mod)
    assert edges.shape[0] == 3_755_500
    assert (core[0], deg[0]) == (2049, 2149) and (core[2150], deg[2150]) == (1, 2149)
    rd, rk = oracle_mod.corea_ranks(core, deg, oracle_mod.KEY_REF32)
    assert rk[0] == rk[2150]
    key32 = (core.astype(np.int64) * N_WRAP + deg) & 0xFFFFFFFF
    assert (key32 >= 2 ** 31).any()
    assert int(deg.max()).bit_length() + int(core.max()).bit_length() > 32


@pytest.mark.parametrize("mode", list(MODES))
def test_g_wrap_graph(ctx, oracle_mod, mode):
    """g.corea, g.results, g.results_csr (each on a fresh graph, so each runs CORE-A itself) and g.summary."""
    u, v = _g_wrap()
    edges, deg, core = _g_wrap_expected(oracle_mod)
    m = MODES[mode]
    exp_max = _exp_max(oracle_mod, core, deg, m)
    with ctx.graph_from_edges(u, v, N_WRAP) as g:
        assert np.array_equal(g.coreness(), core) and np.array_equal(g.degree(), deg)
        oracle_mod.check_corea(g.corea(m), core, deg, m)
        mc, ms = g.summary()
        assert mc == 2049 and abs(ms - exp_max) <= oracle_mod.COREA_ATOL
    with ctx.graph_from_edges(u, v, N_WRAP) as g:
        r = g.results(m)
        assert np.array_equal(oracle_mod.pack_edges(r["u"], r["v"]), edges)
        assert np.array_equal(r["coreness"], core) and np.array_equal(r["degree"], deg)
        oracle_mod.check_corea(r["score"], core, deg, m)
        assert abs(g.summary()[1] - exp_max) <= oracle_mod.COREA_ATOL
    with ctx.graph_from_edges(u, v, N_WRAP) as g:
        r = g.results_csr(m)
        assert r["fwd_ptr"][-1] == edges.shape[0]
        assert np.array_equal(r["coreness"], core) and np.array_equal(r["degree"], deg)
        oracle_mod.check_corea(r["score"], core, deg, m)


# ---- sharded: kombgpu_dist_corea over emulated ranks ---------------------------------------------------------------
WORLDS = [1, 2, 3, 4, 5, 8]


def _whole(case):
    if case == "g_wrap":
        u, v = _g_wrap()
        return "pairs", N_WRAP, u, v
    if case == "n5":                      # five vertices: at world 8 some ranks own none
        return "pairs", 5, np.array([0, 1, 2, 3, 0], np.uint32), np.array([1, 2, 3, 4, 2], np.uint32)
    from test_peer_gpu import _whole as peer_whole
    return peer_whole(case)


@lru_cache(maxsize=None)
def _sharded_expected(oracle_mod, case):
    kind, n, a, b = _whole(case)
    edges = oracle_mod.build_edges(a, b)[0] if kind == "hits" else oracle_mod.simplify(a, b)
    deg, core = oracle_mod.coreness(n, edges)
    return n, deg, core


def _rank_body(comm, case, key_mode):
    import torch
    from komb_b200.peer import DistGraph
    kind, n, a, b = _whole(case)
    rank, world = comm.rank, comm.world
    if kind == "hits":                     # a read's hits stay on one rank
        reads = int(a.max()) + 1 if a.size else 0
        sel = (a >= reads * rank // world) & (a < reads * (rank + 1) // world)
        a, b = a[sel], b[sel]
    else:
        sl = slice(len(a) * rank // world, len(a) * (rank + 1) // world)
        a, b = a[sl], b[sl]
    dev = torch.device("cuda", comm.ctx.device)
    ta = torch.from_numpy(a.view(np.int32).copy()).to(dev)
    tb = torch.from_numpy(b.view(np.int32).copy()).to(dev)
    torch.cuda.synchronize(dev)
    build = DistGraph.from_hits if kind == "hits" else DistGraph.from_pairs
    with build(comm, ta, tb, n) as g:
        g.coreness()
        g.corea(key_mode)
        r = g.results()
        st = g.stats()
        mc, ms = g.summary()
    return {"deg": r["degree"], "core": r["coreness"], "score": r["score"], "stats": st, "max_core": mc, "max_score": ms}


@pytest.mark.parametrize("mode", list(MODES))
@pytest.mark.parametrize("world", WORLDS)
@pytest.mark.parametrize("case", ["g_wrap", "hits_small", "hits_mid", "rmat", "ramp", "hubs", "empty"])
def test_sharded_exact(oracle_mod, monkeypatch, case, world, mode):
    """Every rank's scores from the merged lists of distinct keys equal the whole graph's exact scores.  The peel is
    pinned to the replicated one, which every world size runs alike; the coreness is checked all the same."""
    from komb_b200.peer import run_local
    monkeypatch.setenv("KOMBGPU_DIST_PEEL", "replicated")
    m = MODES[mode]
    n, deg, core = _sharded_expected(oracle_mod, case)
    parts = run_local(world, lambda comm: _rank_body(comm, case, m))
    parts = sorted(parts, key=lambda p: p["stats"]["v_lo"] if p["stats"]["n_local"] else 1 << 40)
    assert np.array_equal(np.concatenate([p["deg"] for p in parts]), deg)
    assert np.array_equal(np.concatenate([p["core"] for p in parts]), core)
    score = np.concatenate([p["score"] for p in parts])
    oracle_mod.check_corea(score, core, deg, m)
    exp_max = _exp_max(oracle_mod, core, deg, m)
    for p in parts:
        assert p["max_core"] == (int(core.max()) if n else 0) and abs(p["max_score"] - exp_max) <= oracle_mod.COREA_ATOL


@pytest.mark.parametrize("mode", list(MODES))
def test_sharded_ranks_that_own_nothing(oracle_mod, monkeypatch, mode):
    from komb_b200.peer import run_local
    monkeypatch.setenv("KOMBGPU_DIST_PEEL", "replicated")
    m = MODES[mode]
    n, deg, core = _sharded_expected(oracle_mod, "n5")
    parts = run_local(8, lambda comm: _rank_body(comm, "n5", m))
    assert sum(p["stats"]["n_local"] for p in parts) == 5 and any(p["stats"]["n_local"] == 0 for p in parts)
    parts = sorted(parts, key=lambda p: p["stats"]["v_lo"] if p["stats"]["n_local"] else 1 << 40)
    assert np.array_equal(np.concatenate([p["core"] for p in parts]), core)
    score = np.concatenate([p["score"] for p in parts])
    oracle_mod.check_corea(score, core, deg, m)
    exp_max = _exp_max(oracle_mod, core, deg, m)
    assert all(abs(p["max_score"] - exp_max) <= oracle_mod.COREA_ATOL for p in parts)
