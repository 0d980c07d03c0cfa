"""Parity of the CUDA path (through the C ABI, komb_b200.api -> libkombgpu.so)
against the CPU oracle and the reference-generated golden fixtures.

Bars (BASELINE.json north_star): edge list and per-unitig coreness bit-exact;
CORE-A within 6e-14 absolute of the scores of the exact ranks (oracle.check_corea)
with an identical anomaly ranking.
"""
import numpy as np
import pytest

from conftest import (corea_case_names, komb2_case_names, load_corea_case,
                      load_komb2_case)
from komb_b200 import synth

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ctx():
    import komb_b200
    c = komb_b200.Context(0)
    yield c
    c.close()


def check_graph_against_oracle(oracle, g, n, exp_edges):
    gn, gm = g.counts()
    assert (gn, gm) == (n, exp_edges.shape[0])
    u, v = g.edges()
    assert np.array_equal(oracle.pack_edges(u, v), exp_edges)            # edge list bit-exact, canonical order
    exp_deg, exp_core = oracle.coreness(n, exp_edges)
    assert np.array_equal(g.degree(), exp_deg)
    row_ptr, col = g.csr()
    assert np.array_equal(np.diff(row_ptr.astype(np.int64)), exp_deg)
    # CSR rows: ascending, symmetric closure of the edge list
    src = np.repeat(np.arange(n, dtype=np.uint64), exp_deg)
    keys = (src << np.uint64(32)) | col.astype(np.uint64)
    assert np.all(np.diff(keys.astype(np.int64)) > 0) if keys.size > 1 else True
    eu, ev = oracle.unpack_edges(exp_edges)
    sym = np.sort(np.concatenate([oracle.pack_edges(eu, ev), oracle.pack_edges(ev, eu)]))
    assert np.array_equal(keys, sym)
    core = g.coreness()
    assert np.array_equal(core, exp_core)                                  # coreness bit-exact
    return exp_deg, exp_core


def check_corea(oracle, got, core, deg, mode):
    # exact ranks, bit-identical scores for the same rank pair, identical anomaly ranking
    oracle.check_corea(got, core, deg, mode)


@pytest.mark.parametrize("name", komb2_case_names())
def test_golden_komb2_cases(ctx, oracle_mod, name):
    sam1, sam2, exp = load_komb2_case(name)
    rk, ut, names = oracle_mod.intern_hits([oracle_mod.tokenise_sam(sam1, exp["threads"]),
                                            oracle_mod.tokenise_sam(sam2, exp["threads"])])
    with ctx.build_graph(rk, ut, len(names)) as g:
        u, v = g.edges()
        got_edges = {tuple(sorted((names[a], names[b]))) for a, b in zip(u.tolist(), v.tolist())}
        assert got_edges == exp["edges"]
        core, deg = g.coreness(), g.degree()
        assert {names[i]: (int(core[i]), int(deg[i])) for i in range(len(names))} == exp["kcore"]
        score = g.corea()
        check_corea(oracle_mod, score, core, deg, oracle_mod.KEY_REF32)
        for i, nm in enumerate(names):      # the reference prints "%f"
            assert abs(score[i] - float(exp["score_text"][nm])) <= 5.0e-7 + 1e-12
        assert f"{score[i]:f}" is not None
        mc, ms = g.summary()
        assert f"Dense Ratio: {float(mc // 2):f}" in exp["stdout_info"]
        assert f"Max CoreA score: {ms:f}" in exp["stdout_info"]


@pytest.mark.parametrize("name", corea_case_names())
def test_golden_corea_cases(ctx, oracle_mod, name):
    core, deg, ref = load_corea_case(name)
    got = ctx.corea(core, deg)                       # ref32 keys, like the reference
    oracle_mod.check_corea(got, core, deg, oracle_mod.KEY_REF32, ranking=False)
    np.testing.assert_allclose(got, ref, rtol=0, atol=oracle_mod.COREA_ATOL)


@pytest.mark.parametrize("seed,n,n_pairs", [(0, 1000, 15000), (1, 50000, 400000), (2, 300000, 3000000)])
def test_hits_to_scores_vs_oracle(ctx, oracle_mod, seed, n, n_pairs):
    m1, m2 = synth.metagenome_hits(n, n_pairs, seed=seed)
    rk = np.concatenate([m1.read_key, m2.read_key])
    ut = np.concatenate([m1.unitig, m2.unitig])
    exp_edges, exp_p, exp_s = oracle_mod.build_edges(rk, ut)
    with ctx.build_graph(rk, ut, n) as g:
        deg, core = check_graph_against_oracle(oracle_mod, g, n, exp_edges)
        st = g.stats()
        assert (st["n_hits"], st["n_unique_hits"], st["n_pairs"], st["n_edges"]) == (rk.shape[0], exp_s, exp_p, exp_edges.shape[0])
        assert st["max_degree"] == deg.max() and st["max_coreness"] == core.max()
        for mode in (oracle_mod.KEY_REF32, oracle_mod.KEY_EXACT64):
            check_corea(oracle_mod, g.corea(mode), core, deg, mode)


@pytest.mark.parametrize("order", ["two_runs", "one_run", "shuffled", "two_runs_sort_forced", "long_read_in_order"])
def test_hit_orders_take_the_same_result(ctx, oracle_mod, monkeypatch, order):
    """The build merges the mate files when the reads come in file order (one or two runs of non-decreasing
    keys) and sorts otherwise, or when a read is too long for the look-back dedup: every route must give the
    reference's sets."""
    n, n_pairs = 20000, 150000
    m1, m2 = synth.metagenome_hits(n, n_pairs, seed=9)
    rk = np.concatenate([m1.read_key, m2.read_key])
    ut = np.concatenate([m1.unitig, m2.unitig])
    if order == "one_run":
        o = np.argsort(rk, kind="stable"); rk, ut = rk[o], ut[o]
    elif order == "shuffled":
        o = np.random.default_rng(1).permutation(rk.shape[0]); rk, ut = rk[o], ut[o]
    elif order == "two_runs_sort_forced":
        monkeypatch.setenv("KOMBGPU_NO_MERGE", "1")
    elif order == "long_read_in_order":   # read 77 gets 300 more hits (with repeats) in mate file 1, in place
        at = int(np.searchsorted(m1.read_key, 77))
        extra = np.random.default_rng(2).integers(0, 500, 300).astype(np.uint32)
        rk = np.concatenate([m1.read_key[:at], np.full(300, 77, np.uint32), m1.read_key[at:], m2.read_key])
        ut = np.concatenate([m1.unitig[:at], extra, m1.unitig[at:], m2.unitig])
    exp_edges, exp_p, exp_s = oracle_mod.build_edges(rk, ut)
    with ctx.build_graph(rk, ut, n) as g:
        check_graph_against_oracle(oracle_mod, g, n, exp_edges)
        st = g.stats()
        assert (st["n_unique_hits"], st["n_pairs"]) == (exp_s, exp_p)


def test_repeat_heavy_reads(ctx, oracle_mod):
    """A few reads with hundreds of hits (bwa -a on repeats): quadratic pair blow-up."""
    rng = np.random.default_rng(3)
    n = 5000
    rk = [np.full(700, 0), np.full(350, 1), np.repeat(np.arange(2, 2002), 2)]
    ut = [rng.integers(0, n, 700), rng.integers(0, 900, 350), rng.integers(0, n, 4000)]
    rk, ut = np.concatenate(rk).astype(np.uint32), np.concatenate(ut).astype(np.uint32)
    exp_edges, exp_p, _ = oracle_mod.build_edges(rk, ut)
    with ctx.build_graph(rk, ut, n) as g:
        check_graph_against_oracle(oracle_mod, g, n, exp_edges)
        assert g.stats()["n_pairs"] == exp_p


@pytest.mark.parametrize("seed,scale,n,m", [(0, 10, 900, 12000), (1, 16, 50000, 600000), (2, 20, 800000, 8000000)])
def test_rmat_edges_vs_oracle(ctx, oracle_mod, seed, scale, n, m):
    u, v = synth.rmat_edges(scale, m, n_vertices=n, seed=seed)
    exp_edges = oracle_mod.simplify(u, v)
    with ctx.graph_from_edges(u, v, n) as g:
        deg, core = check_graph_against_oracle(oracle_mod, g, n, exp_edges)
        check_corea(oracle_mod, g.corea(oracle_mod.KEY_EXACT64), core, deg, oracle_mod.KEY_EXACT64)
        check_corea(oracle_mod, g.corea(oracle_mod.KEY_REF32), core, deg, oracle_mod.KEY_REF32)


def test_deep_core_ramp(ctx, oracle_mod):
    """cfg5 in miniature: hundreds of dependent peeling levels."""
    levels, per = 400, 6
    u, v = synth.ramp_edges(levels, per)
    n = levels * per + 50                      # plus isolated vertices
    exp_edges = oracle_mod.simplify(u, v)
    with ctx.graph_from_edges(u, v, n) as g:
        _, core = check_graph_against_oracle(oracle_mod, g, n, exp_edges)
        st = g.stats()
        assert core.max() == levels == st["max_coreness"]
        assert st["peel_levels"] == len(set(core.tolist()))


@pytest.mark.parametrize("mode", ["warp", "cta"])
def test_peel_modes_hubs_and_wide_frontiers(ctx, oracle_mod, monkeypatch, mode):
    """Both process-phase variants of the peel kernel (KOMBGPU_PEEL_MODE) on shapes that exercise every task kind:
    hub rows above the pool-slice threshold (4096 edges), rows between the warp piece size and that threshold,
    a level-1 frontier wider than the statically dealt part, and a dense core behind long cascades."""
    monkeypatch.setenv("KOMBGPU_PEEL_MODE", mode)
    rng = np.random.default_rng(3)
    n = 400_000
    us, vs = [], []
    # two hubs with 150k and 9k leaves (coreness 1 leaves: one wide frontier), hubs tied into a clique
    us.append(np.zeros(150_000, np.uint32)); vs.append(np.arange(1000, 151_000, dtype=np.uint32))
    us.append(np.ones(9_000, np.uint32)); vs.append(np.arange(200_000, 209_000, dtype=np.uint32))
    iu, iv = np.triu_indices(60, k=1)
    us.append(iu.astype(np.uint32)); vs.append(iv.astype(np.uint32))          # K_60 on vertices 0..59
    # mid-size rows: 300 vertices with ~600 random neighbours each among 60..20000
    for c in range(300, 600):
        nb = rng.choice(np.arange(600, 20_000), size=600, replace=False).astype(np.uint32)
        us.append(np.full(600, c, np.uint32)); vs.append(nb)
    # sparse background
    us.append(rng.integers(0, n, 600_000).astype(np.uint32)); vs.append(rng.integers(0, n, 600_000).astype(np.uint32))
    u, v = np.concatenate(us), np.concatenate(vs)
    exp_edges = oracle_mod.simplify(u, v)
    with ctx.graph_from_edges(u, v, n) as g:
        deg, core = check_graph_against_oracle(oracle_mod, g, n, exp_edges)
        assert deg.max() > 100_000 and core.max() >= 59


def test_cfg2_full_size(ctx, oracle_mod):
    """BASELINE.json config 2 at its full size (1 M unitigs, 5 M read pairs, ~20 M hits): edge list, degree and
    coreness bit-exact against the CPU oracle, CORE-A within tolerance in both key modes."""
    n = 1_000_000
    m1, m2 = synth.metagenome_hits(n, 5_000_000, seed=11)
    rk = np.concatenate([m1.read_key, m2.read_key])
    ut = np.concatenate([m1.unitig, m2.unitig])
    exp_edges, exp_p, exp_s = oracle_mod.build_edges(rk, ut)
    exp_deg, exp_core = oracle_mod.coreness(n, exp_edges)
    with ctx.build_graph(rk, ut, n) as g:
        u, v = g.edges()
        assert np.array_equal(oracle_mod.pack_edges(u, v), exp_edges)
        assert np.array_equal(g.degree(), exp_deg) and np.array_equal(g.coreness(), exp_core)
        st = g.stats()
        assert (st["n_unique_hits"], st["n_pairs"], st["n_edges"]) == (exp_s, exp_p, exp_edges.shape[0])
        for mode in (oracle_mod.KEY_REF32, oracle_mod.KEY_EXACT64):
            check_corea(oracle_mod, g.corea(mode), exp_core, exp_deg, mode)
        assert g.densest_core() == oracle_mod.densest_core(exp_core, exp_edges)


def test_analyse_hits_one_call(ctx, oracle_mod):
    """kombgpu_analyse_hits (host hits in, all results out, edge download overlapped) gives what the staged calls
    give; too small edge buffers are an error, not a truncation."""
    import komb_b200
    n, n_pairs = 30000, 250000
    m1, m2 = synth.metagenome_hits(n, n_pairs, seed=4)
    rk = np.concatenate([m1.read_key, m2.read_key])
    ut = np.concatenate([m1.unitig, m2.unitig])
    exp_edges, _, _ = oracle_mod.build_edges(rk, ut)
    exp_deg, exp_core = oracle_mod.coreness(n, exp_edges)
    pin = {"u": ctx.pinned_empty(exp_edges.shape[0] + 10, np.uint32), "v": ctx.pinned_empty(exp_edges.shape[0] + 10, np.uint32)}
    for out in (None, pin):
        g, r = ctx.analyse_hits(rk, ut, n, oracle_mod.KEY_REF32, out=out)
        with g:
            assert np.array_equal(oracle_mod.pack_edges(r["u"], r["v"]), exp_edges)
            assert np.array_equal(r["degree"], exp_deg) and np.array_equal(r["coreness"], exp_core)
            check_corea(oracle_mod, r["score"], exp_core, exp_deg, oracle_mod.KEY_REF32)
            assert g.stats()["n_edges"] == exp_edges.shape[0]
    with pytest.raises(komb_b200.KombGpuError):
        ctx.analyse_hits(rk, ut, n, edge_capacity=exp_edges.shape[0] - 1)
    g, r = ctx.analyse_hits(np.zeros(0, np.uint32), np.zeros(0, np.uint32), 0)       # empty input
    with g:
        assert r["u"].shape == (0,) and r["score"].shape == (0,)


@pytest.mark.parametrize("n,lo,hi,srt", [
    (1_000_003, 20, 20, 0), (777_777, 20, 23, 1), (500_000, 0, 20, 0), (300_000, 26, 26, 0), (4097, 13, 3, 0),
    (100, 5, 0, 0), (1, 8, 8, 0), (2_000_000, 32, 32, 0),
    # from 2^30 keys on the passes take 64-bit status words: one 1-bit pass, where one digit holds more than 2^30 keys
    # (a count 32-bit words cannot hold); 5 passes over more than 2^17 tiles; the hits shape
    (2**31 + 12345, 1, 0, 0), (1_100_000_000, 20, 20, 0), (1_100_000_000, 20, 23, 1)])
def test_radix_sort_shapes(ctx, n, lo, hi, srt):
    """kombgpu_debug_sort_u64 gives a sorted permutation on the key shapes the path sorts (two key fields with a gap,
    digits that straddle it, narrow last digits, non-decreasing high field, one field only, a partial last tile, fewer
    keys than a tile, 2^30 keys and more)."""
    import ctypes
    from komb_b200 import _lib
    lib = _lib.load()
    ms, ok = ctypes.c_float(), ctypes.c_int()
    rc = lib.kombgpu_debug_sort_u64(ctx._h, n, lo, hi, srt, 1, ctypes.byref(ms), ctypes.byref(ok))
    if n >= 2**30:
        ctx.trim()   # up to 52 GB of keys and buffers: not left cached for the module's later tests
    assert rc == 0 and ok.value == 1, (n, lo, hi, srt, rc, ok.value)


def test_densest_core(ctx, oracle_mod):
    """kombgpu_graph_densest_core against the numpy checker, plus known answers: a K_40 planted in a sparse graph is
    the densest core (density 19.5 = C(40,2)/40); an empty graph gives level 0."""
    rng = np.random.default_rng(5)
    n = 30_000
    iu, iv = np.triu_indices(40, k=1)
    u = np.concatenate([iu + 100, rng.integers(0, n, 90_000)]).astype(np.uint32)
    v = np.concatenate([iv + 100, rng.integers(0, n, 90_000)]).astype(np.uint32)
    exp_edges = oracle_mod.simplify(u, v)
    with ctx.graph_from_edges(u, v, n) as g:
        core = g.coreness()
        got = g.densest_core()
        assert got == oracle_mod.densest_core(core, exp_edges)
        assert got["k"] == 39 and got["n_vertices"] == 40 and got["n_edges"] == 780 and got["density"] == 19.5
    us, vs = synth.rmat_edges(16, 600_000, n_vertices=50_000, seed=3)
    exp_edges = oracle_mod.simplify(us, vs)
    with ctx.graph_from_edges(us, vs, 50_000) as g:
        import komb_b200
        with pytest.raises(komb_b200.KombGpuError):      # needs the coreness first
            g.densest_core()
        core = g.coreness()
        assert g.densest_core() == oracle_mod.densest_core(core, exp_edges)
    with ctx.graph_from_edges(np.zeros(0, np.uint32), np.zeros(0, np.uint32), 7) as g:
        g.coreness()
        assert g.densest_core() == {"k": 0, "n_vertices": 7, "n_edges": 0, "density": 0.0}


def test_kats_and_edge_cases(ctx, oracle_mod):
    def run(n, pairs):
        u = np.array([p[0] for p in pairs], np.uint32)
        v = np.array([p[1] for p in pairs], np.uint32)
        with ctx.graph_from_edges(u, v, n) as g:
            return g.coreness().tolist(), g.degree().tolist(), g.counts()[1]
    k6 = [(i, j) for i in range(6) for j in range(i + 1, 6)]
    assert run(6, k6)[0] == [5] * 6
    assert run(5, [(i, i + 1) for i in range(4)])[0] == [1] * 5
    assert run(6, [(0, i) for i in range(1, 6)])[0] == [1] * 6
    assert run(5, [(i, (i + 1) % 5) for i in range(5)])[0] == [2] * 5
    assert run(8, k6 + [(6, 7)])[0] == [5] * 6 + [1, 1]
    assert run(3, [(0, 1), (1, 0), (0, 0), (0, 1)]) == ([1, 1, 0], [1, 1, 0], 1)   # dup, reversed, loop, isolated
    assert run(4, []) == ([0] * 4, [0] * 4, 0)                                       # no edges
    assert run(1, [(0, 0)]) == ([0], [0], 0)                                         # only a loop
    with ctx.build_graph(np.zeros(0, np.uint32), np.zeros(0, np.uint32), 0) as g:    # empty input
        assert g.counts() == (0, 0)
        assert g.coreness().shape == (0,) and g.corea().shape == (0,)
    # hits: single-unitig reads make vertices but no edges (degree-0 rows, quirk Q4)
    with ctx.build_graph(np.array([0, 1, 2, 2], np.uint32), np.array([0, 1, 2, 2], np.uint32), 3) as g:
        assert g.counts() == (3, 0)
        assert g.coreness().tolist() == [0, 0, 0]
        assert np.array_equal(g.corea(), np.zeros(3))


def test_errors_are_reported_not_swallowed(ctx):
    import komb_b200
    with pytest.raises(komb_b200.KombGpuError) as e:
        ctx.graph_from_edges(np.array([0, 7], np.uint32), np.array([1, 2], np.uint32), 5)   # id >= n
    assert e.value.code == -1
    with pytest.raises(komb_b200.KombGpuError):
        ctx.build_graph(np.array([0], np.uint32), np.array([9], np.uint32), 3)
    with ctx.graph_from_edges(np.array([0], np.uint32), np.array([1], np.uint32), 2) as g:
        with pytest.raises(komb_b200.KombGpuError) as e2:
            g.corea()                                                                         # before coreness
        assert e2.value.code == -5


def test_device_resident_inputs(ctx, oracle_mod):
    import torch
    u, v = synth.rmat_edges(14, 200000, n_vertices=12000, seed=9)
    exp_edges = oracle_mod.simplify(u, v)
    tu = torch.from_numpy(u.view(np.int32)).cuda()
    tv = torch.from_numpy(v.view(np.int32)).cuda()
    torch.cuda.synchronize()
    with ctx.graph_from_edges(tu, tv, 12000) as g:
        check_graph_against_oracle(oracle_mod, g, 12000, exp_edges)
        g.analyse()
        arr = g.device_arrays()
        assert all(arr[k] for k in ("row_ptr", "col", "edges_packed", "degree", "coreness", "score"))


def test_pinned_out_buffers(ctx, oracle_mod):
    u, v = synth.rmat_edges(12, 40000, n_vertices=3000, seed=4)
    exp_edges = oracle_mod.simplify(u, v)
    bu, bv = ctx.pinned_empty(50000, np.uint32), ctx.pinned_empty(50000, np.uint32)
    bc, bs = ctx.pinned_empty(3000, np.int32), ctx.pinned_empty(3000, np.float64)
    with ctx.graph_from_edges(u, v, 3000) as g:
        gu, gv = g.edges(out=(bu, bv))
        assert gu.base is not None and np.array_equal(oracle_mod.pack_edges(gu, gv), exp_edges)
        core = g.coreness(out=bc)
        assert np.array_equal(core, oracle_mod.coreness(3000, exp_edges)[1])
        s = g.corea(out=bs)
        assert s.shape == (3000,) and np.all(s >= 0)
        with pytest.raises(ValueError):
            g.degree(out=np.empty(10, np.int32))


def test_results_one_call(ctx, oracle_mod):
    """kombgpu_graph_results: everything the host writes, edge download overlapped with the peel."""
    m1, m2 = synth.metagenome_hits(30000, 90000, seed=8)
    rk = np.concatenate([m1.read_key, m2.read_key]); ut = np.concatenate([m1.unitig, m2.unitig])
    exp_edges, _, _ = oracle_mod.build_edges(rk, ut)
    exp_deg, exp_core = oracle_mod.coreness(30000, exp_edges)
    out = {"u": ctx.pinned_empty(exp_edges.shape[0] + 10, np.uint32), "v": ctx.pinned_empty(exp_edges.shape[0] + 10, np.uint32)}
    with ctx.build_graph(rk, ut, 30000) as g:
        r = g.results(out=out)
        assert np.array_equal(oracle_mod.pack_edges(r["u"], r["v"]), exp_edges)
        assert np.array_equal(r["degree"], exp_deg) and np.array_equal(r["coreness"], exp_core)
        check_corea(oracle_mod, r["score"], exp_core, exp_deg, oracle_mod.KEY_REF32)
        r2 = g.results(komb_b200_key_exact())       # second call: nothing is recomputed except CORE-A in the other key mode
        assert np.array_equal(r2["coreness"], exp_core)
        check_corea(oracle_mod, r2["score"], exp_core, exp_deg, oracle_mod.KEY_EXACT64)


def pair_multiplicity(rk, ut):
    """numpy restatement: per read the set of unitigs (src/graph.cpp:259-285), every i<j pair (:332-347);
    returns the canonical packed pairs that are not loops and how many reads emitted each."""
    key = np.unique((rk.astype(np.uint64) << np.uint64(32)) | ut.astype(np.uint64))
    r, u = key >> np.uint64(32), key & np.uint64(0xffffffff)
    starts = np.flatnonzero(np.r_[True, r[1:] != r[:-1]])
    ends = np.r_[starts[1:], len(r)]
    out = []
    for s, e in zip(starts.tolist(), ends.tolist()):
        if e - s >= 2:
            a = u[s:e]                                   # ascending: (a[i], a[j]), i<j is already (min, max)
            iu, iv = np.triu_indices(e - s, 1)
            out.append((a[iu] << np.uint64(32)) | a[iv])
    allp = np.concatenate(out) if out else np.zeros(0, np.uint64)
    return np.unique(allp, return_counts=True)


def test_edge_list_csr_form_and_multiplicity(ctx, oracle_mod):
    """kombgpu_graph_edges_csr / _results_csr / kombgpu_analyse_hits_csr give the canonical edge list as forward
    offsets + targets; kombgpu_graph_edge_multiplicity counts the pairs behind every edge (extension X1)."""
    n, n_pairs = 3000, 20000
    m1, m2 = synth.metagenome_hits(n, n_pairs, seed=6)
    rk = np.concatenate([m1.read_key, m2.read_key]); ut = np.concatenate([m1.unitig, m2.unitig])
    exp_edges, exp_p, _ = oracle_mod.build_edges(rk, ut)
    exp_deg, exp_core = oracle_mod.coreness(n, exp_edges)
    pk, cnt = pair_multiplicity(rk, ut)
    assert np.array_equal(pk, exp_edges) and int(cnt.sum()) == exp_p and cnt.max() > 1
    with ctx.build_graph(rk, ut, n) as g:
        fp, v = g.edges_csr()
        assert fp.shape == (n + 1,) and fp[0] == 0 and fp[-1] == exp_edges.shape[0]
        u = np.repeat(np.arange(n, dtype=np.uint32), np.diff(fp.astype(np.int64)))
        assert np.array_equal(oracle_mod.pack_edges(u, v), exp_edges)
        assert np.array_equal(g.edge_multiplicity(), cnt.astype(np.uint32))
        r = g.results_csr()
        assert np.array_equal(r["fwd_ptr"], fp) and np.array_equal(r["v"], v)
        assert np.array_equal(r["degree"], exp_deg) and np.array_equal(r["coreness"], exp_core)
    out = {"fwd_ptr": ctx.pinned_empty(n + 1, np.uint64), "v": ctx.pinned_empty(exp_edges.shape[0] + 7, np.uint32)}
    g, r = ctx.analyse_hits_csr(rk, ut, n, oracle_mod.KEY_REF32, out=out)
    with g:
        assert np.array_equal(r["fwd_ptr"], fp) and np.array_equal(r["v"], v)
        assert np.array_equal(r["coreness"], exp_core)
        check_corea(oracle_mod, r["score"], exp_core, exp_deg, oracle_mod.KEY_REF32)
    import komb_b200
    with pytest.raises(komb_b200.KombGpuError):
        ctx.analyse_hits_csr(rk, ut, n, edge_capacity=exp_edges.shape[0] - 1)
    # duplicate input pairs of an edge list count as multiplicity; loops do not make edges
    uu = np.array([0, 1, 0, 2, 2, 3], np.uint32); vv = np.array([1, 0, 1, 2, 3, 2], np.uint32)
    with ctx.graph_from_edges(uu, vv, 4) as g:
        eu, ev = g.edges()
        assert list(zip(eu.tolist(), ev.tolist())) == [(0, 1), (2, 3)]
        assert g.edge_multiplicity().tolist() == [3, 2]
        fp2, v2 = g.edges_csr()
        assert fp2.tolist() == [0, 1, 1, 2, 2] and v2.tolist() == [1, 3]


def test_adopted_csr_has_no_edge_list(ctx):
    """A graph adopted from a CSR holds no canonical edge list: every entry point that needs one says so
    (KOMBGPU_ESTATE) instead of reading a null pointer."""
    import torch
    import komb_b200
    row_ptr = torch.tensor([0, 2, 4, 6], dtype=torch.int64, device="cuda")
    col = torch.tensor([1, 2, 0, 2, 0, 1], dtype=torch.int32, device="cuda")
    with ctx.graph_from_csr(row_ptr, col, 3) as g:
        assert g.coreness().tolist() == [2, 2, 2]
        for call in (g.edges, g.edges_csr, g.edge_multiplicity, g.densest_core):
            with pytest.raises(komb_b200.KombGpuError) as e:
                call()
            assert e.value.code == -5


def test_two_contexts_in_one_process(oracle_mod):
    """Function attributes (dynamic shared memory of the radix passes) are per device and are set per context."""
    import torch
    import komb_b200
    devs = [0, 1] if torch.cuda.device_count() >= 2 else [0, 0]
    u, v = synth.rmat_edges(14, 100000, n_vertices=9000, seed=2)
    exp = oracle_mod.simplify(u, v)
    ctxs = [komb_b200.Context(d) for d in devs]
    try:
        for c in ctxs:
            with c.graph_from_edges(u, v, 9000) as g:
                gu, gv = g.edges()
                assert np.array_equal(oracle_mod.pack_edges(gu, gv), exp)
    finally:
        for c in ctxs:
            c.close()


def test_max_core_truss(ctx, oracle_mod):
    """kombgpu_graph_max_core_truss (reference Kgraph::runTruss, row N3) against the restatement in the oracle: the
    induced subgraph of the maximal core, the trussness of every edge, the unitigs of the maximal truss; plus known
    answers (K_7: every edge has trussness 7; a triangle-free core: trussness 2)."""
    import komb_b200
    cases = [synth.rmat_edges(11, 30000, n_vertices=1200, seed=2), synth.rmat_edges(14, 200000, n_vertices=9000, seed=5)]
    m1, m2 = synth.metagenome_hits(3000, 9000, seed=3)
    for i, (u, v) in enumerate(cases):
        n = 1200 if i == 0 else 9000
        edges = oracle_mod.simplify(u, v)
        _, core = oracle_mod.coreness(n, edges)
        exp = oracle_mod.max_core_truss(n, edges, core)
        with ctx.graph_from_edges(u, v, n) as g:
            with pytest.raises(komb_b200.KombGpuError):
                g.max_core_truss()                       # needs the coreness first
            g.coreness()
            got = g.max_core_truss()
        for key in ("n_core_vertices", "n_core_edges", "max_trussness"):
            assert got[key] == exp[key], key
        for key in ("u", "v", "trussness", "truss_vertices"):
            assert np.array_equal(got[key], exp[key]), key
    iu, iv = np.triu_indices(7, k=1)
    with ctx.graph_from_edges(iu.astype(np.uint32) + 3, iv.astype(np.uint32) + 3, 12) as g:      # K_7 on ids 3..9
        g.coreness()
        got = g.max_core_truss()
        assert (got["n_core_vertices"], got["n_core_edges"], got["max_trussness"]) == (7, 21, 7)
        assert got["trussness"].tolist() == [7] * 21 and got["truss_vertices"].tolist() == list(range(3, 10))
    ring = np.arange(8, dtype=np.uint32)
    with ctx.graph_from_edges(ring, (ring + 1) % 8, 8) as g:                                      # C_8: no triangles
        g.coreness()
        got = g.max_core_truss()
        assert got["max_trussness"] == 2 and got["trussness"].tolist() == [2] * 8 and got["truss_vertices"].tolist() == list(range(8))
    with ctx.graph_from_edges(np.zeros(0, np.uint32), np.zeros(0, np.uint32), 5) as g:            # no edges
        g.coreness()
        got = g.max_core_truss()
        assert (got["n_core_vertices"], got["n_core_edges"], got["max_trussness"]) == (5, 0, 0)


def komb_b200_key_exact():
    import komb_b200
    return komb_b200.KEY_EXACT64


def test_densest_block(ctx, oracle_mod):
    """kombgpu_graph_densest_block (the bulk form of CombineCoreA::runMerge's greedy peel) against the numpy checker:
    block, sizes, density and pass count identical -- unweighted, with exact (dyadic) weights, with the graph's own
    CORE-A scores (within rounding of the weight sums) -- plus known answers."""
    import komb_b200
    rng = np.random.default_rng(17)
    for seed, scale, m, n in [(1, 12, 30_000, 3000), (2, 16, 600_000, 50_000), (3, 18, 2_000_000, 200_000)]:
        us, vs = synth.rmat_edges(scale, m, n_vertices=n, seed=seed)
        exp_edges = oracle_mod.simplify(us, vs)
        w = rng.integers(0, 8192, n).astype(np.float64) / 1024.0      # every partial sum is exact in double
        with ctx.graph_from_edges(us, vs, n) as g:
            for weight, eps in ((None, 0.5), (None, 0.0), (w, 0.5), (w, 0.05)):
                got = g.densest_block(weight=weight, eps=eps)
                exp = oracle_mod.densest_block_bulk(n, exp_edges, weight, eps)
                assert np.array_equal(got["member"], exp["member"])
                assert {k: got[k] for k in ("n_vertices", "n_edges", "weight_sum", "density", "passes")} == \
                       {k: exp[k] for k in ("n_vertices", "n_edges", "weight_sum", "density", "passes")}
            with pytest.raises(komb_b200.KombGpuError):           # the scores do not exist yet
                g.densest_block(use_scores=True)
            g.coreness(); score = g.corea()
            got = g.densest_block(use_scores=True, eps=0.5)
            exp = oracle_mod.densest_block_bulk(n, exp_edges, score, 0.5)
            assert got["n_vertices"] == exp["n_vertices"] and got["n_edges"] == exp["n_edges"] and got["passes"] == exp["passes"]
            np.testing.assert_allclose(got["density"], exp["density"], rtol=1e-12)
            with pytest.raises(komb_b200.KombGpuError):
                g.densest_block(weight=-w)
    # a K_40 planted in a sparse graph is the densest block: density 19.5
    iu, iv = np.triu_indices(40, k=1)
    u = np.concatenate([iu + 100, rng.integers(0, 30_000, 60_000)]).astype(np.uint32)
    v = np.concatenate([iv + 100, rng.integers(0, 30_000, 60_000)]).astype(np.uint32)
    with ctx.graph_from_edges(u, v, 30_000) as g:
        got = g.densest_block(eps=0.1)
        assert got["density"] >= 19.5 and set(np.flatnonzero(got["member"])) >= set(range(100, 140))
    with ctx.graph_from_edges(np.zeros(0, np.uint32), np.zeros(0, np.uint32), 7) as g:
        got = g.densest_block()
        assert got["n_vertices"] == 7 and got["density"] == 0.0 and got["passes"] == 1 and got["member"].all()
    with ctx.graph_from_edges(np.zeros(0, np.uint32), np.zeros(0, np.uint32), 0) as g:
        assert g.densest_block()["n_vertices"] == 0


def test_corea_histogram_path_equals_sort_path(ctx, oracle_mod, monkeypatch):
    """CORE-A ranks from the 2-D (coreness, degree) histogram (small key spaces, the default there) and from the sort of
    (key, vertex) are the same doubles; both against the oracle."""
    rng = np.random.default_rng(23)
    cases = [(rng.integers(0, 38, 200_000), rng.integers(0, 300, 200_000)),          # cfg2-like: 38 x 300 bins (shared memory)
             (rng.integers(0, 400, 300_000), rng.integers(0, 9000, 300_000)),        # 3.6 M bins (global counters)
             (np.zeros(1000, np.int64), np.zeros(1000, np.int64)),                   # one class
             (np.arange(5000) % 7, np.arange(5000) % 11)]
    for core, deg in cases:
        core, deg = core.astype(np.int32), np.maximum(deg, core).astype(np.int32)
        for mode in (oracle_mod.KEY_REF32, oracle_mod.KEY_EXACT64):
            monkeypatch.delenv("KOMBGPU_COREA_SORT", raising=False)
            a = ctx.corea(core, deg, mode)
            monkeypatch.setenv("KOMBGPU_COREA_SORT", "1")
            b = ctx.corea(core, deg, mode)
            monkeypatch.delenv("KOMBGPU_COREA_SORT", raising=False)
            assert np.array_equal(a, b)
            # (no ranking identity against the CPU here: random (coreness, degree) pairs give thousands of near-tied
            # scores whose order turns on the last bit of log(); the graph-derived cases above hold that bar)
            oracle_mod.check_corea(a, core, deg, mode, ranking=False)
