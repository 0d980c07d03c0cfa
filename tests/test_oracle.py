"""Pin the CPU oracle (oracle/) against the reference's own outputs
(tests/golden, produced by tests/golden/make_golden.py from komb2_ref /
CoreA.h) and against independent implementations (networkx, scipy)."""
import networkx as nx
import numpy as np
import pytest
import scipy.stats

from conftest import (corea_case_names, komb2_case_names, load_corea_case,
                      load_komb2_case)
from komb_b200 import synth


@pytest.mark.parametrize("name", komb2_case_names())
def test_oracle_matches_reference_komb2(oracle_mod, name):
    sam1, sam2, exp = load_komb2_case(name)
    got = oracle_mod.komb2_expected(sam1, sam2, threads=exp["threads"])
    assert got["edges"] == exp["edges"]                       # edge set bit-exact by Name
    assert got["kcore"] == exp["kcore"]                       # Name -> (coreness, degree)
    for nm, txt in exp["score_text"].items():                 # %f text: 6 decimals
        assert abs(got["score"][nm] - float(txt)) <= 5.0e-7 + 1e-12


def test_q1_line_drop_is_modelled(oracle_mod):
    """-t 4 on the same input loses lines (graph.cpp:206-220); -t 1 does not."""
    sam1, sam2, exp = load_komb2_case("mid_s3_t4")
    t1 = oracle_mod.komb2_expected(sam1, sam2, threads=1)
    assert exp["edges"] < t1["edges"]


@pytest.mark.parametrize("name", corea_case_names())
def test_oracle_corea_matches_reference_header(oracle_mod, name):
    core, deg, ref = load_corea_case(name)
    got = oracle_mod.corea(core, deg, oracle_mod.KEY_REF32)
    np.testing.assert_allclose(got, ref, rtol=1e-6, atol=1e-12)
    # ranks are exact half-integers: the only slack is libm log (<= 1 ulp each)
    assert np.max(np.abs(got - ref)) < 1e-13


def test_oracle_corea_overflow_modes_differ(oracle_mod):
    core, deg, ref = load_corea_case("overflow_q5_n40000")
    exact = oracle_mod.corea(core, deg, oracle_mod.KEY_EXACT64)
    assert np.max(np.abs(exact - ref)) > 1.0      # quirk Q5: the reference wraps int32


def test_oracle_ranks_equal_scipy(oracle_mod):
    rng = np.random.default_rng(0)
    deg = rng.integers(0, 50, 5000).astype(np.int32)
    core = np.minimum(deg, rng.integers(0, 9, 5000)).astype(np.int32)
    rd, rk = oracle_mod.corea_ranks(core, deg, oracle_mod.KEY_EXACT64)
    key = core.astype(np.int64) * 5000 + deg
    assert np.array_equal(rd, scipy.stats.rankdata(-deg.astype(np.int64), "average"))
    assert np.array_equal(rk, scipy.stats.rankdata(-key, "average"))


@pytest.mark.parametrize("seed", [0, 1, 2])
def test_oracle_coreness_equals_networkx(oracle_mod, seed):
    u, v = synth.rmat_edges(10, 12000, n_vertices=900, seed=seed)
    edges = oracle_mod.simplify(u, v)
    deg, core = oracle_mod.coreness(900, edges)
    eu, ev = oracle_mod.unpack_edges(edges)
    g = nx.Graph()
    g.add_nodes_from(range(900))
    g.add_edges_from(zip(eu.tolist(), ev.tolist()))
    cn = nx.core_number(g)
    assert [cn[i] for i in range(900)] == core.tolist()
    assert [g.degree(i) for i in range(900)] == deg.tolist()


def test_oracle_kats(oracle_mod):
    def core_of(n, pairs):
        u = np.array([p[0] for p in pairs], np.uint32)
        v = np.array([p[1] for p in pairs], np.uint32)
        return oracle_mod.coreness(n, oracle_mod.simplify(u, v))[1].tolist()
    k6 = [(i, j) for i in range(6) for j in range(i + 1, 6)]
    assert core_of(6, k6) == [5] * 6                                   # K_k -> k-1
    assert core_of(5, [(i, i + 1) for i in range(4)]) == [1] * 5       # path
    assert core_of(6, [(0, i) for i in range(1, 6)]) == [1] * 6        # star
    assert core_of(5, [(i, (i + 1) % 5) for i in range(5)]) == [2] * 5  # ring
    assert core_of(8, k6 + [(6, 7)] ) == [5] * 6 + [1, 1]              # disjoint
    assert core_of(3, [(0, 1), (1, 0), (0, 0), (0, 1)]) == [1, 1, 0]   # dup, loop, isolated


def test_oracle_ramp_has_many_levels(oracle_mod):
    u, v = synth.ramp_edges(levels=40, per_level=8)
    n = 40 * 8
    deg, core = oracle_mod.coreness(n, oracle_mod.simplify(u, v))
    assert core.max() >= 40
    # the closing clique swallows the last (levels+1)/per_level levels; all others are present
    assert set(range(1, 40 - 41 // 8)) <= set(core.tolist())


def test_build_edges_semantics(oracle_mod):
    # read 0: mate1 {5, 3}, mate2 {3, 9} -> set {3,5,9}; read 1: {7}; read 2 (mate2 only): {1, 2}
    rk = np.array([0, 0, 1, 0, 0, 2, 2, 2], np.uint32)
    ut = np.array([5, 3, 7, 3, 9, 1, 2, 1], np.uint32)
    edges, P, S = oracle_mod.build_edges(rk, ut)
    eu, ev = oracle_mod.unpack_edges(edges)
    assert list(zip(eu.tolist(), ev.tolist())) == [(1, 2), (3, 5), (3, 9), (5, 9)]
    assert (P, S) == (4, 6)
    e0, p0, s0 = oracle_mod.build_edges(np.zeros(0, np.uint32), np.zeros(0, np.uint32))
    assert e0.shape[0] == 0 and p0 == 0 and s0 == 0


def test_densest_core_checker_known_answers(oracle_mod):
    """oracle.densest_core (checker of kombgpu_graph_densest_core): K_6 plus a pendant path -> the 5-core K_6,
    density C(6,2)/6 = 2.5 (the empty levels 2..4 name the same block: k is the block's smallest coreness); a
    ring is its own densest core (density 1)."""
    k6 = [(i, j) for i in range(6) for j in range(i + 1, 6)]
    pairs = k6 + [(5, 6), (6, 7), (7, 8)]
    u = np.array([p[0] for p in pairs], np.uint32); v = np.array([p[1] for p in pairs], np.uint32)
    edges = oracle_mod.simplify(u, v)
    _, core = oracle_mod.coreness(9, edges)
    assert oracle_mod.densest_core(core, edges) == {"k": 5, "n_vertices": 6, "n_edges": 15, "density": 2.5}
    ring = oracle_mod.simplify(np.arange(8, dtype=np.uint32), ((np.arange(8) + 1) % 8).astype(np.uint32))
    _, core = oracle_mod.coreness(8, ring)
    assert oracle_mod.densest_core(core, ring) == {"k": 2, "n_vertices": 8, "n_edges": 8, "density": 1.0}


def test_product_code_never_touches_the_oracle():
    """The oracle is test infrastructure: nothing under komb_b200/, host/, include/ or tools/ may import, link or
    execute it (only tests/, __graft_entry__.smoke() and bench.py's CPU leg do)."""
    import re
    from pathlib import Path
    root = Path(__file__).resolve().parents[1]
    pat = re.compile(r"^\s*(from\s+oracle\b|import\s+oracle\b)|oracle/_ref|libkomb_oracle|komb_oracle\.c", re.M)
    offenders = []
    for sub in ("komb_b200", "host", "include", "tools"):
        for f in (root / sub).rglob("*"):
            if f.is_file() and f.suffix in (".py", ".cu", ".cuh", ".h", ".hpp", ".cpp"):
                if pat.search(f.read_text(errors="ignore")):
                    offenders.append(str(f.relative_to(root)))
    assert offenders == [], offenders


def test_truss_restatement_against_networkx(oracle_mod):
    """oracle.max_core_truss (the restated Kgraph::runTruss) against networkx: k_core for the maximal core, k_truss
    for the trussness of every edge."""
    import networkx as nx
    from komb_b200 import synth
    for seed, n, m in [(1, 300, 6000), (2, 1200, 30000)]:
        u, v = synth.rmat_edges(11, m, n_vertices=n, seed=seed)
        edges = oracle_mod.simplify(u, v)
        deg, core = oracle_mod.coreness(n, edges)
        got = oracle_mod.max_core_truss(n, edges, core)
        eu, ev = oracle_mod.unpack_edges(edges)
        g = nx.Graph(); g.add_nodes_from(range(n)); g.add_edges_from(zip(eu.tolist(), ev.tolist()))
        sub = nx.k_core(g)                                   # the maximal core
        assert sub.number_of_nodes() == got["n_core_vertices"] and sub.number_of_edges() == got["n_core_edges"]
        exp = {}
        k = 2
        while True:
            t = nx.k_truss(sub, k)
            if t.number_of_edges() == 0:
                break
            for a, b in t.edges():
                exp[(min(a, b), max(a, b))] = k
            k += 1
        assert {(int(a), int(b)): int(t) for a, b, t in zip(got["u"], got["v"], got["trussness"])} == exp
        assert got["max_trussness"] == k - 1
        top = nx.k_truss(sub, k - 1)
        assert sorted(x for x in top.nodes() if top.degree(x) > 0) == got["truss_vertices"].tolist()


def _dyadic_weights(rng, n):
    """multiples of 1/1024 below 8: every sum the peel forms is exact in double, whatever the order"""
    return rng.integers(0, 8192, n).astype(np.float64) / 1024.0


def test_densest_block_checkers(oracle_mod, tmp_path):
    """The bulk densest-block checker (oracle.densest_block_bulk) against the serial greedy of runMerge: both
    approximate the same optimum, so they bound each other (bulk <= OPT_sym <= OPT_b <= 2 greedy; greedy <= OPT_b <=
    2 OPT_sym <= 4 (1 + eps) bulk), and on a planted clique both find it.  The greedy is the restatement
    (oracle.densest_block_serial) and, where oracle/_ref has been built from the reference tree, also the reference's
    own loop over its HashIndexedMinHeap (oracle/_ref/densest_ref)."""
    from komb_b200 import synth

    def greedies(n, edges, w):
        out = [oracle_mod.densest_block_serial(n, edges, w)]
        if oracle_mod.REF_DENSEST.exists():
            out.append(oracle_mod.densest_block_greedy(n, edges, w, tmp_path))
        return out

    rng = np.random.default_rng(11)
    for seed, n, m, weighted in [(1, 200, 1500, False), (2, 800, 9000, True), (3, 50, 80, True), (4, 1500, 4000, False)]:
        u, v = synth.rmat_edges(11, m, n_vertices=n, seed=seed)
        edges = oracle_mod.simplify(u, v)
        w = _dyadic_weights(rng, n) if weighted else None
        eu, ev = oracle_mod.unpack_edges(edges)
        for greedy in greedies(n, edges, w):
            # the greedy's density is that of its rows and columns: weights of both plus the adjacency entries between
            rows, cols = np.zeros(n, bool), np.zeros(n, bool)
            rows[greedy["rows"]] = True
            cols[greedy["cols"]] = True
            wg = float(w[rows].sum() + w[cols].sum()) if weighted else 0.0
            entries = int((rows[eu] & cols[ev]).sum() + (rows[ev] & cols[eu]).sum())
            assert greedy["density"] == pytest.approx((wg + entries) / (rows.sum() + cols.sum()), rel=1e-12)
            for eps in (0.0, 0.5):
                bulk = oracle_mod.densest_block_bulk(n, edges, w, eps)
                assert bulk["density"] <= 2.0 * greedy["density"] * (1 + 1e-12)
                assert greedy["density"] <= 4.0 * (1.0 + eps) * bulk["density"] * (1 + 1e-12)
                # the reported density is the density of the reported block
                mem = bulk["member"]
                inside = int((mem[eu] & mem[ev]).sum())
                ws = float(w[mem].sum()) if weighted else 0.0
                assert bulk["n_vertices"] == int(mem.sum()) and bulk["n_edges"] == inside
                assert bulk["density"] == (ws + inside) / mem.sum()
    # K_30 planted in a sparse graph: the clique is the densest block for both (density (30 - 1) / 2)
    iu, iv = np.triu_indices(30, k=1)
    u = np.concatenate([iu + 7, rng.integers(0, 3000, 3000)]).astype(np.uint32)
    v = np.concatenate([iv + 7, rng.integers(0, 3000, 3000)]).astype(np.uint32)
    edges = oracle_mod.simplify(u, v)
    bulk = oracle_mod.densest_block_bulk(3000, edges, None, 0.1)
    assert set(np.flatnonzero(bulk["member"])) >= set(range(7, 37)) and bulk["density"] >= 14.5
    for greedy in greedies(3000, edges, None):
        assert set(greedy["rows"]) >= set(range(7, 37)) and greedy["density"] >= 14.5
    # degenerate inputs
    assert oracle_mod.densest_block_bulk(0, np.zeros(0, np.uint64))["n_vertices"] == 0
    one = oracle_mod.densest_block_bulk(5, np.zeros(0, np.uint64), np.array([0.0, 2.0, 0.5, 0.0, 0.0]), 0.5)
    assert one["n_vertices"] == 1 and one["density"] == 2.0 and one["member"].tolist() == [False, True, False, False, False]
