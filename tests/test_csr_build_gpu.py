"""The single-GPU CSR build (csr_from_edges) against a numpy CSR built from the same edge list.

Every row of the symmetric graph is [back neighbours (< v, ascending) | forward neighbours (> v, ascending)], i.e. the
row sorted ascending, so np.lexsort of the 2E directed entries by (source, neighbour) is the reference.  Row starts,
degrees, the max degree and the forward index of the edge list (fwd_ptr) are compared byte for byte.  The cases cover
the shapes the build treats specially: sorts of one to four passes on the second endpoint, fewer than two edges (no
sort pass runs), long runs of ids without edges, a hub whose back half alone is longer than a sort tile, both entry
points (pairs and hits), the path that already holds the forward index (analyse_hits_csr) and the chunked pair path.
"""
import numpy as np
import pytest

from komb_b200 import synth

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ctx():
    import komb_b200
    c = komb_b200.Context(0)
    yield c
    c.close()


def ref_csr(u, v, n):
    """numpy CSR of the simple graph on the sorted unique edges (u < v)."""
    src = np.concatenate([u, v]).astype(np.int64)
    dst = np.concatenate([v, u]).astype(np.int64)
    order = np.lexsort((dst, src))
    deg = np.bincount(src, minlength=n).astype(np.int32)
    row_ptr = np.zeros(n + 1, np.uint64)
    np.cumsum(deg, out=row_ptr[1:])
    return row_ptr, dst[order].astype(np.uint32), deg


def simple_edges(a, b):
    """Canonical sorted unique edges (u < v) of a pair list, loops dropped."""
    a, b = np.asarray(a, np.uint64), np.asarray(b, np.uint64)
    lo, hi = np.minimum(a, b), np.maximum(a, b)
    keep = lo != hi
    keys = np.unique((lo[keep] << np.uint64(32)) | hi[keep])
    return (keys >> np.uint64(32)).astype(np.uint32), (keys & np.uint64(0xffffffff)).astype(np.uint32)


def check_graph(g, n, u=None, v=None):
    """g's CSR, degrees, counts, max degree and forward index against the numpy CSR of its edge list (or of u, v)."""
    gu, gv = g.edges()
    if u is not None:
        assert np.array_equal(gu, u) and np.array_equal(gv, v), "edge list differs"
    assert np.all(gu[1:].astype(np.uint64) << np.uint64(32) | gv[1:] > gu[:-1].astype(np.uint64) << np.uint64(32) | gv[:-1])
    E = gu.shape[0]
    assert g.counts() == (n, E)
    row_ptr, col, deg = ref_csr(gu, gv, n)
    g_row_ptr, g_col = g.csr()
    assert g_row_ptr.tobytes() == row_ptr.tobytes(), "row_ptr differs"
    assert g_col.tobytes() == col.tobytes(), "col differs"
    assert g.degree().tobytes() == deg.tobytes(), "degree differs"
    assert g.stats()["max_degree"] == (int(deg.max()) if n else 0)
    fp, fv = g.edges_csr()
    assert fp.tobytes() == np.searchsorted(gu, np.arange(n + 1), side="left").astype(np.uint64).tobytes()
    assert np.array_equal(fv, gv)
    return E


def from_pairs(ctx, a, b, n):
    u, v = simple_edges(a, b)
    with ctx.graph_from_edges(np.asarray(a, np.uint32), np.asarray(b, np.uint32), n) as g:
        return check_graph(g, n, u, v)


def test_cfg2_shaped_hits(ctx, oracle_mod):
    m1, m2 = synth.metagenome_hits(100_000, 500_000, seed=3)
    rk = np.concatenate([m1.read_key, m2.read_key])
    ut = np.concatenate([m1.unitig, m2.unitig])
    n = 100_000
    exp_edges, _, _ = oracle_mod.build_edges(rk, ut)
    u = (exp_edges >> np.uint64(32)).astype(np.uint32)
    v = (exp_edges & np.uint64(0xffffffff)).astype(np.uint32)
    with ctx.build_graph(rk, ut, n) as g:
        assert check_graph(g, n, u, v) > 100_000
    # the e2e path builds the forward index before the CSR: fwd_ptr, v and degree against the same edge list
    g, r = ctx.analyse_hits_csr(rk, ut, n)
    with g:
        check_graph(g, n, u, v)
        assert r["fwd_ptr"].tobytes() == np.searchsorted(u, np.arange(n + 1), side="left").astype(np.uint64).tobytes()
        assert np.array_equal(r["v"], v)
        assert r["degree"].tobytes() == ref_csr(u, v, n)[2].tobytes()
    # the same edges through the pair entry point
    assert from_pairs(ctx, v, u, n) == u.shape[0]


def test_two_vertices(ctx):
    assert from_pairs(ctx, [1], [0], 2) == 1      # one 1-bit pass, one edge


@pytest.mark.parametrize("a,b", [([], []), ([2], [0]), ([1, 1], [1, 1])], ids=["E0", "E1", "loops_only"])
def test_three_vertices_no_sort_pass(ctx, a, b):
    assert from_pairs(ctx, a, b, 3) == len(simple_edges(a, b)[0])


def test_one_pass_many_edges(ctx):
    rng = np.random.default_rng(1)
    a, b = rng.integers(0, 200, 5000), rng.integers(0, 200, 5000)
    assert from_pairs(ctx, a, b, 200) > 1000


def test_isolated_and_long_empty_ranges(ctx):
    n = 5_000_000
    rng = np.random.default_rng(2)
    ids = np.concatenate([np.arange(1000), np.arange(n - 1000, n)])
    a, b = rng.choice(ids, 40_000), rng.choice(ids, 40_000)
    a = np.concatenate([a, [0, 17]]); b = np.concatenate([b, [n - 1, n - 2]])
    assert from_pairs(ctx, a, b, n) > 30_000


def test_star_hub(ctx):
    n = 300_000
    rng = np.random.default_rng(3)
    hub = n - 5                                  # most of the hub's row is its back half
    leaves = np.setdiff1d(np.arange(n), [hub])[: (1 << 17) + 4321]
    a = np.concatenate([np.full(leaves.shape[0], hub), rng.integers(0, n, 50_000)])
    b = np.concatenate([leaves, rng.integers(0, n, 50_000)])
    E = from_pairs(ctx, a, b, n)
    assert E > (1 << 17)


@pytest.mark.parametrize("n", [(1 << 20) + 3, (1 << 24) + 1], ids=["3_passes", "4_passes"])
def test_multi_pass(ctx, n):
    rng = np.random.default_rng(n)
    a, b = rng.integers(0, n, 400_000), rng.integers(0, n, 400_000)
    a = np.concatenate([a, [0, n - 1, n - 2, 5]]); b = np.concatenate([b, [n - 1, 0, n - 1, n - 1]])
    assert from_pairs(ctx, a, b, n) > 300_000


@pytest.mark.parametrize("entry", ["hits", "pairs"])
def test_chunked_pair_path(ctx, monkeypatch, entry):
    m1, m2 = synth.metagenome_hits(20_000, 60_000, seed=7)
    rk = np.concatenate([m1.read_key, m2.read_key])
    ut = np.concatenate([m1.unitig, m2.unitig])
    n = 20_000
    with ctx.build_graph(rk, ut, n) as g:
        u, v = g.edges()
    monkeypatch.setenv("KOMBGPU_PAIR_CHUNK", "5000")
    if entry == "hits":
        with ctx.build_graph(rk, ut, n) as g:
            assert g.build_chunks() > 1
            check_graph(g, n, u, v)
    else:
        with ctx.graph_from_edges(np.concatenate([v, u[:100]]), np.concatenate([u, v[:100]]), n) as g:
            assert g.build_chunks() > 1
            check_graph(g, n, u, v)
