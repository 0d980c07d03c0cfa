"""Onion layers over the ranks of a communicator (kombgpu_dist_onion, DistGraph.onion, onion.tsv slices): the ranks'
slices, concatenated in rank order, against the C restatement of networkx.onion_layers (tests/onion_ref.c) and the
single-GPU Graph.onion() bit for bit; the coreness the layers imply against the partitioned coreness; every build
layout; the cache; onion.tsv against Graph.format on one GPU; the errors.  The ranks are threads of this process on
device 0 (emulation) and, with two GPUs or more, on distinct devices."""
import functools
import threading

import numpy as np
import pytest

from conftest import komb2_case_names, load_komb2_case
from komb_b200 import synth
from komb_b200._lib import EINVAL, ESTATE
from onion_ref import coreness_from_layers, onion_layers, simple_edges

pytestmark = pytest.mark.gpu

_CTX = None
WORLDS = [1, 2, 3, 4]
FILE_ONION = 3
HEADER = b"#VID\tName\tCoreness\tLayer\n"


def _n_devices():
    import torch
    return torch.cuda.device_count()


@pytest.fixture(scope="module", autouse=True)
def ctx():
    global _CTX
    import komb_b200
    _CTX = komb_b200.Context(0)
    yield _CTX
    _CTX.close()


def _run(world, body, devices=None, timeout=300):
    """run_local with a deadline: a rank that waits for another which never comes fails the test instead of hanging."""
    from komb_b200.peer import run_local
    out, err = [], []

    def go():
        try:
            out.append(run_local(world, body, devices=devices))
        except BaseException as e:   # noqa: BLE001 - re-raised below
            err.append(e)
    t = threading.Thread(target=go, daemon=True)
    t.start()
    t.join(timeout)
    assert not t.is_alive(), "a rank is still waiting"
    if err:
        raise err[0]
    return out[0]


def _hub(k=6, leaves=100_000):
    """A hub whose list is longer than a slice on every rank (ids scrambled) and too long for one CTA's step.  Its
    `leaves` leaves go in layer 1 and leave it at degree k; level k opens with the hub alone.  Its k other neighbours
    hang on a K_10 at degree k + 1 and fall to k only through the hub's list: they must form the very next layer."""
    h, b0, c0 = 0, 1, 1 + k
    l0 = c0 + 10
    cu, cv = np.triu_indices(10, 1)
    u = [np.full(k, h), cu + c0, np.full(leaves, h)]
    v = [np.arange(b0, b0 + k), cv + c0, np.arange(l0, l0 + leaves)]
    for i in range(k):   # b_i -> k members of the K_10
        u.append(np.full(k, b0 + i))
        v.append(c0 + (np.arange(k) + i) % 10)
    n = l0 + leaves
    u = np.concatenate(u).astype(np.uint32)
    v = np.concatenate(v).astype(np.uint32)
    return n, synth.scramble_ids(u, n), synth.scramble_ids(v, n), synth.scramble_ids(np.arange(b0, b0 + k, dtype=np.uint32), n), \
        int(synth.scramble_ids(np.zeros(1, np.uint32), n)[0])


def _path(n):
    u = np.arange(n - 1, dtype=np.uint32)
    return n, u, u + 1


@functools.lru_cache(maxsize=None)
def _case(name):
    """(n, u, v) of a case"""
    if name == "empty":
        return 10, np.zeros(0, np.uint32), np.zeros(0, np.uint32)
    if name == "k4_rank_without_vertices":   # with 3 ranks the last one owns no unitig
        iu, iv = np.triu_indices(4, 1)
        return 4, iu.astype(np.uint32), iv.astype(np.uint32)
    if name == "path":
        n = 60
        return n, synth.scramble_ids(np.arange(n - 1, dtype=np.uint32), n), synth.scramble_ids(np.arange(1, n, dtype=np.uint32), n)
    if name == "star":
        return 301, np.zeros(300, np.uint32), np.arange(1, 301, dtype=np.uint32)
    if name == "clique":
        iu, iv = np.triu_indices(80, 1)
        return 80, iu.astype(np.uint32), iv.astype(np.uint32)
    if name == "rmat":
        u, v = synth.rmat_edges(16, 500_000, seed=16)
        return 1 << 16, u, v
    if name == "ramp":       # hundreds of levels, ids scrambled so every rank holds a share of each
        u, v = synth.ramp_edges(300, 5)
        n = 300 * 5 + 37
        return n, synth.scramble_ids(u, n), synth.scramble_ids(v, n)
    if name == "hub":
        return _hub()[:3]
    if name == "path_2e4":
        return _path(20_000)
    raise KeyError(name)


CASES = ["empty", "k4_rank_without_vertices", "path", "star", "clique", "rmat", "ramp", "hub", "path_2e4"]


@functools.lru_cache(maxsize=None)
def _expected(name):
    n, u, v = _case(name)
    layer, core, n_layers = onion_layers(n, u, v)
    with _CTX.graph_from_edges(u, v, n) as g:
        r = g.onion()
    assert r["n_layers"] == n_layers and np.array_equal(r["layer"], layer), "the single-GPU onion differs from the restatement"
    return layer, core, n_layers


def _pairs_body(n, u, v, again=False):
    def body(comm):
        import torch
        from komb_b200.peer import DistGraph
        sl = slice(len(u) * comm.rank // comm.world, len(u) * (comm.rank + 1) // comm.world)
        dev = torch.device("cuda", comm.ctx.device)
        ta = torch.from_numpy(u[sl].view(np.int32).copy()).to(dev)
        tb = torch.from_numpy(v[sl].view(np.int32).copy()).to(dev)
        torch.cuda.synchronize(dev)
        with DistGraph.from_pairs(comm, ta, tb, n) as g:
            r = g.onion()
            t = g.onion_timing()
            g.analyse()   # results() reads the coreness with the scores
            res = {"onion": r, "timing": t, "coreness": g.results()["coreness"], "stats": g.stats()}
            if again:
                res["cached"] = g.onion()
                res["timing_cached"] = g.onion_timing()
                res["again"] = g.onion(again=True)
            return res
    return body


def _check_parts(name, parts):
    n, u, v = _case(name)
    layer, core, n_layers = _expected(name)
    got = np.concatenate([p["onion"]["layer"] for p in parts])
    assert got.dtype == np.uint32 and got.shape == (n,)
    assert [p["onion"]["v_lo"] for p in parts] == sorted(p["onion"]["v_lo"] for p in parts)
    assert np.array_equal(got, layer)
    assert {p["onion"]["n_layers"] for p in parts} == {n_layers}
    dist_core = np.concatenate([p["coreness"] for p in parts])
    assert np.array_equal(dist_core, core)
    a, b = simple_edges(u, v)
    assert np.array_equal(coreness_from_layers(n, a, b, got), dist_core)


@pytest.mark.parametrize("world", WORLDS)
@pytest.mark.parametrize("name", CASES)
def test_emulated_ranks_match_single_gpu(name, world):
    n, u, v = _case(name)
    parts = _run(world, _pairs_body(n, u, v))
    _check_parts(name, parts)
    if name == "k4_rank_without_vertices" and world == 3:
        assert parts[2]["onion"]["layer"].shape == (0,)
    if name == "empty":
        assert parts[0]["onion"]["n_layers"] == 1
    if name == "hub":
        _, _, _, bs, hub = _hub()
        got = np.concatenate([p["onion"]["layer"] for p in parts])
        assert (got[bs] == got[hub] + 1).all()   # the hub's slices landed inside its layer


def test_long_path_two_ranks():
    """2 x 10^5 vertices at world 2: 10^5 layers, nearly all of them thin steps on one CTA, and a meeting each."""
    n, u, v = _path(200_000)
    parts = _run(2, _pairs_body(n, u, v), timeout=600)
    got = np.concatenate([p["onion"]["layer"] for p in parts])
    assert np.array_equal(got, (np.minimum(np.arange(n), np.arange(n)[::-1]) + 1).astype(np.uint32))
    assert {p["onion"]["n_layers"] for p in parts} == {n // 2}
    for p in parts:
        t = p["timing"]
        assert t["levels"] == 1 and t["meetings"] >= n // 2 and t["solo_steps"] >= n // 2 - 2


@pytest.mark.parametrize("peel", ["log", "async", "replicated"])
def test_every_build_layout(monkeypatch, peel):
    """The build lays the adjacency out for the peel it picked (by neighbour for log, rows for async and replicated);
    the onion walks the by-neighbour layout, built from the rows when the graph holds rows."""
    monkeypatch.setenv("KOMBGPU_DIST_PEEL", peel)
    n, u, v = _case("hub")
    parts = _run(3, _pairs_body(n, u, v))
    assert {p["stats"]["peel_async"] for p in parts} == {{"log": 0, "async": 1, "replicated": 2}[peel]}
    _check_parts("hub", parts)
    assert all((p["timing"]["ms_transpose"] > 0) == (peel != "log") for p in parts)
    name = komb2_case_names()[0]
    single, _ = _single_sam(name)
    got = _dist_sam(3, _sam(name))
    assert b"".join(p["tsv"] for p in got) == single["tsv"]
    assert np.array_equal(np.concatenate([p["layer"] for p in got]), single["layer"])


def test_cache_and_again():
    n, u, v = _case("ramp")
    parts = _run(3, _pairs_body(n, u, v, again=True))
    _check_parts("ramp", parts)
    for p in parts:
        assert np.array_equal(p["cached"]["layer"], p["onion"]["layer"]) and p["cached"]["n_layers"] == p["onion"]["n_layers"]
        assert p["timing_cached"] == p["timing"]   # no second run
        assert np.array_equal(p["again"]["layer"], p["onion"]["layer"]) and p["again"]["n_layers"] == p["onion"]["n_layers"]


def test_distinct_gpus_match_single_gpu():
    nd = _n_devices()
    if nd < 2:
        pytest.skip("one GPU: the emulated ranks above cover the slices")
    world = min(nd, 4)
    for name in ("hub", "ramp", "rmat", "k4_rank_without_vertices"):
        n, u, v = _case(name)
        _check_parts(name, _run(world, _pairs_body(n, u, v), devices=list(range(world))))
    name = komb2_case_names()[0]
    single, _ = _single_sam(name)
    got = _dist_sam(world, _sam(name), devices=list(range(world)))
    assert b"".join(p["tsv"] for p in got) == single["tsv"]


# ---- SAM pairs: DistHits.parse -> DistGraph.from_dist_hits -> onion and onion.tsv

def _synth_pair(n_unitigs=300, n_pairs=400, **kw):
    h1, h2 = synth.metagenome_hits(n_unitigs, n_pairs, seed=5)
    return [synth.render_sam(h1, n_unitigs, 1, **kw), synth.render_sam(h2, n_unitigs, 2, **kw)]


def _sam(name):
    if name == "synthetic":
        return _synth_pair(unmapped_every=7)
    if name == "both_empty":
        return [b"", b""]
    sam1, sam2, _ = load_komb2_case(name)
    return [sam1, sam2]


def _single_sam(name):
    texts = _sam(name)
    with _CTX.sam_parse(texts) as h, h.build_graph() as g:
        r = g.onion()
        return {"layer": r["layer"], "n_layers": r["n_layers"], "tsv": g.format(FILE_ONION, h)}, g.stats()["n_vertices"]


def _dist_sam(world, texts, devices=None):
    from komb_b200.peer import DistGraph, DistHits

    def body(comm):
        with DistHits.parse(comm, texts) as h, DistGraph.from_dist_hits(h) as g:
            r = g.onion()
            return {"layer": r["layer"], "n_layers": r["n_layers"], "tsv": g.format(DistGraph.FILE_ONION, h)}
    return _run(world, body, devices)


SAM_CASES = [c for c in komb2_case_names() if not c.endswith("_t4")] + ["synthetic"]


@pytest.mark.parametrize("world", WORLDS)
@pytest.mark.parametrize("name", SAM_CASES)
def test_sam_pairs_match_single_gpu(name, world):
    single, _ = _single_sam(name)
    parts = _dist_sam(world, _sam(name))
    assert np.array_equal(np.concatenate([p["layer"] for p in parts]), single["layer"])
    assert {p["n_layers"] for p in parts} == {single["n_layers"]}
    assert b"".join(p["tsv"] for p in parts) == single["tsv"]
    assert parts[0]["tsv"].startswith(HEADER) and all(not p["tsv"].startswith(HEADER) for p in parts[1:])


@pytest.mark.parametrize("world", [1, 3])
def test_empty_sam_pair_header_on_rank0_only(world):
    single, n = _single_sam("both_empty")
    assert n == 0 and single["tsv"] == HEADER
    parts = _dist_sam(world, _sam("both_empty"))
    assert [p["tsv"] for p in parts] == [HEADER] + [b""] * (world - 1)
    assert {p["n_layers"] for p in parts} == {0}


def _code(fn):
    import komb_b200
    with pytest.raises(komb_b200.KombGpuError) as exc:
        fn()
    return exc.value.code


def test_errors_leave_graph_and_comm_usable():
    import torch
    from komb_b200.peer import DistGraph, DistHits
    texts = _synth_pair(n_unitigs=200, n_pairs=300)
    other = _synth_pair(n_unitigs=90, n_pairs=100)
    with _CTX.sam_parse(texts) as h1, h1.build_graph() as g1:
        g1.onion()
        exp_tsv = g1.format(FILE_ONION, h1)

    def body(comm):
        res = {}
        with DistHits.parse(comm, texts) as h, DistHits.parse(comm, other) as h_other, DistGraph.from_dist_hits(h) as g:
            res["no_names_early"] = _code(lambda: g.format(FILE_ONION))
            res["state"] = _code(lambda: g.format(FILE_ONION, h))
            res["fetch_first"] = _code(lambda: g._ctx._check(g._lib.kombgpu_dist_graph_format_fetch(g._h, FILE_ONION, None, 0)))
            res["timing_early"] = _code(lambda: g.onion_timing())
            res["which_high"] = _code(lambda: g.format(4, h))
            g.onion()
            res["no_names"] = _code(lambda: g.format(FILE_ONION))
            res["other_names"] = _code(lambda: g.format(FILE_ONION, h_other))
            res["tsv"] = g.format(FILE_ONION, h)
            # a graph built from pairs has no names of its own
            dev = torch.device("cuda", comm.ctx.device)
            a = torch.arange(comm.rank, 40, comm.world, dtype=torch.int32, device=dev)
            with DistGraph.from_pairs(comm, a, (a + 1) % 40, 40) as gp:
                gp.onion()
                res["pairs_names"] = _code(lambda: gp.format(FILE_ONION, h))
                res["pairs_no_names"] = _code(lambda: gp.format(FILE_ONION))
            # the communicator still works: a collective after the errors
            with DistGraph.from_dist_hits(h) as g2:
                g2.onion()
                res["tsv2"] = g2.format(FILE_ONION, h)
        return res
    parts = _run(3, body)
    for p in parts:
        assert p["no_names_early"] == EINVAL and p["state"] == ESTATE and p["fetch_first"] == ESTATE
        assert p["timing_early"] == ESTATE and p["which_high"] == EINVAL
        assert p["no_names"] == EINVAL and p["other_names"] == EINVAL
        assert p["pairs_names"] == EINVAL and p["pairs_no_names"] == EINVAL
    assert b"".join(p["tsv"] for p in parts) == exp_tsv
    assert b"".join(p["tsv2"] for p in parts) == exp_tsv


@pytest.mark.parametrize("who", ["rank0_only", "last_only", "rotated"])
def test_format_is_local(who):
    """Only one rank formats onion.tsv, or each formats its files in its own order: no rank waits for another."""
    from komb_b200.peer import DistGraph, DistHits
    texts = _synth_pair(n_unitigs=400, n_pairs=700)
    with _CTX.sam_parse(texts) as h1, h1.build_graph() as g1:
        g1.onion()
        g1.coreness()
        exp = {1: g1.format(1, h1), FILE_ONION: g1.format(FILE_ONION, h1)}
    world = 3

    def body(comm):
        with DistHits.parse(comm, texts) as h, DistGraph.from_dist_hits(h) as g:
            g.onion()   # collective
            g.coreness()
            r = comm.rank
            if who == "rank0_only" and r != 0 or who == "last_only" and r != world - 1:
                return None
            order = [FILE_ONION, 1] if who == "rotated" and r % 2 else [1, FILE_ONION]
            got = {w: g.format(w, h) for w in order}
            assert got == {w: g.format(w, h) for w in reversed(order)}   # cached: the same bytes
            return got
    parts = _run(world, body)
    if who == "rotated":
        for w in exp:
            assert b"".join(p[w] for p in parts) == exp[w]
    else:
        r = 0 if who == "rank0_only" else world - 1
        assert all(p is None for q, p in enumerate(parts) if q != r)
        assert parts[r][FILE_ONION].startswith(HEADER) == (r == 0)
        assert parts[r][FILE_ONION] in exp[FILE_ONION]
