"""The unitig FASTA over the ranks of a communicator (kombgpu_dist_fasta_*, kombgpu_dist_anomalous): the ranks' extraction
slices, concatenated in rank order, against Context.fasta on one GPU byte for byte; the fence against Graph.anomalous
bit for bit; the errors with the single-GPU messages on every rank; and komb2 on several GPUs writing
anomalous_unitigs.fasta from them.  The ranks are threads of this process on device 0 (emulation) and, with two GPUs
or more, on distinct devices."""
import os
import subprocess
import threading

import numpy as np
import pytest

from conftest import komb2_case_names, load_komb2_case
from test_unitig_fasta_gpu import golden_fasta, make_fasta

pytestmark = pytest.mark.gpu

_CTX = None
REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
KOMB2 = os.path.join(REPO, "bin", "komb2")
WORLDS = [1, 2, 3]


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


def _slice(a, world, rank):
    """The unitig-range partition of the partitioned graph: step = ceil(n / world)."""
    n = len(a)
    step = -(-n // world) if n else 1
    lo = min(n, rank * step)
    return a[lo:min(n, lo + step)]


def _err(fn):
    import komb_b200
    with pytest.raises(komb_b200.KombGpuError) as e:
        fn()
    return e.value.code, str(e.value)


# ---- the golden komb2 cases: join through the DistHits and through host names, anomalous and truss extractions

def _single_golden(sam1, sam2, fasta):
    with _CTX.sam_parse([sam1, sam2]) as h, h.build_graph() as g:
        g.coreness()
        g.corea()
        anom = g.anomalous()
        tmask = np.zeros(anom["member"].shape[0], bool)
        tmask[g.max_core_truss()["truss_vertices"]] = True
        with _CTX.fasta(fasta) as fa:
            miss = fa.join(hits=h)
            return {"anom": anom, "tmask": tmask, "miss": miss, "a": fa.extract(anom["member"]), "t": fa.extract(tmask), "names": h.names()}


def _dist_golden(world, sam1, sam2, fasta, devices=None):
    from komb_b200.peer import DistFasta, DistGraph, DistHits

    def body(comm):
        with DistHits.parse(comm, [sam1, sam2]) as h, DistGraph.from_dist_hits(h) as g, DistFasta.load(comm, fasta) as fa:
            g.coreness()
            g.corea()
            anom = g.anomalous()
            st = g.stats()
            tmask = np.zeros(st["n_global"], bool)
            tmask[g.max_core_truss()["truss_vertices"]] = True
            tmask = tmask[st["v_lo"]:st["v_lo"] + st["n_local"]]
            res = {"anom": anom, "miss_hits": fa.join(hits=h)}
            res["a_hits"], res["t_hits"] = fa.extract(anom["member"]), fa.extract(tmask)
            res["miss_names"] = fa.join(names=h.names())
            res["a_names"], res["t_names"] = fa.extract(anom["member"]), fa.extract(tmask)
            res["counts"] = fa.counts()
            res["timing"] = fa.timing()
            return res
    return _run(world, body, devices)


def _check_golden(world, name, drop=0, devices=None):
    sam1, sam2, _ = load_komb2_case(name)
    fasta, names = golden_fasta(sam1, sam2, _CTX, 41)
    exp = _single_golden(sam1, sam2, fasta)
    if drop:   # vertices that neither mask selects lose their records: counted, not an error
        unselected = np.flatnonzero(~exp["anom"]["member"] & ~exp["tmask"])
        assert unselected.shape[0] >= drop
        rng = np.random.default_rng(drop)
        gone = {names[i] for i in rng.choice(unselected, size=drop, replace=False)}
        fasta = make_fasta([nm for nm in names if nm not in gone] + [b"extra_%d" % i for i in range(10)], 41)
        exp = _single_golden(sam1, sam2, fasta)
        assert exp["miss"] == drop
    parts = _dist_golden(world, sam1, sam2, fasta, devices)
    for p in parts:
        assert p["miss_hits"] == p["miss_names"] == exp["miss"]
        for k in ("q1", "q3", "fence", "n_selected"):
            assert p["anom"][k] == exp["anom"][k], k
        assert p["counts"]["n_records"] == fasta.count(b">")
    assert np.array_equal(np.concatenate([p["anom"]["member"] for p in parts]), exp["anom"]["member"])
    assert sum(p["counts"]["n_records_local"] for p in parts) == parts[0]["counts"]["n_records"]
    assert [p["counts"]["byte_lo"] for p in parts[1:]] == [p["counts"]["byte_hi"] for p in parts[:-1]]
    assert parts[-1]["counts"]["byte_hi"] == len(fasta)
    for k in ("hits", "names"):
        assert b"".join(p["a_" + k] for p in parts) == exp["a"]
        assert b"".join(p["t_" + k] for p in parts) == exp["t"]
    assert exp["t"]
    return parts


@pytest.mark.parametrize("world", WORLDS)
@pytest.mark.parametrize("name", komb2_case_names())
def test_golden_cases_match_single_gpu(name, world):
    parts = _check_golden(world, name)
    for p in parts:
        assert p["timing"]["ms_index"] > 0 and p["timing"]["kernel_launches"] > 0


@pytest.mark.parametrize("world", [2, 3])
def test_golden_missing_records_are_counted(world):
    _check_golden(world, "wide_s4", drop=5)


def test_distinct_gpus_match_single_gpu():
    n = _n_devices()
    if n < 2:
        pytest.skip("one GPU: the emulated ranks cover the slices")
    world = min(n, 4)
    _check_golden(world, "wide_s4", devices=list(range(world)))
    _check_golden(world, "mid_s2", devices=list(range(world)))
    _check_layout(world, LAYOUTS["one_big_record"](), devices=list(range(world)))


# ---- layouts, joined through host names

def _check_layout(world, case, devices=None):
    from komb_b200.peer import DistFasta
    text, names = case
    n = len(names)
    masks = [np.zeros(n, bool), np.ones(n, bool), np.arange(n) % 2 == 0, np.arange(n) % 2 == 1]
    with _CTX.fasta(text) as fa:
        miss = fa.join(names=names)
        exp = [fa.extract(m) for m in masks] if miss == 0 else [fa.extract(masks[0])]

    def body(comm):
        with DistFasta.load(comm, text) as fa:
            mine = _slice(names, comm.world, comm.rank)
            got_miss = fa.join(names=mine)
            ms = masks if got_miss == 0 else masks[:1]
            return got_miss, [fa.extract(_slice(m, comm.world, comm.rank)) for m in ms], fa.counts()
    parts = _run(world, body, devices)
    assert all(p[0] == miss for p in parts)
    for k, e in enumerate(exp):
        assert b"".join(p[1][k] for p in parts) == e, k
    return parts


def _names(k):
    return [b"u%d" % i for i in range(k)]


def _perm(names, seed):
    rng = np.random.default_rng(seed)
    return [names[i] for i in rng.permutation(len(names))]


def _big():
    rng = np.random.default_rng(3)
    s = np.frombuffer(b"ACGT", np.uint8)[rng.integers(0, 4, 100_000)].tobytes()
    return b">s1\nAC\n>big some description\n" + b"".join(s[i:i + 60] + b"\n" for i in range(0, len(s), 60)) + b">s2\nG\n", [b"big", b"s2", b"s1"]


LAYOUTS = {
    "wrapped_crlf_descriptions": lambda: (make_fasta(_names(300), 1), _perm(_names(300), 1)),
    "unterminated_last": lambda: (make_fasta(_names(200), 2)[:-1], _perm(_names(200), 2)),
    "unterminated_last_cr": lambda: (make_fasta(_names(50), 3)[:-1] + b"\r", _names(50)),
    "one_big_record": _big,
    "empty_fasta": lambda: (b"", [b"a", b"b"]),
    "more_ranks_than_records": lambda: (b">a\nAC\n>b\nGT", [b"b", b"a"]),
    "one_record": lambda: (b">only", [b"only"]),
    "whitespace_prefix": lambda: (b"\n\r\n \t\n" + make_fasta(_names(40), 4), _perm(_names(40), 4)),
    "empty_sequences": lambda: (b">a\n>b\n>c\n", [b"c", b"a", b"b"]),
    "no_vertices": lambda: (make_fasta(_names(20), 5), []),
}


@pytest.mark.parametrize("world", WORLDS)
@pytest.mark.parametrize("case", sorted(LAYOUTS))
def test_layouts_match_single_gpu(case, world):
    parts = _check_layout(world, LAYOUTS[case]())
    if case == "one_big_record" and world == 3:   # the big record's slice swallows a later cut: a rank is empty
        assert any(p[2]["n_records_local"] == 0 for p in parts)


# ---- errors: the single-GPU message on every rank, and the communicator still works afterwards

def _single_error(text):
    return _err(lambda: _CTX.fasta(text))


def _empty_name_on_rank2():
    recs = [b">r%d\nACGTACGT\n" % i for i in range(30)]
    recs[27] = b"> nameless\nACGT\n"
    return b"".join(recs)


ERRORS = {
    "prefix": lambda: b"junk\n" + make_fasta(_names(30), 6),
    "empty_name_rank2": _empty_name_on_rank2,
    "duplicate_across_ranks": lambda: make_fasta(_names(40) + [b"u0"], 7),
    "duplicates_twice": lambda: make_fasta([b"x", b"y"] + _names(40) + [b"y", b"x"], 8),
}


@pytest.mark.parametrize("case", sorted(ERRORS))
def test_malformed_fasta_fails_on_every_rank(case):
    from komb_b200.peer import DistFasta
    text = ERRORS[case]()
    code, msg = _single_error(text)
    good = make_fasta(_names(10), 9)

    def body(comm):
        got = _err(lambda: DistFasta.load(comm, text))
        with DistFasta.load(comm, good) as fa:   # the communicator still works
            fa.join(names=_slice(_names(10), comm.world, comm.rank))
            return got, fa.extract(np.ones(len(_slice(_names(10), comm.world, comm.rank)), bool))
    parts = _run(3, body)
    assert all(p[0] == (code, msg) for p in parts), (parts[0][0], msg)
    assert b"".join(p[1] for p in parts) == good


def test_selected_vertex_without_record_fails_on_every_rank():
    from komb_b200.peer import DistFasta
    names = _perm(_names(60), 10)
    gone = names[47]   # on the last of three ranks
    text = make_fasta([nm for nm in names if nm != gone], 11)
    mask = np.zeros(60, bool)
    mask[[3, 47, 58]] = True
    with _CTX.fasta(text) as fa:
        assert fa.join(names=names) == 1
        code, msg = _err(lambda: fa.extract(mask))
        mask2 = mask.copy()
        mask2[47] = False
        exp = fa.extract(mask2)
    assert "vertex 47" in msg and gone.decode() in msg

    def body(comm):
        with DistFasta.load(comm, text) as fa:
            miss = fa.join(names=_slice(names, comm.world, comm.rank))
            got = _err(lambda: fa.extract(_slice(mask, comm.world, comm.rank)))
            wrong_size = _err(lambda: fa.extract(np.zeros(1000, bool)))[0]
            return miss, got, wrong_size, fa.extract(_slice(mask2, comm.world, comm.rank))
    parts = _run(3, body)
    for p in parts:
        assert p[0] == 1 and p[1] == (code, msg) and p[2] != 0
    assert b"".join(p[3] for p in parts) == exp


def test_graph_and_comm_usable_after_errors():
    from komb_b200.peer import DistFasta, DistGraph, DistHits
    sam1, sam2, _ = load_komb2_case("mid_s2")
    fasta, _ = golden_fasta(sam1, sam2, _CTX, 42)
    exp = _single_golden(sam1, sam2, fasta)

    def body(comm):
        with DistHits.parse(comm, [sam1, sam2]) as h, DistGraph.from_dist_hits(h) as g:
            g.coreness()
            early = _err(lambda: g.anomalous())[0]
            g.corea()
            bad = _err(lambda: DistFasta.load(comm, ERRORS["prefix"]()))[0]
            with DistFasta.load(comm, fasta) as fa:
                no_join = _err(lambda: fa.extract(np.zeros(0, bool)))[0]
                fa.join(hits=h)
                return early, bad, no_join, fa.extract(g.anomalous()["member"])
    parts = _run(3, body)
    from komb_b200._lib import EINVAL, ESTATE
    for p in parts:
        assert p[0] == ESTATE and p[1] == EINVAL and p[2] == ESTATE
    assert b"".join(p[3] for p in parts) == exp["a"]


# ---- the fence: ties, n < 4, ranks without unitigs

def _ring_plus(n, extra):
    u = list(range(n)) + [a for a, _ in extra]
    v = [(i + 1) % n for i in range(n)] + [b for _, b in extra]
    return np.array(u, np.int32), np.array(v, np.int32)


FENCE_GRAPHS = {
    "ties": lambda: _ring_plus(200, [(0, k) for k in range(2, 40)] + [(5, 9), (9, 13)]),
    "path3": lambda: (np.array([0, 1], np.int32), np.array([1, 2], np.int32)),
    "edge2": lambda: (np.array([0], np.int32), np.array([1], np.int32)),
    "star": lambda: (np.zeros(30, np.int32), np.arange(1, 31, dtype=np.int32)),
}


@pytest.mark.parametrize("world", [2, 3, 4])
@pytest.mark.parametrize("case", sorted(FENCE_GRAPHS))
def test_fence_matches_single_gpu(case, world):
    import torch
    from komb_b200.peer import DistGraph
    u, v = FENCE_GRAPHS[case]()
    n = int(max(u.max(), v.max())) + 1
    with _CTX.graph_from_edges(u, v, n) as g:
        g.coreness()
        score = g.corea()
        exp = g.anomalous()
    assert len(np.unique(score)) < len(score)   # ties

    def body(comm):
        dev = torch.device("cuda", comm.ctx.device)
        lo, hi = len(u) * comm.rank // comm.world, len(u) * (comm.rank + 1) // comm.world
        du, dv = torch.from_numpy(u[lo:hi]).to(dev), torch.from_numpy(v[lo:hi]).to(dev)
        torch.cuda.synchronize(dev)
        with DistGraph.from_pairs(comm, du, dv, n) as dg:
            dg.analyse()
            r = dg.anomalous()
            r2 = dg.anomalous(whisker=0.25)
            return r, r2, dg.stats()["n_local"]
    parts = _run(world, body)
    with _CTX.graph_from_edges(u, v, n) as g:
        g.coreness()
        g.corea()
        exp2 = g.anomalous(whisker=0.25)
    for k, e in ((0, exp), (1, exp2)):
        for p in parts:
            for f in ("q1", "q3", "fence", "n_selected"):
                assert p[k][f] == e[f], (f, p[k][f], e[f])
        assert np.array_equal(np.concatenate([p[k]["member"] for p in parts]), e["member"])
    if n < world:
        assert any(p[2] == 0 for p in parts)


# ---- komb2 with KOMB_GPU_DEVICES and KOMB_UNITIG_FASTA=anomalous

def _devices_env():
    n = _n_devices()
    return ",".join(str(d) for d in range(min(n, 4))) if n >= 2 else "0,0,0"


def _komb2(tmp, sam1, sam2, fasta, env_extra, multi=True):
    tmp.mkdir(parents=True, exist_ok=True)
    (tmp / "r1.sam").write_bytes(sam1)
    (tmp / "r2.sam").write_bytes(sam2)
    (tmp / "u.fasta").write_bytes(fasta)
    out = tmp / "out"
    out.mkdir(exist_ok=True)
    env = {k: v for k, v in os.environ.items() if k not in ("KOMB_GPU_DEVICES", "KOMB_OUTPUT", "KOMB_TOKENIZE", "KOMB_UNITIG_FASTA")}
    if multi:
        env["KOMB_GPU_DEVICES"] = _devices_env()
    env.update(env_extra)
    r = subprocess.run([KOMB2, "-t", "4", "-l", "100", "-o", str(out), "-i", str(tmp / "r1.sam"), "-j", str(tmp / "r2.sam"),
                        "-u", str(tmp / "u.fasta")], env=env, capture_output=True, text=True, timeout=600)
    return r, {p.name: p.read_bytes() for p in sorted(out.iterdir())}


FILES = ("edgelist.txt", "kcore.tsv", "CoreA_anomaly.txt", "anomalous_unitigs.fasta")


@pytest.mark.parametrize("name", ["mid_s2", "wide_s4"])
@pytest.mark.parametrize("tokenise,output", [("gpu", "gpu"), ("gpu", "host"), ("host", "host")])
def test_komb2_multi_gpu_fasta_matches_one_gpu(tmp_path, name, tokenise, output):
    sam1, sam2, _ = load_komb2_case(name)
    fasta, _ = golden_fasta(sam1, sam2, _CTX, 43)
    env = {"KOMB_UNITIG_FASTA": "anomalous", "KOMB_TOKENIZE": tokenise, "KOMB_OUTPUT": output}
    r_multi, f_multi = _komb2(tmp_path / "multi", sam1, sam2, fasta, env)
    r_one, f_one = _komb2(tmp_path / "one", sam1, sam2, fasta, env, multi=False)
    assert r_multi.returncode == 0, r_multi.stderr
    assert r_one.returncode == 0, r_one.stderr
    for f in FILES:
        assert f in f_multi and f_multi[f] == f_one[f], f
    assert r_multi.stdout.count("\n") == r_one.stdout.count("\n")


@pytest.mark.parametrize("tokenise", ["gpu", "host"])
def test_komb2_multi_gpu_missing_selected_unitig(tmp_path, tokenise):
    sam1, sam2, _ = load_komb2_case("wide_s4")
    exp = _single_golden(sam1, sam2, golden_fasta(sam1, sam2, _CTX, 44)[0])
    names = exp["names"]
    sel = np.flatnonzero(exp["anom"]["member"])
    assert sel.shape[0] > 0
    gone = names[int(sel[0])]
    fasta = make_fasta([nm for nm in names if nm != gone], 45)
    env = {"KOMB_UNITIG_FASTA": "anomalous", "KOMB_TOKENIZE": tokenise}
    r_multi, f_multi = _komb2(tmp_path / "multi", sam1, sam2, fasta, env)
    r_one, f_one = _komb2(tmp_path / "one", sam1, sam2, fasta, env, multi=False)
    assert r_one.returncode == 1 and f"unitig '{gone.decode()}'" in r_one.stderr, r_one.stderr
    assert r_multi.returncode == 1
    assert r_multi.stderr.strip().splitlines()[-1] == r_one.stderr.strip().splitlines()[-1]
    for f in FILES[:3]:   # written before the FASTA is
        assert f_multi[f] == f_one[f], f
