"""The three output files formatted on the device over the ranks of a communicator (kombgpu_dist_graph_format): the
ranks' slices, concatenated in rank order, against kombgpu_graph_format on one GPU, byte for byte; the errors; calls
that only some ranks make; and komb2 on several GPUs writing its files from them.  The ranks are threads of this
process on device 0 (emulation) and, with two GPUs or more, on distinct devices."""
import ctypes
import os
import subprocess
import threading

import numpy as np
import pytest

from conftest import komb2_case_names, load_komb2_case
from komb_b200 import synth
from komb_b200._lib import EINVAL, ESTATE, KEY_EXACT64, KEY_REF32

pytestmark = pytest.mark.gpu

_CTX = None
REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
KOMB2 = os.path.join(REPO, "bin", "komb2")
FILES = (0, 1, 2)   # EDGELIST, KCORE, COREA


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


def _single(texts, key_mode):
    with _CTX.sam_parse(texts) as h, h.build_graph() as g:
        g.analyse(key_mode)
        return [g.format(w, h) for w in FILES]


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


def _dist(world, texts, key_mode, devices=None):
    from komb_b200.peer import DistGraph, DistHits

    def body(comm):
        with DistHits.parse(comm, texts) as h, DistGraph.from_dist_hits(h) as g:
            edges = g.format(0)   # needs only the build
            g.coreness()
            g.corea(key_mode)
            return {"files": [edges, g.format(1, h), g.format(2)], "score": g.results()["score"]}
    return _run(world, body, devices)


def _check(texts, world, key_mode=KEY_REF32, devices=None):
    exp = _single(texts, key_mode)
    parts = _dist(world, texts, key_mode, devices)
    for w in FILES:
        assert b"".join(p["files"][w] for p in parts) == exp[w], ("edgelist.txt", "kcore.tsv", "CoreA_anomaly.txt")[w]
    # the formatter alone: the concatenated scores through the single-GPU formatter
    score = np.concatenate([p["score"] for p in parts])
    assert b"".join(p["files"][2] for p in parts) == _CTX.format_corea(score)
    return parts


WORLDS = [1, 2, 3, 4]


@pytest.mark.parametrize("key_mode", [KEY_REF32, KEY_EXACT64])
@pytest.mark.parametrize("world", WORLDS)
@pytest.mark.parametrize("name", komb2_case_names())
def test_golden_cases_match_single_gpu(name, world, key_mode):
    sam1, sam2, _ = load_komb2_case(name)
    _check([sam1, sam2], world, key_mode)


def _synth_pair(n_unitigs=300, n_pairs=400, **kw):
    h1, h2 = synth.metagenome_hits(n_unitigs, n_pairs, seed=5)
    return [synth.render_sam(h1, n_unitigs, 1, **kw), synth.render_sam(h2, n_unitigs, 2, **kw)]


@pytest.mark.parametrize("world", WORLDS)
@pytest.mark.parametrize("kw", [{"with_header": False}, {"unmapped_every": 7}, {"with_header": False, "unmapped_every": 3}])
def test_render_sam_matches_single_gpu(world, kw):
    _check(_synth_pair(**kw), world)


REC = b"\t0\t%s\t1\t60\t4M\t*\t0\t0\tACGT\tIIII\n"


def _rec(q, r):
    return q + REC.replace(b"%s", r)


# the edge cases of tests/test_dist_sam_gpu.py
EDGE_CASES = {
    "sq_below": [_rec(b"r1/1", b"uC") + b"@SQ\tSN:uB\tLN:4\n" + _rec(b"r2/1", b"uB") + b"@SQ\tSN:uC\tLN:4\n" + _rec(b"r3/1", b"uA"),
                 _rec(b"r1/2", b"uA") + b"@SQ\tSN:uA\tLN:4\n" + _rec(b"r2/2", b"uD")],
    "both_empty": [b"", b""],
    "more_ranks_than_lines": [_rec(b"r1/1", b"u1"), _rec(b"r1/2", b"u2")],
    "mate_far": [b"".join(_rec(b"r%d/1" % i, b"u%d" % (i % 13)) for i in range(40)),
                 b"".join(_rec(b"r%d/2" % i, b"u%d" % (i % 7 + 20)) for i in range(1, 40)) + _rec(b"r0/2", b"uFar") + _rec(b"r0/2", b"u3")],
    "long_names": [b"".join(_rec(b"read%s%d/1" % (b"x" * 70, i), b"unitig_%s_%d" % (b"y" * (i % 90), i % 11)) for i in range(60)),
                   b"".join(_rec(b"read%s%d/2" % (b"x" * 70, i), b"unitig_%s_%d" % (b"y" * (i % 90), i % 17)) for i in range(60))],
}


@pytest.mark.parametrize("world", WORLDS)
@pytest.mark.parametrize("case", sorted(EDGE_CASES))
def test_edge_cases_match_single_gpu(case, world):
    parts = _check(EDGE_CASES[case], world)
    if case == "both_empty":   # the header alone, on rank 0
        assert parts[0]["files"][1] == b"#VID\tName\tCoreness\tDegree\n"
        assert all(p["files"][1] == b"" for p in parts[1:])


@pytest.mark.parametrize("peel", ["log", "async", "replicated"])
def test_every_build_layout(monkeypatch, peel):
    monkeypatch.setenv("KOMBGPU_DIST_PEEL", peel)
    _check(_synth_pair(n_unitigs=500, n_pairs=900, unmapped_every=9), 3)


def test_distinct_gpus_match_single_gpu():
    n = _n_devices()
    if n < 2:
        pytest.skip("one GPU: the emulated ranks above cover the slices")
    world = min(n, 4)
    devices = list(range(world))
    sam1, sam2, _ = load_komb2_case(komb2_case_names()[0])
    _check([sam1, sam2], world, devices=devices)
    _check(_synth_pair(unmapped_every=5), world, KEY_EXACT64, devices=devices)
    _check(EDGE_CASES["mate_far"], world, devices=devices)


@pytest.mark.parametrize("who", ["rank0_only", "last_only", "rotated"])
def test_format_is_local(who):
    """Only some ranks format, or each in its own order: no rank waits for another, and every slice is right."""
    from komb_b200.peer import DistGraph, DistHits
    texts = _synth_pair(n_unitigs=400, n_pairs=700)
    exp = _single(texts, KEY_REF32)
    world = 3

    def body(comm):
        with DistHits.parse(comm, texts) as h, DistGraph.from_dist_hits(h) as g:
            g.analyse()
            r = comm.rank
            if who == "rank0_only" and r != 0 or who == "last_only" and r != world - 1:
                return None
            order = [FILES[(r + k) % 3] for k in range(3)] if who == "rotated" else list(FILES)
            got = {w: g.format(w, h) for w in order}
            again = {w: g.format(w, h) for w in reversed(order)}   # cached: the same bytes
            assert got == again
            return got
    parts = _run(world, body)
    if who == "rotated":
        for w in FILES:
            assert b"".join(p[w] for p in parts) == exp[w]
    else:
        # the slice of the one rank that formatted is the bytes of the single-GPU file at its place
        full = _dist(world, texts, KEY_REF32)
        r = 0 if who == "rank0_only" else world - 1
        assert parts[r] == {w: full[r]["files"][w] for w in FILES}
        assert all(p is None for q, p in enumerate(parts) if q != r)


def _code(fn):
    import komb_b200
    with pytest.raises(komb_b200.KombGpuError) as exc:
        fn()
    return exc.value.code


def test_errors_leave_graph_and_comm_usable():
    from komb_b200.peer import DistGraph, DistHits
    texts = _synth_pair(n_unitigs=200, n_pairs=300)
    other = _synth_pair(n_unitigs=90, n_pairs=100)
    exp = _single(texts, KEY_REF32)

    def body(comm):
        res = {}
        with DistHits.parse(comm, texts) as h, DistHits.parse(comm, other) as h_other, DistGraph.from_dist_hits(h) as g:
            buf = ctypes.create_string_buffer(16)
            res["fetch_first"] = g._lib.kombgpu_dist_graph_format_fetch(g._h, 0, buf, 0)
            res["which_low"] = _code(lambda: g.format(-1))
            res["which_high"] = _code(lambda: g.format(3))
            res["kcore_early"] = _code(lambda: g.format(1, h))
            res["corea_early"] = _code(lambda: g.format(2))
            g.coreness()
            res["kcore_no_names"] = _code(lambda: g.format(1))
            res["kcore_other_names"] = _code(lambda: g.format(1, h_other))
            res["corea_still_early"] = _code(lambda: g.format(2))
            g.corea()   # collective: the communicator still works
            res["files"] = [g.format(w, h) for w in FILES]
            # a graph built from pairs (a ring of 40) has no names of its own
            import torch
            dev = torch.device("cuda", comm.ctx.device)
            u = np.arange(40 * comm.rank // comm.world, 40 * (comm.rank + 1) // comm.world, dtype=np.int32)
            du, dv = torch.from_numpy(u).to(dev), torch.from_numpy((u + 1) % 40).to(dev)
            torch.cuda.synchronize(dev)
            with DistGraph.from_pairs(comm, du, dv, 40) as gp:
                gp.analyse()
                res["pairs_no_names"] = _code(lambda: gp.format(1))
                res["pairs_other_names"] = _code(lambda: gp.format(1, h))
                res["pairs_edges"] = gp.format(0)
        return res

    parts = _run(3, body)
    for p in parts:
        assert p["fetch_first"] == ESTATE
        assert p["which_low"] == EINVAL and p["which_high"] == EINVAL
        assert p["kcore_early"] == ESTATE and p["corea_early"] == ESTATE and p["corea_still_early"] == ESTATE
        assert p["kcore_no_names"] == EINVAL and p["kcore_other_names"] == EINVAL
        assert p["pairs_no_names"] == EINVAL and p["pairs_other_names"] == EINVAL
    for w in FILES:
        assert b"".join(p["files"][w] for p in parts) == exp[w]
    assert b"".join(p["pairs_edges"] for p in parts) == b"".join(b"%d\t%d\n" % e for e in sorted(
        (min(a, b), max(a, b)) for a, b in zip(range(40), [(x + 1) % 40 for x in range(40)])))


def test_parse_still_reports_its_timing():
    from komb_b200.peer import DistHits
    texts = _synth_pair()

    def body(comm):
        with DistHits.parse(comm, texts) as h:
            return h.timing()
    for t in _run(2, body):
        assert t["ms_intern"] > 0 and t["ms_route"] > 0


# ---- komb2 with KOMB_GPU_DEVICES: device output (default) against KOMB_OUTPUT=host and against one GPU

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
    env = {k: v for k, v in os.environ.items() if k not in ("KOMB_GPU_DEVICES", "KOMB_OUTPUT", "KOMB_TOKENIZE")}
    if multi:
        env["KOMB_GPU_DEVICES"] = _devices_env()
    env.update(env_extra)
    r = subprocess.run([KOMB2, "-t", "4", "-l", "100", "-o", str(out), "-i", str(tmp / "r1.sam"), "-j", str(tmp / "r2.sam"),
                        "-u", str(tmp / "u.fasta")], env=env, capture_output=True, text=True, timeout=600)
    return r, {p.name: p.read_bytes() for p in sorted(out.iterdir())}


@pytest.mark.parametrize("case", ["golden", "synth", "more_ranks_than_lines"])
def test_komb2_multi_gpu_device_output_matches_host_and_one_gpu(tmp_path, case):
    if case == "golden":
        sam1, sam2, _ = load_komb2_case(komb2_case_names()[0])
    elif case == "synth":
        sam1, sam2 = _synth_pair(n_unitigs=400, n_pairs=1500, unmapped_every=11)
    else:
        sam1, sam2 = EDGE_CASES[case]
    with _CTX.sam_parse([sam1, sam2]) as h:
        names = h.names()
    fasta = b"".join(b">%s LN:i:8\nACGTACGT\n" % nm for nm in names)
    env = {"KOMB_UNITIG_FASTA": "anomalous"}
    r_dev, f_dev = _komb2(tmp_path / "dev", sam1, sam2, fasta, env)
    r_host, f_host = _komb2(tmp_path / "host", sam1, sam2, fasta, dict(env, KOMB_OUTPUT="host"))
    r_one, f_one = _komb2(tmp_path / "one", sam1, sam2, fasta, env, multi=False)
    r_nofa, f_nofa = _komb2(tmp_path / "nofasta", sam1, sam2, fasta, {})
    for r in (r_dev, r_host, r_one, r_nofa):
        assert r.returncode == 0, r.stderr
    assert r_dev.stdout.count("\n") == r_host.stdout.count("\n")
    for f in ("edgelist.txt", "kcore.tsv", "CoreA_anomaly.txt", "anomalous_unitigs.fasta"):
        assert f in f_dev and f_dev[f] == f_host[f] == f_one[f], f
    for f in ("edgelist.txt", "kcore.tsv", "CoreA_anomaly.txt"):
        assert f_nofa[f] == f_dev[f], f
