"""SAM text -> hits over the ranks of a communicator (kombgpu_dist_sam_parse) against kombgpu_sam_parse on one GPU:
the same unitig numbering and names, the same hits read by read, every read's hits on one rank, the same graph, the
same error message; and komb2 on several GPUs through it, against its host tokeniser.  The ranks are threads of
this process on device 0 (emulation) and, with two GPUs or more, on distinct devices."""
import collections
import os
import subprocess

import numpy as np
import pytest

from conftest import komb2_case_names, load_komb2_case
from komb_b200 import synth

pytestmark = pytest.mark.gpu

_CTX = None
REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
KOMB2 = os.path.join(REPO, "bin", "komb2")


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


def _single(texts):
    with _CTX.sam_parse(texts) as h:
        rk, ut = h.download()
        return h.counts(), h.names(), rk, ut


def _dist(world, texts, devices=None, build=False):
    from komb_b200.peer import DistGraph, DistHits, run_local

    def body(comm):
        with DistHits.parse(comm, texts) as h:
            out = {"counts": h.counts(), "range": h.local_range(), "names": h.names(), "hits": h.hits(), "timing": h.timing()}
            if build:
                with DistGraph.from_dist_hits(h) as g:
                    g.coreness()
                    g.corea()
                    out["graph"] = g.results()
                    out["edges"] = g.edges()
        return out
    return run_local(world, body, devices=devices)


def _reads(rk, ut):
    by = collections.defaultdict(list)
    for r, u in zip(rk.tolist(), ut.tolist()):
        by[r].append(u)
    return by


def _check_parity(texts, world, devices=None):
    counts, names, rk, ut = _single(texts)
    parts = _dist(world, texts, devices)
    for p in parts:
        c = p["counts"]
        assert (c["n_hits"], c["n_reads"], c["n_unitigs"], c["n_lines"]) == \
            (counts["n_hits"], counts["n_reads"], counts["n_unitigs"], counts["n_lines"])
    # the ranks' name ranges concatenate to the single-GPU names, vid by vid
    parts_by_lo = sorted(parts, key=lambda p: p["range"])
    assert [n for p in parts_by_lo for n in p["names"]] == names
    assert sum(p["counts"]["n_hits_local"] for p in parts) == counts["n_hits"]
    # every read's hits on exactly one rank, and the same multiset of per-read unitig lists
    seen, got = set(), collections.Counter()
    for p in parts:
        by = _reads(*p["hits"])
        assert not (seen & set(by)), "a read's hits are on two ranks"
        seen |= set(by)
        got.update(tuple(sorted(v)) for v in by.values())
    exp = collections.Counter(tuple(sorted(v)) for v in _reads(rk, ut).values())
    assert got == exp
    assert len(seen) == counts["n_reads"]
    return parts


WORLDS = [1, 2, 3, 4]


@pytest.mark.parametrize("world", WORLDS)
@pytest.mark.parametrize("name", komb2_case_names())
def test_golden_cases_match_single_gpu(name, world):
    sam1, sam2, _ = load_komb2_case(name)
    _check_parity([sam1, sam2], world)


def _synth_pair(n_unitigs=300, n_pairs=400, **kw):
    h1, h2 = synth.metagenome_hits(n_unitigs, n_pairs, seed=5)
    return [synth.render_sam(h1, n_unitigs, 1, **kw), synth.render_sam(h2, n_unitigs, 2, **kw)]


@pytest.mark.parametrize("world", WORLDS)
@pytest.mark.parametrize("kw", [{}, {"with_header": False}, {"unmapped_every": 7}, {"with_header": False, "unmapped_every": 3}])
def test_render_sam_matches_single_gpu(world, kw):
    _check_parity(_synth_pair(**kw), world)


REC = b"\t0\t%s\t1\t60\t4M\t*\t0\t0\tACGT\tIIII\n"


def _rec(q, r):
    return q + REC.replace(b"%s", r)


EDGE_CASES = {
    # @SQ lines below the first record: they still number before every hit
    "sq_below": [_rec(b"r1/1", b"uC") + b"@SQ\tSN:uB\tLN:4\n" + _rec(b"r2/1", b"uB") + b"@SQ\tSN:uC\tLN:4\n" + _rec(b"r3/1", b"uA"),
                 _rec(b"r1/2", b"uA") + b"@SQ\tSN:uA\tLN:4\n" + _rec(b"r2/2", b"uD")],
    # the last line has no '\n': it is not processed
    "unterminated": [_rec(b"r1/1", b"u1") + _rec(b"r2/1", b"u2") + b"r3/1\t0\tu3\t1",
                     _rec(b"r1/2", b"u2") + b"r9/2\t0\tu9"],
    "empty_file": [_rec(b"r1/1", b"u1") + _rec(b"r2/1", b"u2") + _rec(b"r3/1", b"u1"), b""],
    "both_empty": [b"", b""],
    "more_ranks_than_lines": [_rec(b"r1/1", b"u1"), _rec(b"r1/2", b"u2")],
    # read r0's mate-2 hits are at the END of file 2 (the last rank's slice), its mate-1 hits at the top of file 1
    "mate_far": [b"".join(_rec(b"r%d/1" % i, b"u%d" % (i % 13)) for i in range(40)),
                 b"".join(_rec(b"r%d/2" % i, b"u%d" % (i % 7 + 20)) for i in range(1, 40)) + _rec(b"r0/2", b"uFar") + _rec(b"r0/2", b"u3")],
    # long names: the strings that travel are longer than a warp
    "long_names": [b"".join(_rec(b"read%s%d/1" % (b"x" * 70, i), b"unitig_%s_%d" % (b"y" * (i % 90), i % 11)) for i in range(60)),
                   b"".join(_rec(b"read%s%d/2" % (b"x" * 70, i), b"unitig_%s_%d" % (b"y" * (i % 90), i % 17)) for i in range(60))],
}


@pytest.mark.parametrize("world", WORLDS)
@pytest.mark.parametrize("case", sorted(EDGE_CASES))
def test_edge_cases_match_single_gpu(case, world):
    _check_parity(EDGE_CASES[case], world)


def test_distinct_gpus_match_single_gpu():
    n = _n_devices()
    if n < 2:
        pytest.skip("one GPU: the emulated ranks above cover the protocol")
    world = min(n, 4)
    sam1, sam2, _ = load_komb2_case(komb2_case_names()[0])
    _check_parity([sam1, sam2], world, devices=list(range(world)))
    _check_parity(_synth_pair(unmapped_every=5), world, devices=list(range(world)))
    _check_parity(EDGE_CASES["mate_far"], world, devices=list(range(world)))


@pytest.mark.parametrize("world", [2, 3, 4])
def test_built_graph_matches_single_gpu(ctx, world):
    texts = _synth_pair(n_unitigs=500, n_pairs=900, unmapped_every=9)
    with ctx.sam_parse(texts) as h, h.build_graph() as g:
        exp = g.results()
    parts = sorted(_dist(world, texts, build=True), key=lambda p: p["graph"]["v_lo"] if len(p["graph"]["degree"]) else 1 << 40)
    u = np.concatenate([p["edges"][0] for p in parts])
    v = np.concatenate([p["edges"][1] for p in parts])
    assert np.array_equal(u, exp["u"]) and np.array_equal(v, exp["v"])
    for k in ("degree", "coreness"):
        assert np.array_equal(np.concatenate([p["graph"][k] for p in parts]), exp[k])
    assert np.allclose(np.concatenate([p["graph"]["score"] for p in parts]), exp["score"], rtol=0, atol=1e-9)


def test_malformed_line_fails_on_every_rank_with_the_single_gpu_message(ctx):
    import komb_b200
    from komb_b200.peer import DistHits, run_local
    good = _synth_pair(n_unitigs=50, n_pairs=80)
    lines = good[1].split(b"\n")
    # a line with two fields inside the third quarter of input 1: rank 2's slice of 4, plus a later empty line
    k = len(lines) * 5 // 8
    bad = [good[0], b"\n".join(lines[:k] + [b"r1/2\tonly_two"] + lines[k:k + 3] + [b""] + lines[k + 3:])]
    with pytest.raises(komb_b200.KombGpuError) as exc:
        ctx.sam_parse(bad)
    expect = str(exc.value)
    assert "fewer than 3" in expect and "input 1" in expect

    def body(comm):
        try:
            DistHits.parse(comm, bad)
            err = None
        except komb_b200.KombGpuError as e:
            err = (e.code, str(e))
        with DistHits.parse(comm, good) as h:   # the communicator is still usable
            n = h.counts()["n_hits"]
        return err, n
    res = run_local(4, body)
    n_exp = _single(good)[0]["n_hits"]
    for err, n in res:
        assert err is not None and err[0] == exc.value.code and err[1] == expect
        assert n == n_exp


def test_timing_and_counts_are_reported():
    parts = _dist(2, _synth_pair())
    for p in parts:
        t = p["timing"]
        assert t["ms_parse"] >= 0 and t["ms_intern"] > 0 and t["ms_route"] > 0 and t["hash_rounds"] >= 2


# ---- komb2 with KOMB_GPU_DEVICES: the partitioned parse (default) against the host tokeniser

def _devices_env():
    n = _n_devices()
    return ",".join(str(d) for d in range(min(n, 4))) if n >= 2 else "0,0,0"


def _fasta(names):
    return b"".join(b">%s LN:i:8\nACGTACGT\n" % nm for nm in names)


def _komb2(tmp, sam1, sam2, fasta, env_extra):
    tmp.mkdir(parents=True, exist_ok=True)
    (tmp / "r1.sam").write_bytes(sam1)
    (tmp / "r2.sam").write_bytes(sam2)
    (tmp / "u.fasta").write_bytes(fasta)
    out = tmp / "out"
    out.mkdir(exist_ok=True)
    env = dict(os.environ, KOMB_GPU_DEVICES=_devices_env(), **env_extra)
    r = subprocess.run([KOMB2, "-t", "4", "-l", "100", "-o", str(out), "-i", str(tmp / "r1.sam"), "-j", str(tmp / "r2.sam"),
                        "-u", str(tmp / "u.fasta")], env=env, capture_output=True, text=True, timeout=600)
    return r, {p.name: p.read_bytes() for p in sorted(out.iterdir())}


@pytest.mark.parametrize("case", ["golden", "synth"])
def test_komb2_multi_gpu_default_matches_host_tokeniser(tmp_path, case):
    if case == "golden":
        sam1, sam2, _ = load_komb2_case(komb2_case_names()[0])
    else:
        sam1, sam2 = _synth_pair(n_unitigs=400, n_pairs=1500, unmapped_every=11)
    names = _single([sam1, sam2])[1]
    fasta = _fasta(names)
    env = {"KOMB_UNITIG_FASTA": "anomalous"}
    r_dev, f_dev = _komb2(tmp_path / "dev", sam1, sam2, fasta, env)
    r_host, f_host = _komb2(tmp_path / "host", sam1, sam2, fasta, dict(env, KOMB_TOKENIZE="host"))
    assert r_dev.returncode == 0, r_dev.stderr
    assert r_host.returncode == 0, r_host.stderr
    for f in ("edgelist.txt", "kcore.tsv", "CoreA_anomaly.txt", "anomalous_unitigs.fasta"):
        assert f in f_dev and f_dev[f] == f_host[f], f


def test_komb2_multi_gpu_malformed_sam_exits_1(tmp_path):
    sam1, sam2 = _synth_pair(n_unitigs=40, n_pairs=60)
    bad = sam2 + b"r7/2\tonly_two\n"
    r, _ = _komb2(tmp_path, sam1, bad, b">0\nACGT\n", {})
    assert r.returncode == 1
    assert "malformed SAM" in r.stderr and "fewer than 3" in r.stderr
