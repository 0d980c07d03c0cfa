"""The unitig FASTA path on the device (include/kombgpu.h, unitig FASTA): record index, join by name, the IQR fence on
CORE-A and the extraction through the Python API, against the plain-Python restatements of
tests/test_unitig_fasta_cpu.py; and komb2 with KOMB_UNITIG_FASTA, whose other output files must not change."""
import os
import subprocess
from pathlib import Path

import numpy as np
import pytest

from conftest import corea_case_names, komb2_case_names, load_komb2_case, load_corea_case
from komb_b200 import synth
from test_unitig_fasta_cpu import extract_restated, fence_restated, parse_fasta

ROOT = Path(__file__).resolve().parents[1]
KOMB2 = ROOT / "bin" / "komb2"
EINVAL, ESTATE = -1, -5

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ctx():
    import komb_b200
    c = komb_b200.Context(0)
    yield c
    c.close()


def seq(rng, n: int) -> bytes:
    return np.frombuffer(b"ACGT", np.uint8)[rng.integers(0, 4, n)].tobytes()


def wrap(s: bytes, width: int = 60, eol: bytes = b"\n") -> bytes:
    return b"".join(s[i:i + width] + eol for i in range(0, len(s), width))


def make_fasta(names, seed: int, max_len: int = 400) -> bytes:
    """Records for `names` (in that order): lengths 31..max_len, every third one wrapped at 60 columns, every other
    header with a description (space or tab), one CRLF record in five, a blank line now and then."""
    rng = np.random.default_rng(seed)
    out = []
    for k, nm in enumerate(names):
        s = seq(rng, int(rng.integers(31, max_len)))
        desc = b"" if k % 2 else (b" LN:i:%d KC:i:7" % len(s) if k % 4 else b"\tlen=%d" % len(s))
        eol = b"\r\n" if k % 5 == 4 else b"\n"
        out.append(b">" + nm + desc + eol + (wrap(s, 60, eol) if k % 3 == 0 else s + eol))
        if k % 7 == 6:
            out.append(b"\n")
    return b"".join(out)


def check_index(ctx, text: bytes, seed: int = 0):
    """Counts, names (all join) and record spans (extraction) of the device index = the restatement's."""
    recs = parse_fasta(text)
    names = [r[2] for r in recs]
    rng = np.random.default_rng(seed)
    vnames = [names[i] for i in rng.permutation(len(names))]
    with ctx.fasta(text) as fa:
        assert fa.counts() == {"n_records": len(recs), "n_bytes": len(text)}
        assert fa.join(names=vnames) == 0
        n = len(vnames)
        for mask in (np.ones(n, bool), np.zeros(n, bool), rng.random(n) < 0.3, rng.random(n) < 0.01):
            assert fa.extract(mask) == extract_restated(text, recs, vnames, mask)
    return recs


def test_index_layouts(ctx):
    names = [b"u%d" % i for i in range(500)]
    text = make_fasta(names, 1)
    recs = check_index(ctx, text)
    assert [r[2] for r in recs] == names
    check_index(ctx, text[:-1], 2)                                   # unterminated last record: '\n' appended when selected
    check_index(ctx, text[:-1] + b"\r", 3)
    check_index(ctx, b"\n\r\n \t\n" + text, 4)                       # whitespace before the first record
    check_index(ctx, b">only", 5)
    check_index(ctx, b">a\n>b\n>c\n", 6)                              # empty sequences
    check_index(ctx, b">a\nAC>GT\n>b x>y\nA\n", 7)                    # '>' inside a line is sequence


def test_index_large_records(ctx):
    rng = np.random.default_rng(11)
    big = wrap(seq(rng, 4_500_000))                                  # one record of more than 4 MB among short ones
    text = b">s1\nACGT\n>big some description\n" + big + b">s2\n" + seq(rng, 70_001) + b"\n>s3\nA"
    check_index(ctx, text, 12)
    n = 1_000_000                                                    # 1 M small records
    lens = rng.integers(31, 64, n)
    pool = seq(rng, int(lens.sum()))
    ends = np.cumsum(lens)
    text = b"".join(b">r%d\n%s\n" % (i, pool[e - l:e]) for i, (e, l) in enumerate(zip(ends.tolist(), lens.tolist())))
    check_index(ctx, text, 13)


def test_index_empty_and_malformed(ctx):
    import komb_b200
    with ctx.fasta(b"") as fa:
        assert fa.counts() == {"n_records": 0, "n_bytes": 0}
        assert fa.join(names=[b"a", b"b"]) == 2
        assert fa.extract(np.zeros(2, bool)) == b""
    for bad, what in ((b"junk\n>a\nACGT\n", "before the first record"), (b">a\nA\n>\nA\n", "empty name"), (b"> a\nA\n", "empty name"),
                      (b">a x\nA\n>b\nC\n>a\nG\n", "repeats the name 'a'"), (b"ACGT", "before the first record")):
        with pytest.raises(komb_b200.KombGpuError, match=what) as e:
            ctx.fasta(bad)
        assert e.value.code == EINVAL
    with ctx.fasta(b">a\nA\n") as fa:                                 # the context stays usable
        assert fa.counts()["n_records"] == 1


@pytest.mark.parametrize("name", komb2_case_names())
def test_join_golden_sam_pairs(ctx, name):
    sam1, sam2, _ = load_komb2_case(name)
    rng = np.random.default_rng(len(name))
    with ctx.sam_parse([sam1, sam2]) as hits:
        vnames = hits.names()
        fnames = [vnames[i] for i in rng.permutation(len(vnames))] + [b"not_in_graph_%d" % i for i in range(50)]
        fnames = [fnames[i] for i in rng.permutation(len(fnames))]
        text = make_fasta(fnames, 3)
        recs = parse_fasta(text)
        mask = rng.random(len(vnames)) < 0.4
        with ctx.fasta(text) as fa:
            assert fa.join(hits=hits) == 0
            got_hits = fa.extract(mask)
            assert got_hits == extract_restated(text, recs, vnames, mask)
            assert fa.join(names=vnames) == 0
            assert fa.extract(mask) == got_hits
        dropped = set(rng.choice(len(vnames), size=max(1, len(vnames) // 10), replace=False).tolist())
        text2 = make_fasta([nm for nm in fnames if nm not in {vnames[v] for v in dropped}], 4)
        with ctx.fasta(text2) as fa:
            assert fa.join(hits=hits) == len(dropped)
            assert fa.join(names=vnames) == len(dropped)


def check_fence(got: dict, score):
    exp = fence_restated(score)
    assert (got["q1"], got["q3"], got["fence"], got["n_selected"]) == (exp["q1"], exp["q3"], exp["fence"], exp["n_selected"])
    assert np.array_equal(got["member"], exp["member"])
    if len(score):
        assert got["q1"] == np.percentile(score, 25, method="linear") and got["q3"] == np.percentile(score, 75, method="linear")


@pytest.mark.parametrize("name", corea_case_names())
def test_anomalous_golden_scores(ctx, name):
    _, _, score = load_corea_case(name)
    check_fence(ctx.anomalous(score), score)
    check_fence(ctx.anomalous(-score), -score)


def test_anomalous_small_and_special(ctx):
    import komb_b200
    rng = np.random.default_rng(8)
    for n in range(1, 6):
        for _ in range(20):
            x = np.round(rng.standard_normal(n) * 3, int(rng.integers(0, 3)))
            check_fence(ctx.anomalous(x), x)
    x = np.full(1000, 0.75)
    r = ctx.anomalous(x)
    check_fence(r, x)
    assert r["n_selected"] == 0
    x = -np.abs(rng.standard_normal(5000)) * 10
    x[::97] = 5.0
    check_fence(ctx.anomalous(x), x)
    x = np.array([1.0, 2.0, 3.0, 4.0, 40.0])
    assert ctx.anomalous(x, whisker=3.0)["fence"] == fence_restated(x, 3.0)["fence"]
    r = ctx.anomalous(np.zeros(0))
    assert (r["q1"], r["q3"], r["fence"], r["n_selected"]) == (0.0, 0.0, 0.0, 0) and r["member"].shape == (0,)
    with pytest.raises(komb_b200.KombGpuError, match="NaN") as e:
        ctx.anomalous(np.array([1.0, np.nan, 2.0]))
    assert e.value.code == EINVAL


@pytest.mark.parametrize("seed,n,n_pairs", [(0, 1000, 15000), (1, 50000, 400000), (2, 300000, 3000000)])
def test_graph_anomalous(ctx, seed, n, n_pairs):
    import komb_b200
    m1, m2 = synth.metagenome_hits(n, n_pairs, seed=seed)
    rk = np.concatenate([m1.read_key, m2.read_key])
    ut = np.concatenate([m1.unitig, m2.unitig])
    with ctx.build_graph(rk, ut, n) as g:
        g.coreness()
        with pytest.raises(komb_b200.KombGpuError) as e:
            g.anomalous()
        assert e.value.code == ESTATE
        score = g.corea()
        r = g.anomalous()
        check_fence(r, score)
        check_fence(ctx.anomalous(score), score)
        assert r["n_selected"] > 0


def test_extraction_masks(ctx):
    import komb_b200
    sam1, sam2, _ = load_komb2_case("wide_s4")
    rng = np.random.default_rng(21)
    with ctx.sam_parse([sam1, sam2]) as hits, hits.build_graph() as g:
        vnames = hits.names()
        n = len(vnames)
        g.coreness()
        tv = g.max_core_truss()["truss_vertices"]
        assert tv.shape[0] > 0
        text = make_fasta([vnames[i] for i in rng.permutation(n)], 22, max_len=40000)
        recs = parse_fasta(text)
        with ctx.fasta(text) as fa:
            assert fa.join(hits=hits) == 0
            for k in range(5):
                mask = rng.random(n) < (0.05, 0.3, 0.7, 0.95, 0.5)[k]
                assert fa.extract(mask) == extract_restated(text, recs, vnames, mask)
            assert fa.extract(np.zeros(n, bool)) == b""
            assert fa.extract(np.ones(n, bool)) == text[recs[0][0]:]
            tmask = np.zeros(n, bool)
            tmask[tv] = True
            assert fa.extract(tmask) == extract_restated(text, recs, vnames, tmask)
            with pytest.raises(komb_b200.KombGpuError, match="entries"):
                fa.extract(np.ones(n + 1, bool))
        # a selected vertex without a record: EINVAL naming it
        gone = int(tv[0])
        text2 = make_fasta([nm for nm in vnames if nm != vnames[gone]], 23)
        with ctx.fasta(text2) as fa:
            assert fa.join(hits=hits) == 1
            with pytest.raises(komb_b200.KombGpuError, match=rf"vertex {gone} \(unitig '{vnames[gone].decode()}'\)") as e:
                fa.extract(tmask)
            assert e.value.code == EINVAL
            tmask[gone] = False
            assert fa.extract(tmask) == extract_restated(text2, parse_fasta(text2), vnames, tmask)


# ---- komb2 with KOMB_UNITIG_FASTA ---------------------------------------------------------------------------------

def run_komb2(workdir: Path, sam1: bytes, sam2: bytes, fasta: bytes, threads: int = 2, env=None):
    workdir.mkdir(parents=True, exist_ok=True)
    out = workdir / "out"
    out.mkdir(exist_ok=True)
    (workdir / "r1.sam").write_bytes(sam1)
    (workdir / "r2.sam").write_bytes(sam2)
    (workdir / "unitigs.fasta").write_bytes(fasta)
    cp = subprocess.run([str(KOMB2), "-t", str(threads), "-l", "100", "-o", str(out), "-i", str(workdir / "r1.sam"), "-j", str(workdir / "r2.sam"),
                         "-u", str(workdir / "unitigs.fasta")], capture_output=True, text=True, env={**os.environ, **(env or {})})
    return cp, out


def expected_unitig_fastas(ctx, sam1, sam2, fasta):
    """What the Python API selects and extracts on the same SAM pair."""
    with ctx.sam_parse([sam1, sam2]) as hits, hits.build_graph() as g:
        g.coreness()
        g.corea()
        anom = g.anomalous()["member"]
        tmask = np.zeros(anom.shape[0], bool)
        tmask[g.max_core_truss()["truss_vertices"]] = True
        with ctx.fasta(fasta) as fa:
            assert fa.join(hits=hits) == 0
            return fa.extract(anom), fa.extract(tmask)


def golden_fasta(sam1, sam2, ctx, seed):
    with ctx.sam_parse([sam1, sam2]) as hits:
        names = hits.names()
    rng = np.random.default_rng(seed)
    return make_fasta([names[i] for i in rng.permutation(len(names))] + [b"extra_%d" % i for i in range(10)], seed), names


FILES = ("edgelist.txt", "kcore.tsv", "CoreA_anomaly.txt")


@pytest.mark.parametrize("name", [n for n in komb2_case_names() if not n.endswith("_t4")])
@pytest.mark.parametrize("tokenise,output", [("gpu", "gpu"), ("gpu", "host"), ("host", "host")])
def test_komb2_unitig_fasta(tmp_path, ctx, name, tokenise, output):
    sam1, sam2, _ = load_komb2_case(name)
    fasta, _ = golden_fasta(sam1, sam2, ctx, 31)
    mode = {"KOMB_TOKENIZE": tokenise, "KOMB_OUTPUT": output}
    cp0, out0 = run_komb2(tmp_path / "plain", sam1, sam2, fasta, env=mode)
    cp1, out1 = run_komb2(tmp_path / "fasta", sam1, sam2, fasta, env={**mode, "KOMB_UNITIG_FASTA": "anomalous,truss"})
    assert cp0.returncode == 0 and cp1.returncode == 0, cp1.stderr
    for f in FILES:
        assert (out1 / f).read_bytes() == (out0 / f).read_bytes(), f
    assert not (out0 / "anomalous_unitigs.fasta").exists() and not (out0 / "truss_unitigs.fasta").exists()
    exp_anom, exp_truss = expected_unitig_fastas(ctx, sam1, sam2, fasta)
    assert (out1 / "anomalous_unitigs.fasta").read_bytes() == exp_anom
    assert (out1 / "truss_unitigs.fasta").read_bytes() == exp_truss
    assert exp_truss


def _device_list():
    import torch
    n = torch.cuda.device_count()
    return ",".join(str(d) for d in range(min(n, 4))) if n >= 2 else "0,0,0"


@pytest.mark.parametrize("name", ["mid_s2", "quickstart_s1", "wide_s4"])
def test_komb2_unitig_fasta_multi_gpu(tmp_path, ctx, name):
    sam1, sam2, _ = load_komb2_case(name)
    fasta, _ = golden_fasta(sam1, sam2, ctx, 32)
    devs = {"KOMB_GPU_DEVICES": _device_list()}
    cp, out = run_komb2(tmp_path / "anom", sam1, sam2, fasta, threads=4, env={**devs, "KOMB_UNITIG_FASTA": "anomalous"})
    assert cp.returncode == 0, cp.stderr
    exp_anom, _ = expected_unitig_fastas(ctx, sam1, sam2, fasta)
    assert (out / "anomalous_unitigs.fasta").read_bytes() == exp_anom
    assert not (out / "truss_unitigs.fasta").exists()
    cp, out = run_komb2(tmp_path / "truss", sam1, sam2, fasta, threads=4, env={**devs, "KOMB_UNITIG_FASTA": "truss"})
    assert cp.returncode == 1 and "needs one GPU" in cp.stderr
    assert not (out / "kcore.tsv").exists()


def test_komb2_missing_selected_unitig(tmp_path, ctx):
    sam1, sam2, _ = load_komb2_case("wide_s4")
    with ctx.sam_parse([sam1, sam2]) as hits, hits.build_graph() as g:
        names = hits.names()
        g.coreness()
        gone = names[int(g.max_core_truss()["truss_vertices"][0])]
    fasta = make_fasta([nm for nm in names if nm != gone], 33)
    for tok in ("gpu", "host"):
        cp, _ = run_komb2(tmp_path / tok, sam1, sam2, fasta, env={"KOMB_UNITIG_FASTA": "truss", "KOMB_TOKENIZE": tok})
        assert cp.returncode == 1 and f"unitig '{gone.decode()}'" in cp.stderr, cp.stderr
