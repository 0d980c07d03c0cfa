"""The unitig FASTA path without a GPU: the plain-Python restatement of the IQR fence (include/kombgpu.h, unitig FASTA)
against hand-computed answers and numpy, and komb2's check of KOMB_UNITIG_FASTA before any device work.  The
restatements here (FASTA records, fence, extraction) are what tests/test_unitig_fasta_gpu.py compares the device
against."""
import math
import os
import subprocess
from pathlib import Path

import numpy as np
import pytest

ROOT = Path(__file__).resolve().parents[1]
KOMB2 = ROOT / "bin" / "komb2"
SPACE = b" \t\r\n\v\f"


class FastaError(ValueError):
    pass


def parse_fasta(text: bytes) -> list[tuple[int, int, bytes]]:
    """(start, end, name) of every record: a record starts at a '>' at offset 0 or right after '\\n' and runs to the
    next start or the end of the file; the name is the bytes after '>' up to the first whitespace byte."""
    starts = [i for i in range(len(text)) if text[i:i + 1] == b">" and (i == 0 or text[i - 1:i] == b"\n")] \
        if len(text) < 1 << 16 else _starts_fast(text)
    first = starts[0] if starts else len(text)
    if text[:first].strip(SPACE):
        raise FastaError("bytes before the first record")
    recs, seen = [], set()
    for k, s in enumerate(starts):
        e = starts[k + 1] if k + 1 < len(starts) else len(text)
        i = s + 1
        while i < e and text[i] not in SPACE:
            i += 1
        name = text[s + 1:i]
        if not name:
            raise FastaError("empty name")
        if name in seen:
            raise FastaError("duplicate name")
        seen.add(name)
        recs.append((s, e, name))
    return recs


def _starts_fast(text: bytes) -> list[int]:
    a = np.frombuffer(text, np.uint8)
    gt = np.flatnonzero(a == ord(">"))
    return [int(i) for i in gt if i == 0 or a[i - 1] == ord("\n")]


def extract_restated(text: bytes, recs, vertex_names, mask) -> bytes:
    """The records of the selected vertices, verbatim, in file order; '\\n' after an unterminated selected last record."""
    chosen = {bytes(vertex_names[v]) for v in np.flatnonzero(np.asarray(mask, bool))}
    out = []
    for k, (s, e, name) in enumerate(recs):
        if name in chosen:
            out.append(text[s:e])
            if k == len(recs) - 1 and not text.endswith(b"\n"):
                out.append(b"\n")
    return b"".join(out)


def quartile_restated(s: list[float], p: float) -> float:
    """numpy.percentile(..., method="linear") of the ascending list s, operation by operation, in float64."""
    n = len(s)
    h = n * p - p
    i = math.floor(h)
    j = min(i + 1, n - 1)
    t = h - i
    d = s[j] - s[i]
    return s[i] + d * t if t < 0.5 else s[j] - d * (1 - t)


def fence_restated(score, whisker: float = 1.5) -> dict:
    x = [float(v) for v in np.asarray(score, np.float64)]
    if any(v != v for v in x):
        raise FastaError("NaN score")
    if not x:
        return {"q1": 0.0, "q3": 0.0, "fence": 0.0, "n_selected": 0, "member": np.zeros(0, bool)}
    s = sorted(x)
    q1, q3 = quartile_restated(s, 0.25), quartile_restated(s, 0.75)
    fence = q3 + whisker * (q3 - q1)
    member = np.array([v > fence for v in x], bool)
    return {"q1": q1, "q3": q3, "fence": fence, "n_selected": int(member.sum()), "member": member}


def test_fence_restatement_hand_computed():
    r = fence_restated([1, 2, 3, 4])
    assert (r["q1"], r["q3"], r["fence"]) == (1.75, 3.25, 5.5) and r["n_selected"] == 0
    r = fence_restated([4, 1, 3, 2, 100])
    assert (r["q1"], r["q3"], r["fence"]) == (2.0, 4.0, 7.0) and r["member"].tolist() == [False, False, False, False, True]
    r = fence_restated([7.0])
    assert (r["q1"], r["q3"], r["fence"], r["n_selected"]) == (7.0, 7.0, 7.0, 0)
    r = fence_restated([-3.0, -1.0])
    assert (r["q1"], r["q3"]) == (-2.5, -1.5) and r["fence"] == -1.5 + 1.5 * 1.0
    r = fence_restated([2.0] * 6)
    assert r["fence"] == 2.0 and r["n_selected"] == 0
    assert fence_restated([])["n_selected"] == 0
    with pytest.raises(FastaError):
        fence_restated([1.0, float("nan")])


@pytest.mark.parametrize("n", range(1, 10))
def test_fence_restatement_matches_numpy(n):
    rng = np.random.default_rng(n)
    for trial in range(300):
        x = rng.standard_normal(n) * 10.0 ** rng.integers(-3, 4)
        if trial % 3 == 0:
            x = np.round(x, 1)     # ties
        s = sorted(x.tolist())
        for p in (0.25, 0.75):
            assert quartile_restated(s, p) == np.percentile(x, 100 * p, method="linear")


def test_fasta_restatement():
    text = b"\n>a desc\nAC\nGT\n>b\tx\r\nGG\r\n\n>c"
    assert parse_fasta(text) == [(1, 15, b"a"), (15, 26, b"b"), (26, 28, b"c")]
    assert extract_restated(text, parse_fasta(text), [b"c", b"a"], [1, 1]) == b">a desc\nAC\nGT\n>c\n"
    assert parse_fasta(b"") == [] and parse_fasta(b" \n\t") == []
    assert parse_fasta(b">x\nA>y\n") == [(0, 7, b"x")]      # '>' inside a line is sequence
    for bad in (b"junk\n>a\nA\n", b">\nA\n", b"> a\nA\n", b">a\nA\n>a\nC\n", b"x"):
        with pytest.raises(FastaError):
            parse_fasta(bad)


def _komb2():
    if not KOMB2.exists():
        subprocess.run(["make", "-C", str(ROOT), "bin/komb2"], check=True, capture_output=True)
    return KOMB2


def test_komb2_rejects_unknown_unitig_fasta_words(tmp_path):
    """An unknown KOMB_UNITIG_FASTA word, or truss with several GPUs, exits 1 with a message before any device work."""
    (tmp_path / "r1.sam").write_bytes(b"r1/1\t0\tu1\t1\n")
    (tmp_path / "r2.sam").write_bytes(b"r1/2\t0\tu2\t1\n")
    (tmp_path / "u.fa").write_bytes(b">u1\nACGT\n>u2\nACGT\n")
    cmd = [str(_komb2()), "-i", str(tmp_path / "r1.sam"), "-j", str(tmp_path / "r2.sam"), "-u", str(tmp_path / "u.fa"), "-o", str(tmp_path)]
    for env, word in (({"KOMB_UNITIG_FASTA": "bogus"}, "bogus"), ({"KOMB_UNITIG_FASTA": "anomalous,trus"}, "trus"),
                      ({"KOMB_UNITIG_FASTA": "truss", "KOMB_GPU_DEVICES": "0,0"}, "needs one GPU")):
        cp = subprocess.run(cmd, capture_output=True, text=True, env={**os.environ, **env})
        assert cp.returncode == 1 and word in cp.stderr, (env, cp.stderr)
        assert "cannot use CUDA device" not in cp.stderr
        assert not (tmp_path / "kcore.tsv").exists()
