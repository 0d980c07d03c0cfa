"""Onion layers on the device (kombgpu_graph_onion, Graph.onion, onion.tsv) against the C restatement of
networkx.onion_layers (tests/onion_ref.c, pinned to networkx by tests/test_onion_cpu.py): small shapes, R-MAT, a hub
sliced inside its layer, a long path, the reduced cfg5 ramp, a cfg2-size graph, the golden komb2 cases by name, and
komb2's onion.tsv."""
import os
import re
import subprocess
from pathlib import Path

import networkx as nx
import numpy as np
import pytest

from conftest import komb2_case_names, load_komb2_case
from komb_b200 import synth
from komb_b200._lib import EINVAL, ESTATE
from onion_ref import coreness_from_layers, onion_layers, simple_edges

pytestmark = pytest.mark.gpu

ROOT = Path(__file__).resolve().parents[1]
KOMB2 = ROOT / "bin" / "komb2"


@pytest.fixture(scope="module")
def ctx():
    import komb_b200
    c = komb_b200.Context(0)
    yield c
    c.close()


def check_graph(ctx, n, u, v, core=True):
    """Device layers bit-equal to the restatement on the simple graph of (u, v); the coreness they imply equals
    Graph.coreness().  Returns the device result."""
    exp_layer, exp_core, exp_n = onion_layers(n, u, v)
    with ctx.graph_from_edges(np.asarray(u, np.uint32), np.asarray(v, np.uint32), n) as g:
        r = g.onion()
        assert r["layer"].dtype == np.uint32 and r["layer"].shape == (n,)
        assert r["n_layers"] == exp_n
        assert np.array_equal(r["layer"], exp_layer)
        if core:
            c = g.coreness()
            assert np.array_equal(c, exp_core)
            a, b = simple_edges(u, v)
            assert np.array_equal(coreness_from_layers(n, a, b, r["layer"]), c)
    return r


def _nx(G):
    e = np.array(list(G.edges()), np.int64).reshape(-1, 2)
    return G.number_of_nodes(), e[:, 0].astype(np.uint32), e[:, 1].astype(np.uint32)


SHAPES = {
    "path5": nx.path_graph(5),
    "path5_isolated": nx.union(nx.path_graph(5), nx.empty_graph(range(5, 10))),
    "k4": nx.complete_graph(4),
    "star": nx.star_graph(6),
    "k4_path": nx.union(nx.complete_graph(4), nx.relabel_nodes(nx.path_graph(3), {0: 4, 1: 5, 2: 6})),
    "edgeless": nx.empty_graph(9),
    "ring": nx.cycle_graph(1000),
    "clique": nx.complete_graph(300),
    "big_star": nx.star_graph(20_000),
    "unions": nx.disjoint_union_all([nx.complete_graph(40), nx.path_graph(3000), nx.cycle_graph(77), nx.star_graph(900),
                                     nx.empty_graph(30), nx.barabasi_albert_graph(2000, 3, seed=1)]),
    "gnp": nx.gnp_random_graph(3000, 0.004, seed=3),
    "ba": nx.barabasi_albert_graph(20_000, 4, seed=5),
}


@pytest.mark.parametrize("name", list(SHAPES))
def test_shapes(ctx, name):
    n, u, v = _nx(SHAPES[name])
    r = check_graph(ctx, n, u, v)
    exp = nx.onion_layers(SHAPES[name]) if n <= 3000 else None
    if exp is not None:
        assert r["layer"].tolist() == [exp[i] for i in range(n)]


def test_empty_graph(ctx):
    with ctx.graph_from_edges(np.zeros(0, np.uint32), np.zeros(0, np.uint32), 0) as g:
        r = g.onion()
        assert r["layer"].shape == (0,) and r["n_layers"] == 0


@pytest.mark.parametrize("scale,draws", [(16, 500_000), (18, 3_000_000)])
def test_rmat(ctx, scale, draws):
    u, v = synth.rmat_edges(scale, draws, seed=scale)
    check_graph(ctx, 1 << scale, u, v)


def test_hub_sliced_inside_its_layer(ctx):
    """Level k = 2200 opens with one layer of the hub (degree k) and a K_{k+1}: too many vertices for one CTA, and
    every row longer than a slice.  The hub's 2200 neighbours (degree k + 1) fall to k only through the slices of the
    hub's row and must form the next layer, the two vertices left the one after."""
    k = 2200
    m = k + 2                                   # hub 0; vertices 1 .. m form K_m minus a matching on 1 .. k
    iu, iv = np.triu_indices(m, 1)
    keep = ~((iu % 2 == 0) & (iv == iu + 1) & (iv < k))
    u = np.concatenate([iu[keep] + 1, np.zeros(k, np.int64)])
    v = np.concatenate([iv[keep] + 1, np.arange(1, k + 1)])
    c0 = m + 1                                  # K_{k+1} on c0 .. c0 + k
    cu, cv = np.triu_indices(k + 1, 1)
    u = np.concatenate([u, cu + c0])
    v = np.concatenate([v, cv + c0])
    # plus a star whose centre is sliced in a layer of its own, after its 50 000 leaves
    s0 = c0 + k + 1
    u = np.concatenate([u, np.full(50_000, s0)])
    v = np.concatenate([v, np.arange(s0 + 1, s0 + 50_001)])
    n = s0 + 50_001
    r = check_graph(ctx, n, u, v)
    lay = r["layer"]
    hub_layer = int(lay[0])
    assert (lay[c0:c0 + k + 1] == hub_layer).all()
    assert (lay[1:k + 1] == hub_layer + 1).all() and (lay[k + 1:m + 1] == hub_layer + 2).all()
    assert lay[s0] == lay[s0 + 1] + 1


def test_long_path(ctx):
    """2 x 10^5 vertices: 10^5 layers, nearly all of them run by one CTA; nothing trips."""
    n = 200_000
    u = np.arange(n - 1, dtype=np.uint32)
    with ctx.graph_from_edges(u, u + 1, n) as g:
        r = g.onion()
        t = g.onion_timing()
    assert r["n_layers"] == n // 2
    assert np.array_equal(r["layer"], (np.minimum(np.arange(n), np.arange(n)[::-1]) + 1).astype(np.uint32))
    assert t["thin_layers"] >= n // 2 - 1 and t["levels"] == 1


def ramp_reduced():
    """The cfg5 ramp at a fifth of its depth (1000 levels x 40 unitigs) over an R-MAT background of 2 M unitigs."""
    n_bg = 2_000_000
    ru, rv = synth.ramp_edges(1000, 40)
    bu, bv = synth.rmat_edges(21, 8_000_000, n_bg, seed=7)
    u = np.concatenate([ru.astype(np.int64) + n_bg, bu])
    v = np.concatenate([rv.astype(np.int64) + n_bg, bv])
    return n_bg + 40_000, u.astype(np.uint32), v.astype(np.uint32)


def test_cfg5_ramp_reduced(ctx):
    n, u, v = ramp_reduced()
    r = check_graph(ctx, n, u, v)
    assert r["n_layers"] > 20_000


def test_cfg2_size(ctx):
    """bench.py's cfg2 workload (1 M unitigs, 5 M read pairs): layers and their coreness against the restatement."""
    m1, m2 = synth.metagenome_hits(1_000_000, 5_000_000, seed=11)
    rk = np.concatenate([m1.read_key, m2.read_key])
    ut = np.concatenate([m1.unitig, m2.unitig])
    with ctx.build_graph(rk, ut, 1_000_000) as g:
        u, v = g.edges()
        r = g.onion()
        core = g.coreness()
    exp_layer, exp_core, exp_n = onion_layers(1_000_000, u, v)
    assert r["n_layers"] == exp_n and np.array_equal(r["layer"], exp_layer)
    assert np.array_equal(core, exp_core)


def test_repeat_and_hit_order(ctx):
    """The same layers on every run and whatever order the hits come in; from_edges and from_csr graphs agree."""
    import torch
    m1, m2 = synth.metagenome_hits(30_000, 120_000, seed=3)
    rk = np.concatenate([m1.read_key, m2.read_key])
    ut = np.concatenate([m1.unitig, m2.unitig])
    with ctx.build_graph(rk, ut, 30_000) as g:
        first = g.onion()
        for _ in range(3):
            again = g.onion(again=True)
            assert again["n_layers"] == first["n_layers"] and np.array_equal(again["layer"], first["layer"])
        u, v = g.edges()
        row_ptr, col = g.csr()
    perm = np.random.default_rng(1).permutation(rk.shape[0])
    with ctx.build_graph(rk[perm], ut[perm], 30_000) as g:
        assert np.array_equal(g.onion()["layer"], first["layer"])
    with ctx.graph_from_edges(v, u, 30_000) as g:
        assert np.array_equal(g.onion()["layer"], first["layer"])
    rp = torch.from_numpy(row_ptr.view(np.int64)).cuda()
    cl = torch.from_numpy(col.view(np.int32)).cuda()
    with ctx.graph_from_csr(rp, cl, 30_000) as g:
        assert np.array_equal(g.onion()["layer"], first["layer"])
    exp_layer, _, _ = onion_layers(30_000, u, v)
    assert np.array_equal(first["layer"], exp_layer)


@pytest.mark.parametrize("name", [n for n in komb2_case_names() if not n.endswith("_t4")])
def test_golden_cases_by_name(ctx, name):
    """SAM pair -> device hits -> graph -> onion, against the restatement on the reference's own edge list, by Name;
    onion.tsv is kcore.tsv with the layer in the fourth column."""
    sam1, sam2, exp = load_komb2_case(name)
    ref_names = sorted(exp["kcore"])
    idx = {s: i for i, s in enumerate(ref_names)}
    eu = np.array([idx[a] for a, _ in exp["edges"]], np.uint32)
    ev = np.array([idx[b] for _, b in exp["edges"]], np.uint32)
    ref_layer, ref_core, ref_n = onion_layers(len(ref_names), eu, ev)
    with ctx.sam_parse([sam1, sam2]) as hits:
        names = hits.names()
        with hits.build_graph() as g:
            r = g.onion()
            assert r["n_layers"] == ref_n
            got = {names[i].decode(): int(r["layer"][i]) for i in range(len(names))}
            assert got == {s: int(ref_layer[idx[s]]) for s in ref_names}
            core = g.coreness()
            text = g.format(g.FILE_ONION, hits)
    assert text == b"#VID\tName\tCoreness\tLayer\n" + b"".join(
        b"%d\t%s\t%d\t%u\n" % (i, names[i], int(core[i]), int(r["layer"][i])) for i in range(len(names)))
    assert {names[i].decode(): int(core[i]) for i in range(len(names))} == {s: exp["kcore"][s][0] for s in ref_names}


def test_format_state_and_errors(ctx):
    import komb_b200
    sam1, sam2, _ = load_komb2_case("quickstart_s1")
    with ctx.sam_parse([sam1, sam2]) as hits, hits.build_graph() as g:
        with pytest.raises(komb_b200.KombGpuError) as e:
            g.format(g.FILE_ONION, hits)                        # the onion has not run: state
        assert e.value.code == ESTATE
        g.onion()                                               # needs no coreness
        with pytest.raises(komb_b200.KombGpuError, match="names") as e:
            g.format(g.FILE_ONION)                              # no names
        assert e.value.code == EINVAL
        with ctx.sam_parse([b"a/1\t0\tu1\t1\n", b"a/2\t0\tu2\t1\n"]) as other:
            with pytest.raises(komb_b200.KombGpuError, match="names") as e:
                g.format(g.FILE_ONION, other)                   # names of another graph
            assert e.value.code == EINVAL
        t1 = g.format(g.FILE_ONION, hits)
        assert t1 == g.format(g.FILE_ONION, hits)               # cached
        with pytest.raises(komb_b200.KombGpuError) as e:
            g.format(4, hits)
        assert e.value.code == EINVAL
    with ctx.build_graph(np.array([0, 0, 1, 1], np.uint32), np.array([0, 1, 1, 2], np.uint32), 3) as g2:
        assert g2.onion()["layer"].tolist() == [1, 2, 1]


# ---- komb2 with KOMB_ONION ------------------------------------------------------------------------------------------

FILES = ("edgelist.txt", "kcore.tsv", "CoreA_anomaly.txt")


def run_komb2(workdir: Path, sam1: bytes, sam2: bytes, env=None):
    workdir.mkdir(parents=True, exist_ok=True)
    out = workdir / "out"
    out.mkdir(exist_ok=True)
    (workdir / "r1.sam").write_bytes(sam1)
    (workdir / "r2.sam").write_bytes(sam2)
    (workdir / "unitigs.fasta").write_bytes(b">u\nACGT\n")
    cp = subprocess.run([str(KOMB2), "-t", "2", "-l", "100", "-o", str(out), "-i", str(workdir / "r1.sam"), "-j", str(workdir / "r2.sam"),
                         "-u", str(workdir / "unitigs.fasta")], capture_output=True, text=True, env={**os.environ, **(env or {})})
    return cp, out


def _rows(path, cols):
    lines = path.read_text().splitlines()
    return lines[0], [tuple(ln.split("\t")[:cols]) for ln in lines[1:]]


@pytest.mark.parametrize("name", ["mid_s2", "quickstart_s1", "wide_s4"])
def test_komb2_onion_tsv(tmp_path, name):
    """KOMB_ONION=1: the three files and stdout as without it; onion.tsv byte-identical whether formatted on the device
    or on the host, its rows those of kcore.tsv with the layer, and the layers those of the restatement by name."""
    sam1, sam2, exp = load_komb2_case(name)
    onion = {}
    for mode, base in (("gpu", {}), ("gpu_host_out", {"KOMB_OUTPUT": "host"}), ("host", {"KOMB_TOKENIZE": "host"})):
        cp0, out0 = run_komb2(tmp_path / mode / "plain", sam1, sam2, base)
        cp1, out1 = run_komb2(tmp_path / mode / "onion", sam1, sam2, {**base, "KOMB_ONION": "1"})
        assert cp0.returncode == 0 and cp1.returncode == 0, cp1.stderr
        assert not (out0 / "onion.tsv").exists()
        assert re.sub(r"[0-9.]+", "#", cp1.stdout) == re.sub(r"[0-9.]+", "#", cp0.stdout)   # the same lines but for timings
        for f in FILES:
            assert (out1 / f).read_bytes() == (out0 / f).read_bytes(), (mode, f)
        head, rows = _rows(out1 / "onion.tsv", 4)
        assert head == "#VID\tName\tCoreness\tLayer"
        assert [r[:3] for r in rows] == _rows(out1 / "kcore.tsv", 3)[1]
        onion[mode] = (out1 / "onion.tsv").read_bytes()
    assert onion["gpu_host_out"] == onion["gpu"]
    ref_names = sorted(exp["kcore"])
    idx = {s: i for i, s in enumerate(ref_names)}
    eu = np.array([idx[a] for a, _ in exp["edges"]], np.uint32)
    ev = np.array([idx[b] for _, b in exp["edges"]], np.uint32)
    ref_layer, _, _ = onion_layers(len(ref_names), eu, ev)
    for mode in ("gpu", "host"):
        _, rows = _rows(tmp_path / mode / "onion" / "out" / "onion.tsv", 4)
        assert {r[1]: (int(r[2]), int(r[3])) for r in rows} == {s: (exp["kcore"][s][0], int(ref_layer[idx[s]])) for s in ref_names}
