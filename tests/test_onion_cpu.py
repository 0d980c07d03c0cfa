"""Onion layers without a GPU: the C restatement (tests/onion_ref.c) pinned to networkx.onion_layers and
networkx.core_number, the coreness a layering implies, and komb2's check of KOMB_ONION before any device work."""
import os
import subprocess
from pathlib import Path

import networkx as nx
import numpy as np
import pytest

from onion_ref import coreness_from_layers, onion_layers

ROOT = Path(__file__).resolve().parents[1]
KOMB2 = ROOT / "bin" / "komb2"


def _edges(G):
    e = np.array(list(G.edges()), np.int64).reshape(-1, 2)
    return e[:, 0].astype(np.uint32), e[:, 1].astype(np.uint32)


def _check(G):
    """The C restatement (tests/onion_ref.c) == networkx on G (vertices 0 .. n-1), its coreness == core_number, and
    the coreness implied by the layers == core_number."""
    n = G.number_of_nodes()
    assert sorted(G.nodes()) == list(range(n))
    u, v = _edges(G)
    layer, core, n_layers = onion_layers(n, u, v)
    exp = nx.onion_layers(G) if n else {}
    assert layer.tolist() == [exp[i] for i in range(n)]
    assert n_layers == (max(exp.values()) if n else 0)
    cn = nx.core_number(G) if n else {}
    assert core.tolist() == [cn[i] for i in range(n)]
    assert coreness_from_layers(n, u, v, layer).tolist() == [cn[i] for i in range(n)]


KNOWN = [
    ("path", nx.path_graph(5), {0: 1, 4: 1, 1: 2, 3: 2, 2: 3}),
    ("path_isolated", nx.union(nx.path_graph(5), nx.empty_graph(range(5, 10))), {9: 1, 0: 2, 4: 2, 1: 3, 3: 3, 2: 4}),
    ("k4", nx.complete_graph(4), {i: 1 for i in range(4)}),
    ("star", nx.star_graph(6), {0: 2, **{i: 1 for i in range(1, 7)}}),
    ("k4_path", nx.union(nx.complete_graph(4), nx.relabel_nodes(nx.path_graph(3), {0: 4, 1: 5, 2: 6})),
     {4: 1, 6: 1, 5: 2, 0: 3, 1: 3, 2: 3, 3: 3}),
]


@pytest.mark.parametrize("name,G,exp", KNOWN, ids=[k[0] for k in KNOWN])
def test_known_answers(name, G, exp):
    n = G.number_of_nodes()
    u, v = _edges(G)
    layer, _, _ = onion_layers(n, u, v)
    got = {i: int(layer[i]) for i in range(n) if i in exp}
    assert got == exp
    if name == "path_isolated":   # vertices 5..8 are isolated as well: layer 1 with 9
        assert layer[5:9].tolist() == [1] * 4
    _check(G)


def test_empty_and_edgeless():
    layer, core, nl = onion_layers(0, [], [])
    assert layer.shape == (0,) and core.shape == (0,) and nl == 0
    _check(nx.empty_graph(0))
    layer, core, nl = onion_layers(7, [], [])
    assert layer.tolist() == [1] * 7 and core.tolist() == [0] * 7 and nl == 1
    _check(nx.empty_graph(7))


@pytest.mark.parametrize("n", [1, 2, 3, 10, 101])
def test_paths_rings_stars_cliques(n):
    for G in (nx.path_graph(n), nx.cycle_graph(n) if n >= 3 else nx.path_graph(n), nx.star_graph(n), nx.complete_graph(n)):
        _check(nx.convert_node_labels_to_integers(G))


def test_disjoint_unions():
    G = nx.disjoint_union_all([nx.complete_graph(6), nx.path_graph(9), nx.cycle_graph(5), nx.star_graph(4), nx.empty_graph(3),
                               nx.complete_graph(3)])
    _check(G)


@pytest.mark.parametrize("seed", range(6))
def test_random_graphs(seed):
    _check(nx.gnp_random_graph(60 + 20 * seed, 0.02 + 0.03 * seed, seed=seed))
    _check(nx.barabasi_albert_graph(200 + 50 * seed, 1 + seed % 4, seed=seed))


def test_loops_and_duplicates_are_ignored():
    """The restatement works on the simple graph: self-loops and repeated pairs change nothing."""
    G = nx.barabasi_albert_graph(300, 3, seed=9)
    u, v = _edges(G)
    rng = np.random.default_rng(0)
    dup = rng.integers(0, u.shape[0], 200)
    loops = rng.integers(0, 300, 20).astype(np.uint32)
    uu = np.concatenate([u, v[dup], loops])
    vv = np.concatenate([v, u[dup], loops])
    assert np.array_equal(onion_layers(300, uu, vv)[0], onion_layers(300, u, v)[0])


def test_long_path_layers():
    """A path of 2 x 10^4 vertices peels from both ends: 10^4 layers, all at coreness 1."""
    n = 20_000
    u = np.arange(n - 1, dtype=np.uint32)
    layer, core, nl = onion_layers(n, u, u + 1)
    assert nl == n // 2
    assert np.array_equal(layer, np.minimum(np.arange(n), np.arange(n)[::-1]).astype(np.uint32) + 1)
    assert (core == 1).all()


def _komb2():
    if not KOMB2.exists():
        subprocess.run(["make", "-C", str(ROOT), "bin/komb2"], check=True, capture_output=True)
    return KOMB2


def test_komb2_rejects_onion_with_several_gpus(tmp_path):
    """KOMB_ONION=1 with several GPUs, or a value other than 0 / 1, exits 1 with a message before any device work."""
    (tmp_path / "r1.sam").write_bytes(b"r1/1\t0\tu1\t1\n")
    (tmp_path / "r2.sam").write_bytes(b"r1/2\t0\tu2\t1\n")
    (tmp_path / "u.fa").write_bytes(b">u1\nACGT\n>u2\nACGT\n")
    cmd = [str(_komb2()), "-i", str(tmp_path / "r1.sam"), "-j", str(tmp_path / "r2.sam"), "-u", str(tmp_path / "u.fa"), "-o", str(tmp_path)]
    for env, word in (({"KOMB_ONION": "1", "KOMB_GPU_DEVICES": "0,0"}, "needs one GPU"),
                      ({"KOMB_ONION": "1", "KOMB_GPU_DEVICES": "0,1,2"}, "needs one GPU"),
                      ({"KOMB_ONION": "yes"}, "KOMB_ONION=yes")):
        cp = subprocess.run(cmd, capture_output=True, text=True, env={**os.environ, **env})
        assert cp.returncode == 1 and word in cp.stderr, (env, cp.stderr)
        assert "cannot use CUDA device" not in cp.stderr
        assert not (tmp_path / "kcore.tsv").exists() and not (tmp_path / "onion.tsv").exists()
