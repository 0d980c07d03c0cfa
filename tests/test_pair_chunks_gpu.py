"""Clique pairs reduced in chunks (build.cu, chunked path): a build whose pairs reach 2^32 emits, sorts and reduces
them a chunk at a time and merges each chunk's (edge, count) list into the running one.

- Forcing chunks of any size (KOMBGPU_PAIR_CHUNK) leaves every output bit-identical to the one-shot path.
- A repeat-family hit set with P > 2^32 builds exactly: edges, multiplicities, degree and coreness against an analytic
  oracle (reads with the same unitig set collapse into one weighted clique), CORE-A against oracle.check_corea.
- graph_from_edges_dev takes 2^32 + 7 pairs; a multiplicity saturates at 2^32 - 1.
- More than 2^32 simple edges fail with KOMBGPU_EINVAL and leave the context usable.
- komb2 gives the same files with and without chunks, and builds the repeat-family SAM pair.

The test of the analytic oracle itself runs on the CPU.
"""
from pathlib import Path

import numpy as np
import pytest

from conftest import komb2_case_names, load_komb2_case
from komb_b200 import synth

ROOT = Path(__file__).resolve().parents[1]
KOMB2 = ROOT / "bin" / "komb2"

K_EMIT_TILE = 2048                        # build.cu kEmitTile: pairs per emission CTA
K_PAIR_CHUNK = (1 << 30) - (1 << 20)      # build.cu kPairChunk: the default chunk
EINVAL = -1


# ---- analytic oracle --------------------------------------------------------------------------------------------

def weighted_cliques(rk, ut):
    """Per read the set of its unitigs (src/graph.cpp:259-285); every i<j pair of a set (:332-347).  Reads with the
    same set emit the same pairs, so each distinct set is one clique weighted by its number of reads.  Returns the
    canonical packed edges (ascending), how many reads emitted each (uint64) and P, the pairs emitted in all."""
    key = np.unique((rk.astype(np.uint64) << np.uint64(32)) | ut.astype(np.uint64))
    r, u = key >> np.uint64(32), key & np.uint64(0xffffffff)
    starts = np.flatnonzero(np.r_[True, r[1:] != r[:-1]])
    ends = np.r_[starts[1:], len(r)]
    sets = {}
    for s, e in zip(starts.tolist(), ends.tolist()):
        if e - s >= 2:
            b = u[s:e].tobytes()
            sets[b] = sets.get(b, 0) + 1
    keys, wts, P = [], [], 0
    for b, w in sets.items():
        a = np.frombuffer(b, np.uint64)                  # ascending: (a[i], a[j]), i<j is already (min, max)
        iu, iv = np.triu_indices(a.shape[0], 1)
        keys.append((a[iu] << np.uint64(32)) | a[iv])
        wts.append(np.full(iu.shape[0], w, np.uint64))
        P += w * iu.shape[0]
    if not keys:
        return np.zeros(0, np.uint64), np.zeros(0, np.uint64), 0
    allk, allw = np.concatenate(keys), np.concatenate(wts)
    o = np.argsort(allk, kind="stable")
    allk, allw = allk[o], allw[o]
    heads = np.flatnonzero(np.r_[True, allk[1:] != allk[:-1]])
    return allk[heads], np.add.reduceat(allw, heads), P


def both_mates(m1, m2):
    return np.concatenate([m1.read_key, m2.read_key]), np.concatenate([m1.unitig, m2.unitig])


def test_weighted_cliques_oracle(oracle_mod):
    """CPU: the weighted-clique restatement equals the pair-by-pair one (every pair of every read, simplified by the C
    oracle, counted by numpy) on a small repeat-family instance."""
    m1, m2 = synth.repeat_family_hits(n_unitigs=600, family_size=40, overlap=6, reads_per_family=7, n_background=400, seed=3)
    rk, ut = both_mates(m1, m2)
    edges, mult, P = weighted_cliques(rk, ut)
    exp_edges, exp_p, _ = oracle_mod.build_edges(rk, ut)
    assert np.array_equal(edges, exp_edges) and P == exp_p
    key = np.unique((rk.astype(np.uint64) << np.uint64(32)) | ut.astype(np.uint64))
    r, u = key >> np.uint64(32), key & np.uint64(0xffffffff)
    pu, pv = [], []
    for rr in np.unique(r).tolist():
        a = u[r == rr]
        iu, iv = np.triu_indices(a.shape[0], 1)
        pu.append(a[iv]); pv.append(a[iu])              # reversed orientation: simplify canonicalises
    pu, pv = np.concatenate(pu).astype(np.uint32), np.concatenate(pv).astype(np.uint32)
    assert pu.shape[0] == P
    assert np.array_equal(oracle_mod.simplify(pu, pv), edges)
    pk, cnt = np.unique((np.minimum(pu, pv).astype(np.uint64) << np.uint64(32)) | np.maximum(pu, pv), return_counts=True)
    assert np.array_equal(pk, edges) and np.array_equal(cnt.astype(np.uint64), mult)
    assert mult.max() == 7 * 2 and mult.min() == 1      # unitigs shared by two families carry both families' reads


# ---- GPU ----------------------------------------------------------------------------------------------------------

@pytest.fixture(scope="module")
def ctx():
    import komb_b200
    c = komb_b200.Context(0)
    yield c
    c.close()


def snapshot(g):
    """Every output of a graph, for bit-for-bit comparison."""
    fp, fv = g.edges_csr()
    row_ptr, col = g.csr()
    st = g.stats()
    out = {"edges": g.edges(), "edges_csr": (fp, fv), "mult": g.edge_multiplicity(), "csr": (row_ptr, col),
           "degree": g.degree(), "coreness": g.coreness(),
           "corea_ref32": g.corea(0).view(np.uint64), "corea_exact64": g.corea(1).view(np.uint64),
           "summary": g.summary(),
           "stats": {k: st[k] for k in ("n_hits", "n_unique_hits", "n_pairs", "n_edges", "max_degree", "max_coreness",
                                        "peel_levels")}}
    return out


def assert_same(a, b):
    assert a.keys() == b.keys()
    for k in a:
        x, y = a[k], b[k]
        if isinstance(x, tuple) and x and isinstance(x[0], np.ndarray):
            assert all(np.array_equal(p, q) for p, q in zip(x, y)), k
        elif isinstance(x, np.ndarray):
            assert x.dtype == y.dtype and np.array_equal(x, y), k
        else:
            assert x == y, k


def caps_for(P):
    """Chunk caps: every cap on a small P; a cap under kEmitTile only where one chunk per pair or two stays quick."""
    caps = {-(-P // 3), P - 1, P}
    if P <= 300_000:
        caps |= {K_EMIT_TILE - 1, K_EMIT_TILE, K_EMIT_TILE + 1}
    if P <= 5_000:
        caps |= {1, 2}
    return sorted(c for c in caps if c >= 1)


def hit_inputs():
    """name -> (read_key, unitig, n_vertices)"""
    out = {}
    for seed, n, pairs in [(0, 1000, 15000), (1, 50000, 400000), (2, 300000, 3000000)]:   # test_gpu_parity's seeds
        out[f"metagenome_s{seed}"] = (*both_mates(*synth.metagenome_hits(n, pairs, seed=seed)), n)
    out["metagenome_tiny"] = (*both_mates(*synth.metagenome_hits(200, 400, seed=3)), 200)
    out["local_window"] = (*both_mates(*synth.metagenome_hits(20000, 150000, seed=5, local_window=64)), 20000)
    rk, ut = both_mates(*synth.metagenome_hits(20000, 150000, seed=9))
    o = np.random.default_rng(1).permutation(rk.shape[0])
    out["shuffled"] = (rk[o], ut[o], 20000)                       # out of read order: the sort path
    rng = np.random.default_rng(3)                                # reads with more than 64 hits: the look-back gives up
    rk = np.concatenate([np.full(700, 0), np.full(350, 1), np.repeat(np.arange(2, 2002), 2)]).astype(np.uint32)
    ut = np.concatenate([rng.integers(0, 5000, 700), rng.integers(0, 900, 350), rng.integers(0, 5000, 4000)]).astype(np.uint32)
    out["long_reads"] = (rk, ut, 5000)
    out["no_pairs"] = (np.arange(500, dtype=np.uint32), np.arange(500, dtype=np.uint32)[::-1].copy(), 500)
    out["one_read"] = (np.zeros(100, np.uint32), rng.permutation(3000)[:100].astype(np.uint32), 3000)
    return out


HIT_INPUTS = ["metagenome_s0", "metagenome_s1", "metagenome_s2", "metagenome_tiny", "local_window", "shuffled", "long_reads",
              "no_pairs", "one_read"] + [f"komb2_{n}" for n in komb2_case_names()]
_hit_cache = {}


def get_hits(oracle_mod, name):
    if name not in _hit_cache:
        if name.startswith("komb2_"):
            sam1, sam2, exp = load_komb2_case(name[len("komb2_"):])
            rk, ut, names = oracle_mod.intern_hits([oracle_mod.tokenise_sam(sam1, exp["threads"]),
                                                    oracle_mod.tokenise_sam(sam2, exp["threads"])])
            _hit_cache[name] = (rk, ut, len(names))
        else:
            _hit_cache.update(hit_inputs())
    return _hit_cache[name]


def build_hits(ctx, entry, rk, ut, n):
    """(graph, extra outputs) through one entry point that builds from hits"""
    if entry == "host":
        return ctx.build_graph(rk, ut, n), {}
    if entry == "device":
        import torch
        g = ctx.build_graph(torch.from_numpy(rk.view(np.int32)).cuda(), torch.from_numpy(ut.view(np.int32)).cuda(), n)
        return g, {}
    with ctx.build_graph(rk, ut, n) as g0:                       # size the caller's edge buffers
        cap = max(g0.counts()[1], 1)
    if entry == "analyse":
        g, r = ctx.analyse_hits(rk, ut, n, 1, edge_capacity=cap)
        return g, {k: r[k] for k in ("u", "v", "degree", "coreness", "score")}
    g, r = ctx.analyse_hits_csr(rk, ut, n, 0, edge_capacity=cap)
    return g, {k: r[k] for k in ("fwd_ptr", "v", "degree", "coreness", "score")}


def run_all_caps(monkeypatch, build):
    """build() with the knob unset, then under every cap: outputs bit-identical, the chunk count as planned"""
    monkeypatch.delenv("KOMBGPU_PAIR_CHUNK", raising=False)
    g, extra = build()
    with g:
        ref, ref_extra = snapshot(g), extra
        assert g.build_chunks() == 1
    P = ref["stats"]["n_pairs"]
    for cap in caps_for(P):
        monkeypatch.setenv("KOMBGPU_PAIR_CHUNK", str(cap))
        g, extra = build()
        with g:
            assert g.build_chunks() == (-(-P // cap) if P > cap else 1), cap
            assert_same(snapshot(g), ref)
            assert extra.keys() == ref_extra.keys()
            for k in extra:
                assert np.array_equal(extra[k], ref_extra[k]), (cap, k)
    monkeypatch.delenv("KOMBGPU_PAIR_CHUNK", raising=False)
    return P


@pytest.mark.gpu
@pytest.mark.parametrize("entry", ["host", "device", "analyse", "analyse_csr"])
@pytest.mark.parametrize("name", HIT_INPUTS)
def test_chunks_equal_one_shot_hits(ctx, oracle_mod, monkeypatch, name, entry):
    rk, ut, n = get_hits(oracle_mod, name)
    P = run_all_caps(monkeypatch, lambda: build_hits(ctx, entry, rk, ut, n))
    if name == "no_pairs":
        assert P == 0


@pytest.mark.gpu
@pytest.mark.parametrize("name", komb2_case_names() + ["rendered"])
def test_chunks_equal_one_shot_sam(ctx, monkeypatch, name):
    """sam_parse -> Hits.build_graph: the device tokeniser's hits"""
    if name == "rendered":
        m1, m2 = synth.metagenome_hits(3000, 20000, seed=6)
        texts = [synth.render_sam(m1, 3000, 1), synth.render_sam(m2, 3000, 2)]
    else:
        sam1, sam2, _ = load_komb2_case(name)
        texts = [sam1, sam2]
    with ctx.sam_parse(texts) as hits:
        run_all_caps(monkeypatch, lambda: (hits.build_graph(), {}))


def pair_inputs():
    u0, v0 = synth.rmat_edges(10, 3000, n_vertices=900, seed=0)          # duplicates, loops, both orientations
    u1, v1 = synth.rmat_edges(16, 600000, n_vertices=50000, seed=1)
    u2 = np.array([0, 1, 0, 2, 2, 3, 5, 5, 4, 1], np.uint32)
    v2 = np.array([1, 0, 1, 2, 3, 2, 5, 4, 5, 0], np.uint32)
    return {"rmat_small": (u0, v0, 900), "rmat_mid": (u1, v1, 50000), "hand": (u2, v2, 6)}


@pytest.mark.gpu
@pytest.mark.parametrize("entry", ["host", "device"])
@pytest.mark.parametrize("name", ["rmat_small", "rmat_mid", "hand"])
def test_chunks_equal_one_shot_pairs(ctx, monkeypatch, name, entry):
    u, v, n = pair_inputs()[name]
    if entry == "device":
        import torch
        du, dv = torch.from_numpy(u.view(np.int32)).cuda(), torch.from_numpy(v.view(np.int32)).cuda()
        build = lambda: (ctx.graph_from_edges(du, dv, n), {})   # noqa: E731
    else:
        build = lambda: (ctx.graph_from_edges(u, v, n), {})     # noqa: E731
    assert run_all_caps(monkeypatch, build) == u.shape[0]


# ---- P > 2^32 ---------------------------------------------------------------------------------------------------

@pytest.fixture(scope="module")
def repeat_families():
    m1, m2 = synth.repeat_family_hits()
    rk, ut = both_mates(m1, m2)
    edges, mult, P = weighted_cliques(rk, ut)
    return m1, m2, rk, ut, edges, mult, P


@pytest.mark.gpu
@pytest.mark.parametrize("entry", ["build_graph", "analyse_hits_csr"])
def test_more_than_2p32_pairs_from_hits(ctx, oracle_mod, monkeypatch, repeat_families, entry):
    monkeypatch.delenv("KOMBGPU_PAIR_CHUNK", raising=False)
    _, _, rk, ut, edges, mult, P = repeat_families
    n = 200_000
    assert P > 1 << 32 and P - 4_497_750_000 < 10_000_000
    exp_deg, exp_core = oracle_mod.coreness(n, edges)
    if entry == "build_graph":
        g = ctx.build_graph(rk, ut, n)
        fp, v = g.edges_csr()
        deg, core = g.degree(), g.coreness()
        score = g.corea(0)
    else:
        out = {"v": np.empty(edges.shape[0], np.uint32)}
        g, r = ctx.analyse_hits_csr(rk, ut, n, 0, out=out)
        fp, v, deg, core, score = r["fwd_ptr"], r["v"], r["degree"], r["coreness"], r["score"]
    with g:
        st = g.stats()
        assert st["n_pairs"] == P and st["n_edges"] == edges.shape[0]
        assert g.build_chunks() == -(-P // K_PAIR_CHUNK) and g.build_chunks() >= 5
        u = np.repeat(np.arange(n, dtype=np.uint32), np.diff(fp.astype(np.int64)))
        assert np.array_equal(oracle_mod.pack_edges(u, v), edges)
        assert np.array_equal(g.edge_multiplicity(), mult.astype(np.uint32))
        assert np.array_equal(deg, exp_deg) and np.array_equal(core, exp_core)
        oracle_mod.check_corea(score, exp_core, exp_deg, oracle_mod.KEY_REF32)
        if entry == "build_graph":
            oracle_mod.check_corea(g.corea(1), exp_core, exp_deg, oracle_mod.KEY_EXACT64)


def free_gb():
    import torch
    return torch.cuda.mem_get_info()[0] / 1e9


# 2^32 + 7 uint32 pairs are 34.4 GB on the device; the chunk buffers add 21.5 GB
FROM_EDGES_GB = 64


@pytest.mark.gpu
def test_from_edges_dev_2p32_plus_7_pairs(ctx, monkeypatch):
    import torch
    monkeypatch.delenv("KOMBGPU_PAIR_CHUNK", raising=False)
    if free_gb() < FROM_EDGES_GB:
        pytest.skip(f"needs {FROM_EDGES_GB} GB of free device memory for 2^32 + 7 input pairs, {free_gb():.0f} GB free")
    N = (1 << 32) + 7
    u = torch.full((N,), 3, dtype=torch.int32, device="cuda")
    v = torch.full((N,), 5, dtype=torch.int32, device="cuda")
    # a few other pairs, at both ends and across chunk boundaries: a duplicate in both orientations, loops, (3, 5) reversed
    at = [0, 1, K_PAIR_CHUNK - 1, K_PAIR_CHUNK, 3 * K_PAIR_CHUNK + 5, (1 << 32) - 1, 1 << 32, N - 1]
    uv = [(7, 2), (2, 7), (9, 9), (0, 1), (5, 3), (9, 9), (1, 8), (2, 7)]
    for p, (a, b) in zip(at, uv):
        u[p], v[p] = a, b
    torch.cuda.synchronize()
    with ctx.graph_from_edges(u, v, 10) as g:
        del u, v
        assert g.stats()["n_pairs"] == N
        assert g.build_chunks() == -(-N // K_PAIR_CHUNK)
        eu, ev = g.edges()
        got = dict(zip(zip(eu.tolist(), ev.tolist()), g.edge_multiplicity().tolist()))
        assert got == {(0, 1): 1, (1, 8): 1, (2, 7): 3, (3, 5): (1 << 32) - 1}


# one read with 92 683 distinct unitigs: C(92 683, 2) = 4 295 022 903 distinct edges; the running list at the limit
# (4.29e9 x 12 bytes) and the one before it plus the chunk buffers need about 112 GB
EDGE_LIMIT_GB = 120


@pytest.mark.gpu
def test_edge_limit_fails_cleanly(ctx, monkeypatch):
    import komb_b200
    monkeypatch.delenv("KOMBGPU_PAIR_CHUNK", raising=False)
    if free_gb() < EDGE_LIMIT_GB:
        pytest.skip(f"needs {EDGE_LIMIT_GB} GB of free device memory to reach 2^32 edges, {free_gb():.0f} GB free")
    k = 92_683
    assert k * (k - 1) // 2 == 4_295_022_903
    rk = np.zeros(k, np.uint32)
    ut = np.random.default_rng(5).permutation(k).astype(np.uint32)
    with pytest.raises(komb_b200.KombGpuError) as ei:
        ctx.build_graph(rk, ut, k)
    assert ei.value.code == EINVAL
    assert "per-device edge limit" in str(ei.value)
    ctx.trim()
    # the same context builds the next graph as a fresh one does
    rk2, ut2 = both_mates(*synth.metagenome_hits(50000, 400000, seed=1))
    with ctx.build_graph(rk2, ut2, 50000) as g:
        got = snapshot(g)
    fresh = komb_b200.Context(0)
    try:
        with fresh.build_graph(rk2, ut2, 50000) as g:
            assert_same(snapshot(g), got)
    finally:
        fresh.close()


# ---- komb2 --------------------------------------------------------------------------------------------------------

def run_komb2_files(oracle_mod, sam1, sam2, workdir, env):
    oracle_mod.run_komb2(KOMB2, sam1, sam2, workdir, extra_env=env)
    out = Path(workdir) / "out"
    return {f: (out / f).read_bytes() for f in ("edgelist.txt", "kcore.tsv", "CoreA_anomaly.txt")}


@pytest.mark.gpu
@pytest.mark.parametrize("name", komb2_case_names())
def test_komb2_files_identical_with_chunks(tmp_path, oracle_mod, monkeypatch, name):
    monkeypatch.delenv("KOMBGPU_PAIR_CHUNK", raising=False)
    sam1, sam2, _ = load_komb2_case(name)
    ref = run_komb2_files(oracle_mod, sam1, sam2, tmp_path / "ref", {})
    got = run_komb2_files(oracle_mod, sam1, sam2, tmp_path / "chunked", {"KOMBGPU_PAIR_CHUNK": "3"})
    assert got == ref


@pytest.mark.gpu
def test_komb2_more_than_2p32_pairs(tmp_path, oracle_mod, monkeypatch, repeat_families):
    monkeypatch.delenv("KOMBGPU_PAIR_CHUNK", raising=False)
    m1, m2, _, _, edges, _, P = repeat_families
    n = 200_000
    got, stdout = oracle_mod.run_komb2(KOMB2, synth.render_sam(m1, n, 1), synth.render_sam(m2, n, 2), tmp_path)
    hit = np.zeros(n, bool)
    hit[m1.unitig] = True
    hit[m2.unitig] = True
    deg, core = oracle_mod.coreness(n, edges)
    ids = np.flatnonzero(hit)                          # komb2's vertices: the unitigs that occur in the SAM files
    assert got["kcore"] == {str(i): (int(core[i]), int(deg[i])) for i in ids.tolist()}
    eu, ev = oracle_mod.unpack_edges(edges)
    assert got["edges"] == {tuple(sorted((str(a), str(b)))) for a, b in zip(eu.tolist(), ev.tolist())}
    score = oracle_mod.corea(core[ids], deg[ids], oracle_mod.KEY_REF32)
    for i, s in zip(ids.tolist(), score.tolist()):     # the reference prints "%f"
        assert abs(got["score"][str(i)] - s) <= 5.0e-7 + 1e-12
