"""Clique pairs of the peer-memory multi-GPU build reduced in rounds (pbuild.cu): when the pairs of all ranks reach 2^32
(or some rank's exceed KOMBGPU_PAIR_CHUNK), every rank emits its next pairs, routes them to the owner of min(u, v), and
the owner sorts them and merges their (edge, count) list into its running slice, round after round.

- Forcing rounds of any size leaves every rank's outputs bit-identical to the one-shot multi-GPU build and to the
  single-GPU build's slice, over 1, 2 and 3 ranks, from hits and from pairs; the round count is as planned.
- One rank whose own pairs exceed 2^32, and an owner that receives more than 2^32 pairs while every rank emits fewer,
  build exactly (edges, multiplicities, degree, coreness against the weighted-clique oracle; CORE-A by check_corea).
- A rank that fails in a late round makes every rank fail with KOMBGPU_EINVAL, and the communicator builds on.
- komb2 over several ranks writes the same files with rounds of 3 pairs, and builds the repeat-family SAM pair.

Ranks are emulated (threads of this process, every rank on device 0), and run one GPU per rank where the box has enough.
"""
import numpy as np
import pytest

from conftest import komb2_case_names, load_komb2_case
from komb_b200 import synth
from test_pair_chunks_gpu import (EINVAL, K_PAIR_CHUNK, KOMB2, both_mates, free_gb, get_hits, pair_inputs, run_komb2_files,
                                  weighted_cliques)

pytestmark = pytest.mark.gpu

N_REPEAT = 200_000   # unitigs of synth.repeat_family_hits
# Device memory the repeat-family builds take with every rank on one device, measured with tools/dist_pair_chunk_probe.py
# (profiles/r3/r3c_dist_pair_chunk_probe.json): 51.0 GB for 2 ranks (a rank holds one round: its pairs, the receive
# buffer, the sort's second buffer and the counts), 81.1 GB for 3; plus a margin.  komb2's repeat case runs 3 ranks.
RANGE_W2_GB = 60
ROUNDROBIN_W3_GB = 90


def n_gpus():
    import torch
    return torch.cuda.device_count()


def placement_devices(placement, world):
    if placement == "emulated":
        return None
    if n_gpus() < world:
        pytest.skip(f"needs {world} GPUs, the box has {n_gpus()}")
    return list(range(world))


def split_hits(rk, ut, rank, world, how="range"):
    """A read's hits stay on one rank: by read range (komb2's split), or whole reads dealt round-robin."""
    if how == "range":
        reads = int(rk.max()) + 1 if rk.size else 0
        sel = (rk >= reads * rank // world) & (rk < reads * (rank + 1) // world)
    else:
        sel = rk % world == rank
    return rk[sel], ut[sel]


def split_pairs(u, v, rank, world):
    sl = slice(len(u) * rank // world, len(u) * (rank + 1) // world)
    return u[sl], v[sl]


def dist_snapshot(g):
    """Every output of one rank's share, for bit-for-bit comparison."""
    u, v, mult = g.edges(with_mult=True)
    fp, fv = g.edges_csr()
    g.coreness()
    g.corea(0)
    r = g.results()
    summary = g.summary()
    score32 = r["score"].view(np.uint64).copy()
    g.corea(1)
    score64 = g.results()["score"].view(np.uint64).copy()
    st = g.stats()
    return {"edges": (u, v), "mult": mult, "edges_csr": (fp, fv), "degree": r["degree"], "coreness": r["coreness"],
            "corea_ref32": score32, "corea_exact64": score64, "summary": summary,
            "stats": {k: st[k] for k in ("v_lo", "n_local", "n_fwd_local", "n_edges_global", "n_pairs_local", "n_pairs_received",
                                         "n_directed_local", "max_degree", "max_coreness")},
            "rounds": g.build_rounds()}


def dist_build(kind, a, b, n, world, devices=None, how="range"):
    """Every rank's snapshot of a multi-GPU build of the whole input (a, b)."""
    from komb_b200.peer import DistGraph, run_local

    def body(comm):
        import torch
        x, y = split_hits(a, b, comm.rank, world, how) if kind == "hits" else split_pairs(a, b, comm.rank, world)
        dev = torch.device("cuda", comm.ctx.device)
        tx, ty = torch.from_numpy(x.view(np.int32)).to(dev), torch.from_numpy(y.view(np.int32)).to(dev)
        torch.cuda.synchronize(dev)
        build = DistGraph.from_hits if kind == "hits" else DistGraph.from_pairs
        with build(comm, tx, ty, n) as g:
            return dist_snapshot(g)
    return run_local(world, body, devices=devices)


def same(x, y):
    if isinstance(x, tuple) and x and isinstance(x[0], np.ndarray):
        return len(x) == len(y) and all(p.dtype == q.dtype and np.array_equal(p, q) for p, q in zip(x, y))
    if isinstance(x, np.ndarray):
        return x.dtype == y.dtype and np.array_equal(x, y)
    return x == y


def single_slice(ref, v_lo, n_local):
    """The single-GPU build's outputs restricted to the unitigs [v_lo, v_lo + n_local) one rank owns."""
    u, v = ref["edges"]
    sel = (u >= v_lo) & (u < v_lo + n_local)
    fp, fv = ref["edges_csr"]
    fp = fp.astype(np.uint64)
    rows = fp[v_lo:v_lo + n_local + 1]
    lo = rows[0] if rows.size else np.uint64(0)
    vs = slice(v_lo, v_lo + n_local)
    return {"edges": (u[sel], v[sel]), "mult": ref["mult"][sel], "edges_csr": (rows - lo, fv[int(lo):int(lo) + int(sel.sum())]),
            "degree": ref["degree"][vs], "coreness": ref["coreness"][vs], "corea_ref32": ref["corea_ref32"][vs],
            "corea_exact64": ref["corea_exact64"][vs], "summary": ref["summary"]}


def single_build(kind, a, b, n):
    import komb_b200
    ctx = komb_b200.Context(0)
    try:
        with (ctx.build_graph(a, b, n) if kind == "hits" else ctx.graph_from_edges(a, b, n)) as g:
            fp, fv = g.edges_csr()
            out = {"edges": g.edges(), "mult": g.edge_multiplicity(), "edges_csr": (fp, fv), "degree": g.degree(),
                   "coreness": g.coreness(), "corea_ref32": g.corea(0).view(np.uint64).copy()}
            out["summary"] = g.summary()
            out["corea_exact64"] = g.corea(1).view(np.uint64).copy()
            return out
    finally:
        ctx.close()


def planned_rounds(p_local, world, cap):
    """pbuild.cu's decision: one shot while the pairs of all ranks stay below 2^32 and no rank's exceed the cap."""
    max_p, sum_p = max(p_local), sum(p_local)
    if cap and max_p > cap:
        chunk = min(cap, 0xffffffff // world)
    elif sum_p >= 1 << 32:
        chunk = K_PAIR_CHUNK // world
    else:
        return 1
    return -(-max_p // chunk)


MAX_ROUNDS = 1500   # caps of 1 and 3 pairs only where the rounds stay this few (every round meets the other ranks twice)


def caps_for(max_p):
    caps = {1, 3, 1000, max_p - 1}
    return sorted(c for c in caps if c >= 1 and -(-max_p // c) <= MAX_ROUNDS)


def small_repeat_family():
    return both_mates(*synth.repeat_family_hits(n_unitigs=600, family_size=40, overlap=6, reads_per_family=7, n_background=400,
                                                seed=3)) + (600,)


INPUTS = [f"komb2_{n}" for n in komb2_case_names()] + ["metagenome_tiny", "metagenome_s0", "repeat_small", "pairs_rmat_small",
                                                      "pairs_hand"]


def get_input(oracle_mod, name):
    if name == "repeat_small":
        return ("hits",) + small_repeat_family()
    if name.startswith("pairs_"):
        return ("pairs",) + pair_inputs()[name[len("pairs_"):]]
    return ("hits",) + get_hits(oracle_mod, name)


@pytest.mark.parametrize("world,placement", [(1, "emulated"), (2, "emulated"), (3, "emulated"), (2, "gpus"), (3, "gpus")])
@pytest.mark.parametrize("name", INPUTS)
def test_rounds_equal_one_shot(oracle_mod, monkeypatch, name, world, placement):
    devices = placement_devices(placement, world)
    kind, a, b, n = get_input(oracle_mod, name)
    monkeypatch.delenv("KOMBGPU_PAIR_CHUNK", raising=False)
    ref = dist_build(kind, a, b, n, world, devices)
    single = single_build(kind, a, b, n)
    p_local = [p["stats"]["n_pairs_local"] for p in ref]
    assert all(p["rounds"] == 1 for p in ref)
    for p in ref:
        exp = single_slice(single, p["stats"]["v_lo"], p["stats"]["n_local"])
        for k, x in exp.items():
            assert same(p[k], x), (k, p["stats"]["v_lo"])
    if name == "repeat_small":                       # cliques of 780 pairs: a cap of 1000 cuts through them
        assert max(p_local) > 3000
    for cap in caps_for(max(p_local)):
        monkeypatch.setenv("KOMBGPU_PAIR_CHUNK", str(cap))
        got = dist_build(kind, a, b, n, world, devices)
        for p, q in zip(got, ref):
            assert p["rounds"] == planned_rounds(p_local, world, cap), cap
            for k in q:
                if k != "rounds":
                    assert same(p[k], q[k]), (cap, k, p["stats"]["v_lo"])
    monkeypatch.delenv("KOMBGPU_PAIR_CHUNK", raising=False)


# ---- more than 2^32 pairs ------------------------------------------------------------------------------------------

def repeat_instance(**kw):
    rk, ut = both_mates(*synth.repeat_family_hits(**kw))
    edges, mult, P = weighted_cliques(rk, ut)
    return rk, ut, edges, mult, P


def check_exact(oracle_mod, parts, edges, mult):
    parts = sorted(parts, key=lambda p: p["stats"]["v_lo"])
    u = np.concatenate([p["edges"][0] for p in parts])
    v = np.concatenate([p["edges"][1] for p in parts])
    assert np.array_equal(oracle_mod.pack_edges(u, v), edges)
    assert np.array_equal(np.concatenate([p["mult"] for p in parts]), mult.astype(np.uint32))
    deg, core = oracle_mod.coreness(N_REPEAT, edges)
    assert np.array_equal(np.concatenate([p["degree"] for p in parts]), deg)
    assert np.array_equal(np.concatenate([p["coreness"] for p in parts]), core)
    for mode, key in ((oracle_mod.KEY_REF32, "corea_ref32"), (oracle_mod.KEY_EXACT64, "corea_exact64")):
        oracle_mod.check_corea(np.concatenate([p[key] for p in parts]).view(np.float64), core, deg, mode)
    for p in parts:
        assert p["stats"]["n_edges_global"] == edges.shape[0]
        assert p["summary"][0] == int(core.max())


def need_gb(gb):
    import torch
    torch.cuda.empty_cache()
    if free_gb() < gb:
        pytest.skip(f"needs {gb} GB of free device memory, {free_gb():.0f} GB free")


@pytest.mark.parametrize("placement", ["emulated", "gpus"])
def test_one_rank_with_more_than_2p32_pairs(oracle_mod, monkeypatch, placement):
    """Reads split by read range over 2 ranks: all 2 250 family reads land on rank 0, whose own pairs exceed 2^32."""
    monkeypatch.delenv("KOMBGPU_PAIR_CHUNK", raising=False)
    devices = placement_devices(placement, 2)
    need_gb(RANGE_W2_GB)
    rk, ut, edges, mult, P = repeat_instance()
    parts = dist_build("hits", rk, ut, N_REPEAT, 2, devices)
    p_local = [p["stats"]["n_pairs_local"] for p in parts]
    assert p_local[0] >= 1 << 32 and sum(p_local) == P
    assert all(p["rounds"] == planned_rounds(p_local, 2, 0) for p in parts) and parts[0]["rounds"] > 1
    check_exact(oracle_mod, parts, edges, mult)


@pytest.mark.parametrize("placement", ["emulated", "gpus"])
def test_owner_receives_more_than_2p32_pairs(oracle_mod, monkeypatch, placement):
    """Whole reads dealt round-robin over 3 ranks: every rank emits fewer than 2^32 pairs (P = 9.0e9 in all), but the
    owner of the low unitig ids receives more than 2^32 of them."""
    monkeypatch.delenv("KOMBGPU_PAIR_CHUNK", raising=False)
    devices = placement_devices(placement, 3)
    need_gb(ROUNDROBIN_W3_GB)
    rk, ut, edges, mult, P = repeat_instance(reads_per_family=1500)
    parts = dist_build("hits", rk, ut, N_REPEAT, 3, devices, how="roundrobin")
    p_local = [p["stats"]["n_pairs_local"] for p in parts]
    assert all(p < 1 << 32 for p in p_local) and sum(p_local) == P
    assert max(p["stats"]["n_pairs_received"] for p in parts) >= 1 << 32
    assert sum(p["stats"]["n_pairs_received"] for p in parts) == P
    assert all(p["rounds"] == planned_rounds(p_local, 3, 0) for p in parts)
    check_exact(oracle_mod, parts, edges, mult)


# ---- failure in a late round ---------------------------------------------------------------------------------------

@pytest.mark.parametrize("world", [2, 3])
def test_failure_in_a_late_round_fails_every_rank(monkeypatch, world):
    """Rank 1's last pair names a unitig >= n: it fails in its last round; every rank returns KOMBGPU_EINVAL (nobody
    waits for ever), then the same communicator builds a graph equal to a fresh communicator's."""
    import torch
    import komb_b200
    from komb_b200.peer import DistGraph, run_local
    monkeypatch.setenv("KOMBGPU_PAIR_CHUNK", "3")
    u, v, n = pair_inputs()["rmat_small"]

    def share(comm, bad):
        a, b = split_pairs(u, v, comm.rank, world)
        a = a.copy()
        if bad and comm.rank == 1:
            a[-1] = n
        return torch.from_numpy(a.view(np.int32)).cuda(), torch.from_numpy(b.view(np.int32)).cuda()

    def body(comm):
        code = 0
        try:
            DistGraph.from_pairs(comm, *share(comm, True), n).close()
        except komb_b200.KombGpuError as e:
            code = e.code
        with DistGraph.from_pairs(comm, *share(comm, False), n) as g:
            return code, dist_snapshot(g)

    def fresh(comm):
        with DistGraph.from_pairs(comm, *share(comm, False), n) as g:
            return dist_snapshot(g)

    got = run_local(world, body)
    assert [c for c, _ in got] == [EINVAL] * world
    ref = run_local(world, fresh)
    assert ref[0]["rounds"] > 100
    for (_, p), q in zip(got, ref):
        for k in q:
            assert same(p[k], q[k]), k


# ---- komb2 -----------------------------------------------------------------------------------------------------------

def device_list():
    """Distinct GPUs when the box has them, else three ranks on device 0 (the library's emulation)."""
    return ",".join(str(d) for d in range(min(n_gpus(), 4))) if n_gpus() >= 2 else "0,0,0"


@pytest.mark.parametrize("name", komb2_case_names())
def test_komb2_multi_gpu_files_identical_with_rounds(tmp_path, oracle_mod, monkeypatch, name):
    monkeypatch.delenv("KOMBGPU_PAIR_CHUNK", raising=False)
    sam1, sam2, _ = load_komb2_case(name)
    env = {"KOMB_GPU_DEVICES": device_list()}
    ref = run_komb2_files(oracle_mod, sam1, sam2, tmp_path / "ref", env)
    got = run_komb2_files(oracle_mod, sam1, sam2, tmp_path / "rounds", {**env, "KOMBGPU_PAIR_CHUNK": "3"})
    assert got == ref


def test_komb2_multi_gpu_more_than_2p32_pairs(tmp_path, oracle_mod, monkeypatch):
    monkeypatch.delenv("KOMBGPU_PAIR_CHUNK", raising=False)
    need_gb(ROUNDROBIN_W3_GB)
    m1, m2 = synth.repeat_family_hits()
    edges, _, P = weighted_cliques(*both_mates(m1, m2))
    assert P > 1 << 32
    got, _ = oracle_mod.run_komb2(KOMB2, synth.render_sam(m1, N_REPEAT, 1), synth.render_sam(m2, N_REPEAT, 2), tmp_path,
                                  extra_env={"KOMB_GPU_DEVICES": device_list()})
    hit = np.zeros(N_REPEAT, bool)
    hit[m1.unitig] = True
    hit[m2.unitig] = True
    deg, core = oracle_mod.coreness(N_REPEAT, edges)
    ids = np.flatnonzero(hit)                          # komb2's vertices: the unitigs that occur in the SAM files
    assert got["kcore"] == {str(i): (int(core[i]), int(deg[i])) for i in ids.tolist()}
    eu, ev = oracle_mod.unpack_edges(edges)
    assert got["edges"] == {tuple(sorted((str(a), str(b)))) for a, b in zip(eu.tolist(), ev.tolist())}
    score = oracle_mod.corea(core[ids], deg[ids], oracle_mod.KEY_REF32)
    for i, s in zip(ids.tolist(), score.tolist()):     # the reference prints "%f"
        assert abs(got["score"][str(i)] - s) <= 5.0e-7 + 1e-12
