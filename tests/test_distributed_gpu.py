"""The CUDA partition kernels (kombgpu_part_* / kombgpu_edgeset_*, dist.cu) through
komb_b200.distributed: world 1 in-process, and world 2 as two processes (gloo for the
host exchange, so it also runs on a single-GPU box: both ranks then share cuda:0 —
the per-rank kernels never wait on another rank, the host does the exchange)."""
import os
import pickle
import socket
import sys
from pathlib import Path

import numpy as np
import pytest
import torch.multiprocessing as mp

ROOT = Path(__file__).resolve().parents[1]
pytestmark = pytest.mark.gpu


def _inputs(case, rank, world):
    from komb_b200 import synth
    n, reads, seed, kind = case
    if kind == "hits":
        m1, m2 = synth.metagenome_hits(n, reads, seed=seed)
        lo, hi = reads * rank // world, reads * (rank + 1) // world
        s1 = (m1.read_key >= lo) & (m1.read_key < hi)
        s2 = (m2.read_key >= lo) & (m2.read_key < hi)
        return np.concatenate([m1.read_key[s1], m2.read_key[s2]]), np.concatenate([m1.unitig[s1], m2.unitig[s2]])
    u, v = synth.rmat_edges(18, reads, n_vertices=n, seed=seed)
    sl = slice(len(u) * rank // world, len(u) * (rank + 1) // world)
    return u[sl], v[sl]


def _expected(oracle, case):
    from komb_b200 import synth
    n, reads, seed, kind = case
    if kind == "hits":
        m1, m2 = synth.metagenome_hits(n, reads, seed=seed)
        edges, _, _ = oracle.build_edges(np.concatenate([m1.read_key, m2.read_key]), np.concatenate([m1.unitig, m2.unitig]))
    else:
        u, v = synth.rmat_edges(18, reads, n_vertices=n, seed=seed)
        edges = oracle.simplify(u, v)
    deg, core = oracle.coreness(n, edges)
    return edges, deg, core, oracle.corea(core, deg, oracle.KEY_REF32)


def _run_rank(rank, world, case, peel_mode="partitioned"):
    import torch
    import komb_b200
    from komb_b200.distributed import Comm, CudaEngine, analyse_partitioned
    dev = rank % torch.cuda.device_count()
    torch.cuda.set_device(dev)
    ctx = komb_b200.Context(dev)
    a, b = _inputs(case, rank, world)
    ta = torch.from_numpy(a.view(np.int32)).cuda()
    tb = torch.from_numpy(b.view(np.int32)).cuda()
    torch.cuda.synchronize()
    eng = CudaEngine(ctx)
    if case[3] == "hits":
        res = analyse_partitioned(eng, Comm(), case[0], read_key=ta, unitig=tb, peel_mode=peel_mode)
    else:
        res = analyse_partitioned(eng, Comm(), case[0], pairs=(ta, tb), peel_mode=peel_mode)
    out = {"v_lo": res.v_lo, "v_hi": res.v_hi, "deg": res.degree.cpu().numpy(), "core": res.coreness.cpu().numpy(),
           "score": res.score.cpu().numpy(), "max_core": res.max_coreness, "n_edges": res.n_edges, "stats": res.stats}
    ctx.close()
    return out


def _worker(rank, world, port, out_dir, case, peel_mode):
    sys.path.insert(0, str(ROOT))
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    out = _run_rank(rank, world, case, peel_mode)
    with open(Path(out_dir) / f"rank{rank}.pkl", "wb") as f:
        pickle.dump(out, f)
    dist.barrier()
    dist.destroy_process_group()


def _check(parts, exp):
    edges, deg, core, _ = exp
    assert np.array_equal(np.concatenate([p["deg"] for p in parts]), deg)
    assert np.array_equal(np.concatenate([p["core"] for p in parts]), core)
    from oracle import oracle
    oracle.check_corea(np.concatenate([p["score"] for p in parts]), core, deg, oracle.KEY_REF32)
    for p in parts:
        assert p["n_edges"] == edges.shape[0] and p["max_core"] == core.max()


@pytest.mark.parametrize("case", [(3000, 9000, 3, "hits"), (150000, 1500000, 7, "pairs")])
def test_partition_kernels_world1(oracle_mod, case):
    _check([_run_rank(0, 1, case)], _expected(oracle_mod, case))


@pytest.mark.parametrize("case,peel_mode", [((40000, 120000, 5, "hits"), "partitioned"), ((150000, 1500000, 7, "pairs"), "partitioned"),
                                            ((40000, 120000, 5, "hits"), "gather"), ((150000, 1500000, 7, "pairs"), "auto")])
def test_partition_kernels_world2(tmp_path, oracle_mod, case, peel_mode):
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    mp.spawn(_worker, args=(2, port, str(tmp_path), case, peel_mode), nprocs=2, join=True)
    parts = [pickle.load(open(tmp_path / f"rank{r}.pkl", "rb")) for r in range(2)]
    _check(parts, _expected(oracle_mod, case))
    if peel_mode == "partitioned":
        assert parts[0]["stats"]["exchange_subrounds"] > 0
    else:
        assert parts[0]["stats"]["peel_mode"] == "gather"


def test_part_build_rejects_misrouted_entries():
    """A directed entry whose source is not one of the rank's rows, or whose target is not a unitig of the graph, is an
    error (KOMBGPU_EINVAL), not a write past the rank's arrays."""
    import torch
    import komb_b200
    from komb_b200.distributed import CudaEngine
    ctx = komb_b200.Context(0)
    eng = CudaEngine(ctx)
    ok = torch.tensor([(10 << 32) | 3, (11 << 32) | 10, (19 << 32) | 0], dtype=torch.int64, device="cuda")
    part = eng.build_part(ok, 10, 20, 30)
    assert eng.part_counts(part) == {"n_local": 10, "n_directed": 3, "max_degree": 1}
    eng.lib.kombgpu_part_destroy(part)
    for bad in ((25 << 32) | 3, (9 << 32) | 3, (12 << 32) | 30):
        entries = torch.tensor([(10 << 32) | 3, bad], dtype=torch.int64, device="cuda")
        with pytest.raises(komb_b200.KombGpuError, match="outside this rank's rows"):
            eng.build_part(entries, 10, 20, 30)
    ctx.close()
