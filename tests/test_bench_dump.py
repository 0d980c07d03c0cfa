"""bench.py --dump-outputs on the CPU: file names, dtype, the sample cap, sample positions fixed from call to call, and
the 64 MB bound on a cfg2-sized result."""
import numpy as np

import bench

NAMES = {"counts", "vertex_index", "edge_index", "degree", "coreness", "score", "edges_u", "edges_v"}


def _results(n, E, seed):
    rng = np.random.default_rng(seed)
    return {"u": np.sort(rng.integers(0, n, E)).astype(np.uint32), "v": rng.integers(0, n, E).astype(np.uint32),
            "degree": rng.integers(0, 1000, n).astype(np.int32), "coreness": rng.integers(0, 40, n).astype(np.int32),
            "score": rng.random(n)}


def _load(d):
    return {p.stem: np.load(p) for p in d.glob("*.npy")}


def test_dump_outputs_cfg2_size(tmp_path):
    n, E = 1_000_000, 3 * bench.DUMP_SAMPLE + 7           # vertex arrays whole, the edge list sampled
    r = _results(n, E, 0)
    bench.dump_outputs(str(tmp_path / "a"), r)
    bench.dump_outputs(str(tmp_path / "b"), _results(n, E, 1))
    a, b = _load(tmp_path / "a"), _load(tmp_path / "b")
    assert set(a) == NAMES
    assert all(x.dtype == np.float64 for x in a.values())
    assert a["counts"].tolist() == [n, E]
    assert np.array_equal(a["vertex_index"], np.arange(n))
    ei = a["edge_index"].astype(np.int64)
    assert ei.shape[0] == bench.DUMP_SAMPLE and np.all(np.diff(ei) > 0) and ei[-1] < E
    assert np.array_equal(a["edge_index"], b["edge_index"])          # same positions whatever the values
    assert np.array_equal(a["edges_u"], r["u"][ei]) and np.array_equal(a["edges_v"], r["v"][ei])
    assert np.array_equal(a["degree"], r["degree"]) and np.array_equal(a["coreness"], r["coreness"])
    assert np.array_equal(a["score"], r["score"])
    assert sum(p.stat().st_size for p in (tmp_path / "a").glob("*.npy")) < 64 << 20


def test_dump_outputs_samples_vertices_too(tmp_path):
    n, E = bench.DUMP_SAMPLE + 100, 50
    r = _results(n, E, 2)
    bench.dump_outputs(str(tmp_path), r)
    a = _load(tmp_path)
    vi = a["vertex_index"].astype(np.int64)
    assert vi.shape[0] == bench.DUMP_SAMPLE and np.all(np.diff(vi) > 0)
    assert np.array_equal(a["score"], r["score"][vi]) and np.array_equal(a["degree"], r["degree"][vi])
    assert np.array_equal(a["edge_index"], np.arange(E)) and np.array_equal(a["edges_v"], r["v"])
