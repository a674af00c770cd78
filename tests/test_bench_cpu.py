"""CPU-side tests of bench.py's host logic (no GPU): configuration presets, the per-box index cache, the SumEmbeddings
workload generator (its file images must be what the reference's constructors read — checked through the oracle) and
the line's bookkeeping helpers."""
import json
import sys

import numpy as np
import pytest


@pytest.fixture()
def bench(monkeypatch):
    monkeypatch.setattr(sys, "argv", ["bench.py"])
    import bench as b

    return b


def _args(bench, monkeypatch, *argv):
    monkeypatch.setattr(sys, "argv", ["bench.py"] + list(argv))
    return bench.parse_args()


def test_default_is_the_metrics_own_configuration(bench, monkeypatch):
    a = _args(bench, monkeypatch)
    assert (a.kind, a.n, a.dim, a.mode) == ("angular", 100_000_000, 128, "replicated")
    assert "configs[3]" in a.baseline_config and a.nq == 1024 and a.max_search == 200 and a.k == 10
    a = _args(bench, monkeypatch, "--config", "c3")
    assert (a.kind, a.n, a.dim) == ("angular_int", 10_000_000, 100)
    a = _args(bench, monkeypatch, "--config", "c5", "--elements", "2000000")
    assert (a.kind, a.n, a.dim, a.mode) == ("angular_int", 2_000_000, 96, "partitioned")
    a = _args(bench, monkeypatch, "--config", "c2", "--dim", "300", "--dist", "uniform")
    assert (a.n, a.dim, a.dist) == (1_000_000, 300, "uniform")
    cfg = bench.workload_config(a, "ours", a.n, 1, {"source": "built"})
    assert cfg["n"] == 1_000_000 and cfg["index_provenance"]["source"] == "built" and "shared" in cfg["index_provenance"]


def test_index_cache_round_trip(bench, monkeypatch, tmp_path):
    a = _args(bench, monkeypatch, "--config", "c2", "--cache", str(tmp_path / "cache"))
    path = bench.cache_path(a, a.n, 1234)
    assert path.endswith(".granne") and "1000000x128" in path and "seed1234" in path
    assert bench.cache_load(path) == (None, None)
    data = np.random.default_rng(0).integers(0, 255, size=3_000_000, dtype=np.uint8)
    bench.cache_store(path, data, {"built_by": "test", "build_s": 1.5})
    got, meta = bench.cache_load(path)
    assert np.array_equal(got, data) and meta["built_by"] == "test" and meta["bytes"] == data.size
    # a truncated or altered file is not trusted
    with open(path, "r+b") as f:
        f.write(b"\x00" * 64)
    assert bench.cache_load(path) == (None, None)
    a.cache = ""
    assert bench.cache_path(a, a.n, 1234) is None


def test_pack_le_and_sum_container_images(bench, monkeypatch, oracle):
    assert bench.pack_le([1, 0x01020304, 0x0A0B0C0D0E], 5).tolist() == [1, 0, 0, 0, 0, 4, 3, 2, 1, 0, 0x0E, 0x0D, 0x0C,
                                                                       0x0B, 0x0A]
    a = _args(bench, monkeypatch, "--config", "emb", "--elements", "6000")

    class Dev:
        index = 0

    c = bench.SumContainer(None, None, Dev(), a, a.n, 1234)
    el = c.to_oracle(oracle)                      # SumEmbeddings::from_bytes reads both images
    assert len(el) == 6000
    lens = np.diff(c.offsets.astype(np.int64))
    assert lens.min() == 2 and lens.max() == 9 and abs(c.terms_per_element - lens.mean()) < 1e-9
    for i in (0, 17, 5999):
        terms = c.terms[int(c.offsets[i]):int(c.offsets[i + 1])]
        v = c.raw_vectors(np.array([terms.size]), terms)[0]
        assert np.allclose(v / np.linalg.norm(v), el.get(i), atol=1e-5)
    q = c.queries(32, 4321)
    assert q.shape == (32, a.dim) and np.isfinite(q).all()
    assert np.array_equal(q, c.queries(32, 4321))  # seeded: both arms see the same queries


def test_dump_outputs_types_and_size_cap(bench, monkeypatch, tmp_path):
    a = _args(bench, monkeypatch, "--config", "c2", "--steps", "3", "--dump-outputs", str(tmp_path / "out"))
    assert a.steps == 3 and a.dump_outputs == str(tmp_path / "out")
    with pytest.raises(SystemExit):
        _args(bench, monkeypatch, "--steps", "0")
    rng = np.random.default_rng(1)
    ids = rng.integers(0, 1 << 32, size=(1000, 10), dtype=np.uint64).astype(np.uint32)
    ids[0, -1] = 0xFFFFFFFF
    dists = rng.random((1000, 10), dtype=np.float32)
    counts = np.full(1000, 10, dtype=np.int32)
    bench.dump_outputs(a.dump_outputs, {"ids": ids, "distances": dists, "counts": counts})
    got = {n: np.load(tmp_path / "out" / (n + ".npy")) for n in ("ids", "distances", "counts")}
    assert got["ids"].dtype == np.float64 and np.array_equal(got["ids"], ids.astype(np.float64))
    assert got["distances"].dtype == np.float32 and np.array_equal(got["distances"], dists)
    assert got["counts"].dtype == np.float64 and not (tmp_path / "out" / "rows.npy").exists()
    # above the cap: the same seeded sample of rows every time, row numbers alongside
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), {"ids": ids, "distances": dists}, limit=40_000)
    rows = np.load(tmp_path / "a" / "rows.npy").astype(np.int64)
    assert sum((tmp_path / "a" / f).stat().st_size - 128 for f in ("ids.npy", "distances.npy", "rows.npy")) <= 40_000
    assert np.array_equal(rows, np.load(tmp_path / "b" / "rows.npy")) and np.all(np.diff(rows) > 0)
    assert np.array_equal(np.load(tmp_path / "a" / "ids.npy"), ids[rows].astype(np.float64))


def test_numa_and_peak_helpers_do_not_raise(bench):
    assert isinstance(bench.spread_over_all_cores(), str)
    peak, src = bench.measured_peak_gbs()
    assert peak > 1000 and isinstance(src, str)
    json.dumps(bench.CONFIGS)
