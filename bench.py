#!/usr/bin/env python
"""bench.py — QPS of the granne search path on B200 (BASELINE.json metric), with roofline, e2e and CPU baseline.

Workload (config.workload).  The default is BASELINE.json configs[3], the configuration the metric is quoted on:
100M x 128-d angular f32, M=30, build max_search=200, search max_search=200, k=10, index replicated on every GPU,
1024 queries per GPU per step (it fits one GPU: 51 GB of vectors + 13 GB of adjacency rows).  `--config c2|c3|c5`
select the other BASELINE configurations (1M x 128 f32; 10M x 100 i8; range-partitioned i8 shards, one per GPU),
`--elements` overrides the element count.  Synthetic clustered vectors (SURVEY.md §8d) so that recall@10 >= 0.95 is
reachable; recall is measured against an exact brute force and reported.

Setup (outside the timed region): the vectors are generated ON THE GPU (seeded torch generators, element-wise
arithmetic only, so every rank and both arms produce the same bits), turned into elements by the library
(Vector::from per row) and handed over as a device-resident container; the index is built once per box by the GPU
GranneBuilder and its granne FILE IMAGE is cached under /dev/shm, so that every later run on the box — other N, and
the reference arm — loads the very same index bytes.

One step = one batch of 1024 queries per rank through Granne::search semantics (granne_b200_search_batch*).  Steps
are independent batches; they are issued round-robin on 8 CUDA streams (a serving system would do the same), then
the whole timed region is bracketed by barrier + synchronize and timed with CUDA events (max over ranks).
  value   device-resident: queries already in HBM, results left in HBM (+ the fused peer-store gather, N > 1)
  e2e     host buffers through the public API (granne_b200.Granne.search_batch -> granne_b200_search_batch): H2D of
          the queries and D2H of the results inside the timed region, issued from persistent host threads
Multi-GPU: replicated mode = every rank searches its own 1024 queries per step ("weak" scaling: per-GPU work fixed),
results gathered by peer stores; partitioned mode (`--config c5` / `--mode partitioned`) = one independent index per
rank, every rank searches ALL queries of the step on its shard, the tiles are all-gathered and merged by
(distance, global id) on the GPU inside the timed region.

`--impl reference` times the CPU restatement of the reference (oracle/, all host threads) on the same index image.
`--dump-outputs DIR` writes what the last timed step returned (ids, distances, counts) as .npy files.  Data and queries
are seeded and the index image comes from the --cache directory once built (the GPU builder's graph depends on thread
interleaving), so two builds of the project run against the same cache can be compared output for output.
"""
import argparse
import hashlib
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "QPS @ recall@10>=0.95, angular HNSW search (granne Granne::search), per-box aggregate"


def metric_name(a, n):
    """BASELINE.json's metric, named on the configuration this line was measured on (the same string in both arms)."""
    et = {"angular": "f32", "angular_int": "i8", "embeddings": "sum-of-embeddings f32"}[a.kind]
    size = "%dMx%d-d" % (n // 1_000_000, a.dim) if n % 1_000_000 == 0 else "%dx%d-d" % (n, a.dim)
    return "QPS @ recall@10>=0.95, %s angular %s (granne Granne::search), per-box aggregate" % (size, et)
UNIT = "queries/s"
GEN_VERSION = 2          # bump when the synthetic generator changes (part of the cache key)
CHUNK = 1 << 20          # rows per generation chunk (the generator is seeded per chunk)
DATA_SEED, QUERY_SEED = 1234, 4321

CONFIGS = {
    # name: (kind, n, dim, mode, BASELINE.json config it stands for)
    "c2": ("angular", 1_000_000, 128, "replicated", "BASELINE.json configs[1]"),
    "c3": ("angular_int", 10_000_000, 100, "replicated", "BASELINE.json configs[2]"),
    "c4": ("angular", 100_000_000, 128, "replicated", "BASELINE.json configs[3]"),
    "c5": ("angular_int", 12_500_000, 96, "partitioned", "BASELINE.json configs[4] family (1B/8 = 125M per shard "
                                                          "scaled to what builds in the time budget)"),
    "emb": ("embeddings", 1_000_000, 100, "replicated", "not a BASELINE config: granne's third element type, "
                                                         "SumEmbeddings — elements of 2..9 terms over n/5 embeddings"),
}


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=400)
    ap.add_argument("--warmup", type=int, default=8)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default=os.environ.get("GRANNE_B200_BENCH_CONFIG", "c4"), choices=sorted(CONFIGS))
    ap.add_argument("--elements", dest="n", type=int, default=0,
                    help="number of indexed elements (per shard in partitioned mode); 0 = the config's own "
                         "(not --n: torchrun would claim that prefix)")
    ap.add_argument("--dim", type=int, default=0)
    ap.add_argument("--kind", default="", choices=["", "angular", "angular_int", "embeddings"])
    ap.add_argument("--mode", default="", choices=["", "replicated", "partitioned"])
    ap.add_argument("--nq", type=int, default=1024, help="queries per step (per GPU in replicated mode)")
    ap.add_argument("--max-search", type=int, default=200)
    ap.add_argument("--k", type=int, default=10)
    ap.add_argument("--num-neighbors", type=int, default=30)
    ap.add_argument("--streams", type=int, default=8)
    ap.add_argument("--gather", default="p2p", choices=["p2p", "nccl"],
                    help="replicated, N > 1: p2p = kernels store result tiles into every peer's buffer (fused "
                         "epilogue over NVLink peer memory); nccl = one all-gather per step")
    ap.add_argument("--dist", default="clustered", choices=["clustered", "uniform"],
                    help="uniform = the reference's own test distribution U(-0.5, 0.5) (src/test_helper.rs:3-6)")
    ap.add_argument("--cpu-seconds", type=float, default=12.0, help="target duration of the cpu_baseline sample")
    ap.add_argument("--cache", default=os.environ.get("GRANNE_B200_BENCH_CACHE", "/dev/shm/granne_b200_bench_cache"),
                    help="directory for the index file image shared by all runs on this box ('' = no cache)")
    ap.add_argument("--no-fallback", action="store_true", help="fail instead of retrying with 10x fewer elements")
    ap.add_argument("--dump-outputs", default="", metavar="DIR",
                    help="write the results of the last timed step as DIR/<name>.npy (float32 / float64), so that "
                         "two builds can be compared output for output on the same seeded inputs")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be >= 1")
    kind, n, dim, mode, base = CONFIGS[a.config]
    a.kind = a.kind or kind
    a.n = a.n or n
    a.dim = a.dim or dim
    a.mode = a.mode or mode
    a.baseline_config = base
    return a


# ---- synthetic data ----------------------------------------------------------------------------------------------------
def mixture(n, dim, sub_dim=16, basis_seed=7):
    """Gaussian mixture on a random low-dimensional subspace (SURVEY.md §8d measurement distribution): the small
    basis / centre tables are made on the host, the points on the device."""
    n_centers = max(8, int(4096 * (n / 1e6) ** 0.5))
    brng = np.random.default_rng(basis_seed)
    basis = brng.standard_normal((sub_dim, dim)).astype(np.float32)
    centers = brng.standard_normal((n_centers, sub_dim)).astype(np.float32)
    return basis, centers


def clustered(n, dim, seed, n_centers, sub_dim=16, spread=0.3, basis_seed=7):
    """Host (numpy) version of the same mixture, for tests and tools that need host arrays (tests/test_fullsize_gpu.py,
    tools/prof_search.py); bench.py itself generates on the device."""
    brng = np.random.default_rng(basis_seed)
    basis = brng.standard_normal((sub_dim, dim)).astype(np.float32)
    centers = brng.standard_normal((n_centers, sub_dim)).astype(np.float32)
    rng = np.random.default_rng(seed)
    out = np.empty((n, dim), dtype=np.float32)
    step = 1 << 18
    for s in range(0, n, step):
        m = min(step, n - s)
        which = rng.integers(0, n_centers, size=m)
        pts = centers[which] + spread * rng.standard_normal((m, sub_dim)).astype(np.float32)
        out[s:s + m] = pts @ basis
    return out


def raw_chunk_device(torch, dev, a, tables, seed, chunk_index, rows, spread=0.3):
    """`rows` raw vectors of chunk `chunk_index` of stream `seed` as a CUDA float32 tensor.  Seeded per chunk, only
    element-wise arithmetic (no GEMM), so the same (seed, chunk) gives the same bits in every process on this GPU type."""
    g = torch.Generator(device=dev)
    g.manual_seed(seed * 1000003 + chunk_index)
    if a.dist == "uniform":
        return torch.rand((rows, a.dim), generator=g, device=dev, dtype=torch.float32) - 0.5
    basis, centers = tables
    which = torch.randint(0, centers.shape[0], (rows,), generator=g, device=dev)
    pts = centers[which] + spread * torch.randn((rows, centers.shape[1]), generator=g, device=dev, dtype=torch.float32)
    out = torch.zeros((rows, a.dim), device=dev, dtype=torch.float32)
    for k in range(basis.shape[0]):
        out.addcmul_(pts[:, k:k + 1], basis[k:k + 1])
    return out


def device_tables(torch, dev, a, n_total):
    if a.dist == "uniform":
        return None
    basis, centers = mixture(n_total, a.dim)
    return torch.from_numpy(basis).to(dev), torch.from_numpy(centers).to(dev)


def make_elements_device(torch, granne_b200, dev, a, n, seed, tables):
    """The element container [n, dim] (normalised f32 / i8) in HBM, generated chunk by chunk."""
    dt = torch.int8 if a.kind == "angular_int" else torch.float32
    el = torch.empty((n, a.dim), dtype=dt, device=dev)
    for ci, s in enumerate(range(0, n, CHUNK)):
        m = min(CHUNK, n - s)
        raw = raw_chunk_device(torch, dev, a, tables, seed, ci, m)
        granne_b200.elements_from_raw_device(a.kind, raw, out=el[s:s + m])
        del raw
    torch.cuda.synchronize(dev)
    return el


def make_queries_device(torch, dev, a, nq_total, seed, tables):
    out = torch.empty((nq_total, a.dim), dtype=torch.float32, device=dev)
    for ci, s in enumerate(range(0, nq_total, CHUNK)):
        m = min(CHUNK, nq_total - s)
        out[s:s + m] = raw_chunk_device(torch, dev, a, tables, seed, ci, m)
    return out


# ---- element containers ------------------------------------------------------------------------------------------------
class DenseContainer:
    """angular / angular_int: element rows resident in HBM (a CUDA tensor [n, dim])."""

    def __init__(self, torch, granne_b200, dev, a, n, seed, tables):
        self.torch, self.gb, self.a, self.n = torch, granne_b200, a, n
        self.rows = make_elements_device(torch, granne_b200, dev, a, n, seed, tables)
        self.terms_per_element = 0.0

    def open(self, index_bytes):
        return self.gb.Granne.from_device_elements(index_bytes, self.a.kind, self.rows)

    def builder(self):
        return self.gb.GranneBuilder.from_device_elements(self.a.kind, self.rows, num_neighbors=self.a.num_neighbors,
                                                          max_search=200)

    def ground_truth_block(self, s0, s1):
        blk = self.rows[s0:s1]
        return blk if self.a.kind == "angular" else self.torch.nn.functional.normalize(blk.float(), dim=1)

    def to_oracle(self, go):
        host = self.rows.cpu().numpy()
        return go.Elements.angular(host, as_is=True) if self.a.kind == "angular" else go.Elements.angular_int(host)

    def free(self):
        self.rows = None
        self.torch.cuda.empty_cache()


def pack_le(values, nbytes):
    """little-endian `nbytes`-byte integers, vectorised (odd_byte_int.rs:3-36)"""
    v = np.asarray(values, dtype=np.uint64)
    out = np.empty((v.size, nbytes), dtype=np.uint8)
    for b in range(nbytes):
        out[:, b] = (v >> np.uint64(8 * b)) & np.uint64(0xFF)
    return out.reshape(-1)


class SumContainer:
    """embeddings::SumEmbeddings: an embedding table + per-element term lists (file images, as the reference's own
    constructors take them: SumEmbeddings::from_bytes, src/elements/embeddings/mod.rs:56-61)."""

    def __init__(self, torch, granne_b200, dev, a, n, seed):
        self.torch, self.gb, self.a, self.n, self.dev = torch, granne_b200, a, n, dev
        n_emb = max(1000, n // 5)
        n_centers = max(8, int(4096 * (n_emb / 1e6) ** 0.5))
        rng = np.random.default_rng(seed)
        brng = np.random.default_rng(7)
        basis = brng.standard_normal((16, a.dim)).astype(np.float32)
        centers = brng.standard_normal((n_centers, 16)).astype(np.float32)
        which = rng.integers(0, n_centers, size=n_emb)
        emb = (centers[which] + 0.3 * rng.standard_normal((n_emb, 16)).astype(np.float32)) @ basis
        self.emb = emb.astype(np.float32)
        order = np.argsort(which, kind="stable")
        counts = np.bincount(which, minlength=n_centers)
        starts = np.concatenate([[0], np.cumsum(counts)[:-1]])
        self.groups = (order, starts, counts, np.nonzero(counts)[0])
        lens, terms = self.sample_elements(rng, n)
        self.offsets = np.concatenate([[0], np.cumsum(lens)]).astype(np.uint64)
        self.terms = terms
        self.terms_per_element = float(lens.mean())
        self.elements_image = np.concatenate([np.frombuffer(int(n).to_bytes(8, "little"), dtype=np.uint8),
                                              pack_le(self.offsets, 5), pack_le(terms, 3)])
        self.embeddings_image = np.concatenate([np.frombuffer(int(a.dim).to_bytes(8, "little"), dtype=np.uint8),
                                                self.emb.reshape(-1).view(np.uint8)])
        self._rows = None

    def sample_elements(self, rng, n):
        """elements of 2 + i % 8 terms (src/test_helper.rs:39-43) drawn from ONE cluster of embeddings each"""
        order, starts, counts, nonempty = self.groups
        c = nonempty[rng.integers(0, nonempty.size, size=n)]
        lens = 2 + (np.arange(n) % 8)
        pick = starts[c][:, None] + np.floor(rng.random((n, 9)) * counts[c][:, None]).astype(np.int64)
        mask = np.arange(9)[None, :] < lens[:, None]
        return lens, order[pick][mask].astype(np.uint32)

    def raw_vectors(self, lens, terms):
        """un-normalised sums of the term rows (what a caller of the reference passes as a query vector)"""
        owner = np.repeat(np.arange(lens.size), lens)
        out = np.zeros((lens.size, self.a.dim), dtype=np.float32)
        np.add.at(out, owner, self.emb[terms])
        return out

    def queries(self, nq_total, seed):
        lens, terms = self.sample_elements(np.random.default_rng(seed), nq_total)
        return self.raw_vectors(lens, terms)

    def open(self, index_bytes):
        return self.gb.Granne.from_bytes(index_bytes, "embeddings", self.elements_image, self.embeddings_image,
                                         device=self.dev.index)

    def builder(self):
        return self.gb.GranneBuilder("embeddings", self.elements_image, self.embeddings_image,
                                     num_neighbors=self.a.num_neighbors, max_search=200, device=self.dev.index)

    def ground_truth_block(self, s0, s1):
        torch = self.torch
        if self._rows is None:
            emb = torch.from_numpy(self.emb).to(self.dev)
            lens = np.diff(self.offsets.astype(np.int64))
            owner = torch.from_numpy(np.repeat(np.arange(self.n), lens)).to(self.dev)
            rows = torch.zeros((self.n, self.a.dim), dtype=torch.float32, device=self.dev)
            rows.index_add_(0, owner, emb[torch.from_numpy(self.terms.astype(np.int64)).to(self.dev)])
            self._rows = torch.nn.functional.normalize(rows, dim=1)
        return self._rows[s0:s1]

    def to_oracle(self, go):
        return go.Elements.from_bytes("embeddings", self.elements_image.tobytes(), self.embeddings_image.tobytes())

    def free(self):
        self._rows = None
        self.torch.cuda.empty_cache()


def make_container(torch, granne_b200, dev, a, n, seed, tables):
    if a.kind == "embeddings":
        return SumContainer(torch, granne_b200, dev, a, n, seed)
    return DenseContainer(torch, granne_b200, dev, a, n, seed, tables)


# ---- index cache -------------------------------------------------------------------------------------------------------
def cache_path(a, n, seed):
    if not a.cache:
        return None
    key = "%s_%dx%d_M%d_ef200_%s_seed%d_gen%d" % (a.kind, n, a.dim, a.num_neighbors, a.dist, seed, GEN_VERSION)
    return os.path.join(a.cache, key + ".granne")


def cache_load(path):
    if path and os.path.exists(path) and os.path.exists(path + ".json"):
        try:
            meta = json.load(open(path + ".json"))
            data = np.fromfile(path, dtype=np.uint8)
            if data.size == meta["bytes"] and hashlib.sha1(data[:1 << 20].tobytes()).hexdigest() == meta["head_sha1"]:
                return data, meta
        except Exception:
            pass
    return None, None


def cache_store(path, index_bytes, meta):
    if not path:
        return
    try:
        os.makedirs(os.path.dirname(path), exist_ok=True)
        tmp = "%s.tmp.%d" % (path, os.getpid())
        np.asarray(index_bytes).tofile(tmp)
        meta = dict(meta, bytes=int(np.asarray(index_bytes).size),
                    head_sha1=hashlib.sha1(np.asarray(index_bytes)[:1 << 20].tobytes()).hexdigest())
        json.dump(meta, open(tmp + ".json", "w"))
        os.replace(tmp + ".json", path + ".json")
        os.replace(tmp, path)
    except OSError as e:  # cache is an optimisation only
        print("bench: index cache not written (%r)" % (e,), file=sys.stderr)


def build_or_load_index(torch, granne_b200, a, dev, container, seed):
    """(index handle, index file image, provenance dict).  The image is what both arms search."""
    path = cache_path(a, container.n, seed)
    data, meta = cache_load(path)
    t0 = time.time()
    if data is not None:
        index = container.open(data)
        return index, data, {"source": "cache", "built_by": meta.get("built_by"), "build_s": meta.get("build_s"),
                             "load_s": time.time() - t0}
    b = container.builder()
    b.build()
    build_s = time.time() - t0
    index = b.get_index()
    t1 = time.time()
    data = b.index_bytes()
    write_s = time.time() - t1
    b.close()
    prov = {"source": "built", "built_by": "granne_b200 GPU GranneBuilder", "build_s": build_s,
            "write_index_s": write_s}
    cache_store(path, data, prov)
    return index, data, prov


DUMP_LIMIT = 64 << 20    # bytes written by --dump-outputs at most


def dump_outputs(directory, arrays, limit=DUMP_LIMIT):
    """Writes `arrays` (one row per query; ids as u32 bits or i64, distances, counts) as DIR/<name>.npy: float32 stays
    float32, every integer type becomes float64 (exact for ids below 2^53).  When they would exceed `limit` bytes, a
    fixed seeded sample of the rows is written instead, with the sampled row numbers as rows.npy."""
    out = {name: v if v.dtype == np.float32 else v.astype(np.float64) for name, v in arrays.items()}
    nrows = next(iter(out.values())).shape[0]
    total = sum(v.nbytes for v in out.values())
    if total > limit:
        keep = int(nrows * limit // (total + 8 * nrows))
        rows = np.sort(np.random.default_rng(0).choice(nrows, size=keep, replace=False))
        out = {name: v[rows] for name, v in out.items()}
        out["rows"] = rows.astype(np.float64)
    os.makedirs(directory, exist_ok=True)
    for name, v in out.items():
        np.save(os.path.join(directory, name + ".npy"), np.ascontiguousarray(v))


def workload_config(a, impl, n_used, world, prov=None):
    et = {"angular": "f32", "angular_int": "i8", "embeddings": "sum-of-embeddings f32"}[a.kind]
    shards = world if a.mode == "partitioned" else 1
    return {"workload": "%s%dx%d angular %s HNSW (M=%d, build max_search=200), search max_search=%d k=%d, "
                        "%d queries/step%s" % ("%d shards x " % shards if shards > 1 or a.mode == "partitioned" else "",
                                               n_used, a.dim, et, a.num_neighbors, a.max_search, a.k, a.nq,
                                               "/GPU" if a.mode == "replicated" else " (every shard searches all)"),
            "baseline_config": a.baseline_config, "requested_n": a.n, "n": n_used, "dim": a.dim,
            "max_search": a.max_search, "k": a.k, "queries_per_step_per_gpu": a.nq, "mode": a.mode,
            "distribution": a.dist,
            "index": ("replicated, queries sharded" if world > 1 else "single GPU") if a.mode == "replicated"
            else "range-partitioned: one independent index per GPU, merged by (distance, global id)",
            "index_provenance": dict(prov or {}, shared="both arms search the same granne index file image "
                                                         "(cached per box)"),
            "l2": "inputs larger than L2 (%.0f MB vectors + adjacency; query batches rotate)"
                  % (n_used * a.dim * (1 if a.kind == "angular_int" else 4) / 1e6), "streams": a.streams, "impl": impl}


class ClockSampler:
    """SM clock and throttle reasons sampled DURING the timed region (B200_PROFILING.md clocks line).  The timed
    region is a few milliseconds to a few hundred, so the samples come from NVML in-process (about every 0.5 ms) rather
    than from an nvidia-smi subprocess (100 ms period: it would miss the region)."""

    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}

    def __init__(self, torch, gpu_index):
        self.rows, self.bits, self.thread, self.h, self.nv = [], 0, None, None, None
        self.running = False
        try:
            import pynvml

            pynvml.nvmlInit()
            p = torch.cuda.get_device_properties(gpu_index)
            try:
                bus = "%08x:%02x:%02x.0" % (p.pci_domain_id, p.pci_bus_id, p.pci_device_id)
                self.h = pynvml.nvmlDeviceGetHandleByPciBusId(bus.encode())
            except Exception:
                self.h = pynvml.nvmlDeviceGetHandleByIndex(gpu_index)
            self.nv = pynvml
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
        except Exception:
            self.h = None

    def _loop(self):
        nv, h = self.nv, self.h
        reasons = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or getattr(
            nv, "nvmlDeviceGetCurrentClocksThrottleReasons")
        while self.running:
            try:
                self.rows.append(float(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)))
                self.bits |= int(reasons(h))
            except Exception:
                break
            time.sleep(0.0003)

    def sample_now(self):
        """one sample taken by the caller itself (while the GPU is draining the issued steps): a very short timed
        region can end before the sampler thread has been scheduled once"""
        if self.h is None:
            return
        try:
            nv = self.nv
            reasons = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or getattr(
                nv, "nvmlDeviceGetCurrentClocksThrottleReasons")
            self.rows.append(float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)))
            self.bits |= int(reasons(self.h))
        except Exception:
            pass

    def start(self):
        if self.h is None:
            return
        self.old_interval = sys.getswitchinterval()
        sys.setswitchinterval(0.0002)  # let the sampler run between the launches the main thread issues
        self.running = True
        self.thread = threading.Thread(target=self._loop, daemon=True)
        self.thread.start()

    def stop(self):
        if self.h is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "samples": 0, "reasons": ["nvml unavailable"]}
        self.running = False
        self.thread.join()
        sys.setswitchinterval(self.old_interval)
        return {"sm_mhz": float(np.median(self.rows)) if self.rows else None, "sm_max_mhz": self.max_mhz,
                "samples": len(self.rows), "source": "nvml, sampled inside the timed region",
                "reasons": sorted(name for bit, name in self.REASONS.items() if self.bits & bit)}


def measured_peak_gbs():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def pin_to_gpu_numa(local):
    """Pins this process (and the threads it starts) to the CPUs of the GPU's NUMA node: the e2e path is host-issue
    bound at 8 ranks x 8 threads, and cross-socket pinned buffers cost latency on every copy."""
    try:
        bus = subprocess.run(["nvidia-smi", "-i", str(local), "--query-gpu=pci.bus_id", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=20).stdout.strip().lower()
        if bus.startswith("00000000:"):
            bus = bus[4:]
        cpus = open("/sys/bus/pci/devices/%s/local_cpulist" % bus).read().strip()
        ids = set()
        for part in cpus.split(","):
            lo, _, hi = part.partition("-")
            ids.update(range(int(lo), int(hi or lo) + 1))
        if ids:
            os.sched_setaffinity(0, ids)
            return cpus
    except Exception:
        pass
    return None


def spread_over_all_cores():
    """The CPU arms get the whole host: every logical CPU, and memory interleaved over all NUMA nodes (a search thread
    gathers random rows of a 51 GB array: with first-touch placement half of the threads would read remote memory)."""
    ncpu = os.cpu_count() or 1
    try:
        os.sched_setaffinity(0, range(ncpu))
    except OSError:
        pass
    try:
        import ctypes

        nodes = len([d for d in os.listdir("/sys/devices/system/node") if d.startswith("node") and d[4:].isdigit()])
        if nodes > 1:
            mask = ctypes.c_ulong((1 << nodes) - 1)
            libc = ctypes.CDLL(None, use_errno=True)
            libc.syscall(238, 3, ctypes.byref(mask), 65)  # set_mempolicy(MPOL_INTERLEAVE, all nodes)
            return "interleaved over %d NUMA nodes" % nodes
    except Exception:
        pass
    return "default placement"


# ---- CPU side (the oracle: test infrastructure, used here only as the timed CPU baseline / reference arm) -------------
def oracle_index(a, index_bytes, container):
    from oracle import granne_oracle as go

    el = container.to_oracle(go)
    g = go.Granne.from_bytes(np.asarray(index_bytes), el)   # compressed adjacency decoded per expansion (faithful)
    return go, el, g


def cpu_baseline(a, index_bytes, container, queries, seconds):
    """The CPU restatement of the reference (oracle/) on this box's host cores, bounded sample."""
    threads = os.cpu_count() or 1
    placement = spread_over_all_cores()
    go, el, g = oracle_index(a, index_bytes, container)
    container.free()
    gf = g.to_fixed()                                  # pre-decoded adjacency (the stronger CPU variant)
    probe = queries[:max(threads * 2, 64)]
    t = time.time()
    gf.search_batch(probe, a.max_search, a.k, threads=threads)
    rate = probe.shape[0] / max(time.time() - t, 1e-6)
    nsample = int(min(queries.shape[0], max(probe.shape[0], rate * seconds / 2)))
    sample = queries[:nsample]
    out = {}
    for name, idx in (("compressed_adjacency", g), ("decoded_adjacency", gf)):
        t = time.time()
        idx.search_batch(sample, a.max_search, a.k, threads=threads)
        out[name] = nsample / max(time.time() - t, 1e-9)
    best = max(out.values())
    return {"value": best, "unit": UNIT, "cores": threads,
            "kind": "port (C++ restatement of the Rust reference; not pinned against a run of the Rust binary: no "
                    "rustc in the image)",
            "sample": "%d queries of the bench workload on the SAME index image, %d threads, one query per task in "
                      "static chunks, memory %s; best of compressed (%.0f QPS) and pre-decoded (%.0f QPS) adjacency" %
                      (nsample, threads, placement, out["compressed_adjacency"], out["decoded_adjacency"])}


def run_reference(a):
    """Reference arm: the oracle's CPU search (all host threads) on the same configuration AND the same index image
    as the ours arm (taken from the box cache; built by the GPU builder as a setup step when the cache is cold — the
    timed path is the CPU search only).  Rank 0 only."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import torch

    import granne_b200
    from granne_b200 import build as gb_build

    if not torch.cuda.is_available():
        raise SystemExit("bench.py --impl reference generates the shared synthetic data on the GPU")
    gb_build.build()
    granne_b200.load_library()
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    threads = os.cpu_count() or 1
    placement = spread_over_all_cores()
    world = a.gpus if a.mode == "partitioned" else 1
    n = a.n
    while True:
        try:
            shards = []
            t_setup = time.time()
            for r in range(world):
                tables = device_tables(torch, dev, a, n)
                cont = make_container(torch, granne_b200, dev, a, n, DATA_SEED + r, tables)
                index, data, prov = build_or_load_index(torch, granne_b200, a, dev, cont, DATA_SEED + r)
                index.close()
                del index
                go, el, g = oracle_index(a, data, cont)
                if r == world - 1 and a.kind == "embeddings":
                    query_src = cont
                cont.free()
                shards.append((el, g, g.to_fixed(), prov))
            break
        except (RuntimeError, MemoryError, granne_b200.GranneError) as e:
            if a.no_fallback or n <= 1_000_000:
                raise
            print("bench: reference setup failed at n=%d (%r); retrying with %d" % (n, e, n // 10), file=sys.stderr)
            n //= 10
            torch.cuda.empty_cache()
    tables = device_tables(torch, dev, a, n)
    pool = 16
    if a.kind == "embeddings":
        queries = query_src.queries(max(a.nq * pool, 1 << 15), QUERY_SEED)
    else:
        queries = make_queries_device(torch, dev, a, max(a.nq * pool, 1 << 15), QUERY_SEED, tables).cpu().numpy()
    setup_s = time.time() - t_setup

    from granne_b200.distributed import merge_topk_host

    def search(qs):
        if len(shards) == 1:
            return shards[0][2].search_batch(qs, a.max_search, a.k, threads=threads)
        parts = [s[2].search_batch(qs, a.max_search, a.k, threads=threads) for s in shards]
        return merge_topk_host(np.stack([p[0] for p in parts]), np.stack([p[1] for p in parts]),
                               [r * n for r in range(len(shards))], a.k)

    probe = queries[:max(threads * 4, 256)]
    t = time.time()
    search(probe)
    rate = probe.shape[0] / max(time.time() - t, 1e-6)
    # the faithful variant (compressed adjacency decoded per expansion, as Granne::from_bytes serves it) on a bounded
    # sample, reported next to the pre-decoded one that the timed steps use (the stronger CPU baseline)
    compressed_qps = None
    if len(shards) == 1:
        sample = queries[:min(queries.shape[0], max(probe.shape[0], int(rate * 2)))]
        t = time.time()
        shards[0][1].search_batch(sample, a.max_search, a.k, threads=threads)
        compressed_qps = sample.shape[0] / max(time.time() - t, 1e-6)
    # a step must keep every host thread busy (>= 128 queries per thread) yet the whole run must stay bounded
    per_step_s = min(2.0, 90.0 / max(1, a.steps + a.warmup))
    per_step = int(max(min(16384, queries.shape[0]), min(queries.shape[0], rate * per_step_s)))
    per_step = min(per_step, queries.shape[0])
    for _ in range(min(a.warmup, 3)):
        search(queries[:per_step])
    t0 = time.time()
    for s in range(a.steps):
        off = (s * 4099) % (queries.shape[0] - per_step + 1)
        last = search(queries[off:off + per_step])
    dt = time.time() - t0
    if a.dump_outputs:
        dump_outputs(a.dump_outputs, dict(zip(("ids", "distances", "counts"), last)))
    qps = a.steps * per_step / dt
    prov = shards[0][3]
    line = {"metric": metric_name(a, n), "value": qps, "unit": UNIT, "n_gpus": a.gpus, "steps": a.steps, "warmup": a.warmup,
            "ms_per_step": dt / a.steps * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "i8" if a.kind == "angular_int" else "f32", "data": "synthetic", "impl": "reference",
            "config": workload_config(a, "reference", n, a.gpus, prov),
            "cpu_baseline": {"value": qps, "unit": UNIT, "cores": threads,
                             "kind": "port (C++ restatement of the Rust reference; not pinned against a run of the "
                                     "Rust binary: no rustc in the image)",
                             "sample": "%d queries per step (bounded; >= %d per host thread), pre-decoded adjacency, "
                                       "%d threads (nproc %d), memory %s, same index image as the ours arm (%s); "
                                       "setup %.0f s (index build by the GPU builder: %s s); compressed-adjacency "
                                       "variant on a bounded sample: %s QPS"
                                       % (per_step, per_step // threads, threads, threads, placement,
                                          prov.get("source"), setup_s,
                                          "%.0f" % prov["build_s"] if prov.get("build_s") else "n/a",
                                          "%.0f" % compressed_qps if compressed_qps else "n/a")},
            "e2e": {"value": qps, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


# ---- the GPU arm -------------------------------------------------------------------------------------------------------
def main():
    a = parse_args()
    if a.impl == "reference":
        run_reference(a)
        return
    import torch
    import torch.distributed as dist

    import granne_b200

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the granne_b200 search path has no CPU fallback")
    cpus = pin_to_gpu_numa(local)
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    from granne_b200 import build as gb_build

    if rank == 0:
        gb_build.build()
    if world > 1:
        dist.barrier()
    granne_b200.load_library()
    partitioned = a.mode == "partitioned"

    # ---- multi-GPU parity gate: the 2-GPU assertions of tests/multi_gpu_check.py (small oracle-built fixtures, both
    # modes + the fused gather, bit-compared with the CPU oracle) run before anything is timed
    parity_checked = None
    if world > 1:
        sys.path.insert(0, os.path.join(ROOT, "tests"))
        import multi_gpu_check

        multi_gpu_check.check(rank, world, local, dev)
        parity_checked = True

    # ---- synthetic data, elements, index ---------------------------------------------------------------------------
    n = a.n
    t_all = time.time()
    while True:
        try:
            seed = DATA_SEED + (rank if partitioned else 0)
            t0 = time.time()
            tables = device_tables(torch, dev, a, n)
            cont = make_container(torch, granne_b200, dev, a, n, seed, tables)
            t_data = time.time() - t0
            t0 = time.time()
            path = cache_path(a, n, seed)
            if partitioned or rank == 0 or (path and os.path.exists(path)):
                index, index_bytes, prov = build_or_load_index(torch, granne_b200, a, dev, cont, seed)
                ok = 1
            else:
                index, index_bytes, prov, ok = None, None, None, 1
            if world > 1:
                dist.barrier()          # rank 0 has built and published the image
                if index is None:
                    data, meta = cache_load(path)
                    if data is None:  # no shared cache directory: fall back to a broadcast of the image
                        ok = 0
                    else:
                        index = cont.open(data)
                        index_bytes, prov = data, {"source": "cache", "built_by": meta.get("built_by"),
                                                   "build_s": meta.get("build_s")}
                flag = torch.tensor([ok], device=dev)
                dist.all_reduce(flag, op=dist.ReduceOp.MIN)
                if int(flag.item()) == 0 and not partitioned:
                    size = torch.tensor([len(index_bytes) if rank == 0 else 0], dtype=torch.int64, device=dev)
                    dist.broadcast(size, 0)
                    buf = torch.empty(int(size.item()), dtype=torch.uint8, device=dev)
                    if rank == 0:
                        buf.copy_(torch.from_numpy(np.asarray(index_bytes)))
                    dist.broadcast(buf, 0)
                    if index is None:
                        index_bytes = buf.cpu().numpy()
                        index = cont.open(index_bytes)
                        prov = {"source": "broadcast from rank 0"}
                    del buf
            t_build = time.time() - t0
            break
        except (RuntimeError, MemoryError, granne_b200.GranneError) as e:
            if a.no_fallback or n <= 1_000_000 or world > 1:
                raise
            print("bench: setup failed at n=%d (%r); retrying with %d elements" % (n, e, n // 10), file=sys.stderr)
            n //= 10
            cont = index = None
            torch.cuda.empty_cache()

    # ---- queries: a rotating pool of distinct batches per rank --------------------------------------------------------
    pool = 16
    qseed = QUERY_SEED + (0 if partitioned else rank)      # partitioned: every rank searches the same queries
    if a.kind == "embeddings":
        q_host = cont.queries(a.nq * pool, qseed)
        q_dev = torch.from_numpy(q_host).to(dev)
    else:
        q_dev = make_queries_device(torch, dev, a, a.nq * pool, qseed, tables)
        q_host = q_dev.cpu().numpy()
    streams = [torch.cuda.Stream(device=dev) for _ in range(max(1, a.streams))]
    # per stream: one int32 buffer [2, nq, k] = ids | distance bits (a single all-gather collects both), + counts
    bufs = [torch.empty((2, a.nq, a.k), dtype=torch.int32, device=dev) for _ in streams]
    outs = [(b[0], b[1].view(torch.float32), torch.empty((a.nq,), dtype=torch.int32, device=dev)) for b in bufs]
    gathered, groups, fused = None, None, None
    if world > 1 and a.gather == "p2p" and not partitioned:
        try:
            from granne_b200.distributed import FusedGather

            fused = FusedGather(a.nq, a.k, slots=len(streams))
        except Exception as e:  # symmetric memory unavailable: use the NCCL all-gather
            fused = None
            if rank == 0:
                print("fused peer gather unavailable (%r): falling back to NCCL all-gather" % (e,), file=sys.stderr)
        ok = torch.tensor([1 if fused is not None else 0], device=dev)
        dist.all_reduce(ok, op=dist.ReduceOp.MIN)
        if int(ok.item()) == 0:
            fused = None
    if world > 1 and fused is None:
        gathered = [torch.empty((world * 2 * a.nq, a.k), dtype=torch.int32, device=dev) for _ in streams]
        # one communicator per stream: collectives of different in-flight steps do not serialise behind each other
        groups = [dist.new_group(backend="nccl") for _ in streams]
    merged = None
    if partitioned:
        from granne_b200.api import merge_topk_device

        bases = [r * n for r in range(world)]
        merged = [(torch.empty((a.nq, a.k), dtype=torch.int64, device=dev),
                   torch.empty((a.nq, a.k), dtype=torch.float32, device=dev)) for _ in streams]

    qin = [torch.empty((a.nq, a.dim), dtype=torch.float32, device=dev) for _ in streams]
    seq = [0]

    def step_body(slot):
        if fused is not None:  # result tiles go straight into every peer's gathered buffer
            seq[0] += 1
            index.search_batch_device_gather(qin[slot], fused.spec(slot, seq[0]), a.max_search, a.k,
                                             stream=streams[slot].cuda_stream)
            return
        index.search_batch_device(qin[slot], a.max_search, a.k, out=outs[slot], stream=streams[slot].cuda_stream)
        if world > 1:  # collect every rank's result tile (NCCL all-gather over NVLink)
            dist.all_gather_into_tensor(gathered[slot], bufs[slot].view(2 * a.nq, a.k), group=groups[slot])
        if partitioned:  # k-way merge of the per-shard tiles by (distance, global id) on this rank's GPU
            if world > 1:
                g = gathered[slot].view(world, 2, a.nq, a.k)
                part_ids, part_d = g[:, 0].contiguous(), g[:, 1].contiguous().view(torch.float32)
            else:
                part_ids, part_d = bufs[slot][0][None], bufs[slot][1][None].view(torch.float32)
            merge_topk_device(local, part_ids, part_d, bases, out_ids=merged[slot][0], out_dists=merged[slot][1],
                              stream=streams[slot].cuda_stream)

    def device_step(s):
        slot = s % len(streams)
        st = streams[slot]
        with torch.cuda.stream(st):
            qin[slot].copy_(q_dev[(s % pool) * a.nq:(s % pool + 1) * a.nq], non_blocking=True)
            step_body(slot)

    def sync_all():
        for st in streams:
            st.synchronize()
        torch.cuda.synchronize(dev)

    # recall + algorithmic bytes per query (counters are parity-checked against the oracle in tests/)
    stats = torch.zeros((a.nq, 4), dtype=torch.int64, device=dev)
    ids0, _, _ = index.search_batch_device(q_dev[:a.nq], a.max_search, a.k, stats=stats)
    torch.cuda.synchronize(dev)
    index.stream_status()
    st_np = stats.cpu().numpy()
    n_dist, n_expand, n_nbr = st_np[:, 0].mean(), st_np[:, 1].mean(), st_np[:, 2].mean()
    retried = float((st_np[:, 3] != 0).mean())
    esz = 1 if a.kind == "angular_int" else 4
    # SURVEY.md §8(d): vectors + adjacency + query; SumEmbeddings: t term rows + 3-byte ids + two 5-byte offsets per
    # distance (t = mean terms per element of the container)
    per_dist = a.dim * esz if a.kind != "embeddings" else cont.terms_per_element * (a.dim * 4 + 3) + 10
    bytes_per_query = n_dist * per_dist + n_nbr * 4 + a.dim * esz
    nsamp = min(256, a.nq)
    if a.kind != "angular_int":
        qn = torch.nn.functional.normalize(q_dev[:nsamp], dim=1)
    else:  # ground truth under the same i8 angular distance: cosine of the quantised vectors
        qq = q_dev[:nsamp]
        qq = torch.trunc(qq * 127.0 / qq.abs().amax(dim=1, keepdim=True))
        qn = torch.nn.functional.normalize(qq, dim=1)
    best = None
    for s0 in range(0, n, 1 << 20):  # exact brute force in slabs over the device-resident elements (off the hot path)
        blk = cont.ground_truth_block(s0, min(n, s0 + (1 << 20)))
        sc = qn @ blk.T
        v, i = torch.topk(sc, a.k, dim=1)
        i = i + s0
        if best is None:
            best = (v, i)
        else:
            vv = torch.cat([best[0], v], dim=1)
            ii = torch.cat([best[1], i], dim=1)
            tv, ti = torch.topk(vv, a.k, dim=1)
            best = (tv, torch.gather(ii, 1, ti))
        del blk, sc
    gt = best[1].cpu().numpy()
    got = ids0[:nsamp].cpu().numpy()
    recall = float(np.mean([len(set(gt[i].tolist()) & set(got[i].tolist())) / a.k for i in range(nsamp)]))
    # the container is only needed again by the CPU baseline (rank 0, N = 1), which copies it to the host
    want_cpu = world == 1 and rank == 0 and a.cpu_seconds > 0 and not partitioned
    if not want_cpu:
        cont.free()

    # ---- device-resident timed region ------------------------------------------------------------------------------------
    for s in range(max(a.warmup, len(streams))):
        device_step(s)
    sync_all()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize(dev)
    sampler = ClockSampler(torch, local)
    if rank == 0:
        sampler.start()
    launches0 = index.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.nvtx.range_push("timed")
    e0.record(torch.cuda.current_stream(dev))
    for st in streams:
        st.wait_stream(torch.cuda.current_stream(dev))
    t_issue = time.perf_counter()
    for s in range(a.steps):
        device_step(a.warmup + s)
    issue_ms = (time.perf_counter() - t_issue) * 1e3
    for st in streams:
        torch.cuda.current_stream(dev).wait_stream(st)
    e1.record(torch.cuda.current_stream(dev))
    if rank == 0:
        sampler.sample_now()  # everything is issued, the GPU is still inside the timed region
    sync_all()
    torch.cuda.nvtx.range_pop()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize(dev)
    ms = e0.elapsed_time(e1)
    launches = index.launch_count() - launches0 + (a.steps if partitioned else 0)
    clocks = sampler.stop() if rank == 0 else None
    index.stream_status()
    if world > 1:
        t = torch.tensor([ms], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    job_queries = a.steps * a.nq * (1 if partitioned else world)
    value = job_queries / (ms / 1e3)
    last = None
    if a.dump_outputs and rank == 0:  # copied now: the solo launches below reuse outs[0]
        slot = (a.warmup + a.steps - 1) % len(streams)
        if fused is not None:
            last = {"ids": fused.ids(slot), "distances": fused.dists(slot)}
        elif partitioned:
            last = {"ids": merged[slot][0], "distances": merged[slot][1]}
        elif world > 1:
            g = gathered[slot].view(world, 2, a.nq, a.k)
            last = {"ids": g[:, 0].reshape(-1, a.k), "distances": g[:, 1].reshape(-1, a.k).view(torch.float32)}
        else:
            last = {"ids": outs[slot][0], "distances": outs[slot][1], "counts": outs[slot][2]}
        last = {name: t.cpu().numpy() for name, t in last.items()}
        if last["ids"].dtype == np.int32:
            last["ids"] = last["ids"].view(np.uint32)

    # kernel-alone duration (single stream, one launch at a time) for the per-launch roofline
    solo = []
    for s in range(6):
        k0, k1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        qb = q_dev[(s % pool) * a.nq:(s % pool + 1) * a.nq]
        k0.record()
        index.search_batch_device(qb, a.max_search, a.k, out=outs[0])
        k1.record()
        torch.cuda.synchronize(dev)
        solo.append(k0.elapsed_time(k1))
    solo_ms = float(np.median(solo[1:]))

    # ---- end to end through the public host API ------------------------------------------------------------------------
    # persistent worker threads (started and parked on a barrier BEFORE t0), each issuing whole batches through
    # granne_b200_search_batch: memcpy into pinned staging, H2D, kernels, one packed D2H, memcpy out
    # client concurrency: 8..16 host threads, the count that splits the timed steps most evenly (20 steps -> 10
    # threads x 2 calls instead of 8 threads of which half make a third call while the others idle)
    nthreads = max(1, min(a.steps, min(range(8, 17), key=lambda t: (-(-a.steps // t) * t - a.steps, t))))
    h2d = a.nq * a.dim * 4
    d2h = a.nq * a.k * 8 + a.nq * 4 + 16

    class HostPool:
        def __init__(self):
            self.go = threading.Barrier(nthreads + 1)
            self.done = threading.Barrier(nthreads + 1)
            self.plan = None
            self.stop = False
            self.issue_s = [0.0] * nthreads
            self.threads = [threading.Thread(target=self.work, args=(t,), daemon=True) for t in range(nthreads)]
            [t.start() for t in self.threads]

        def work(self, t):
            while True:
                self.go.wait()
                if self.stop:
                    return
                count, offset = self.plan
                mine = count // nthreads + (1 if t < count % nthreads else 0)
                t0 = time.perf_counter()
                for s in range(mine):
                    b = (offset + s * nthreads + t) % pool
                    index.search_batch(q_host[b * a.nq:(b + 1) * a.nq], a.max_search, a.k)
                self.issue_s[t] = time.perf_counter() - t0
                self.done.wait()

        def run(self, count, offset):
            self.plan = (count, offset)
            self.go.wait()
            self.done.wait()

        def close(self):
            self.stop = True
            self.go.wait()

    if partitioned:
        # range-partitioned: the end-to-end path of one step is host queries -> every rank's GPU -> local search ->
        # all-gather -> merge -> merged (global id, distance) tiles back on the host.  Collectives are issued from
        # one thread per rank (NCCL), round-robin on the same streams, with pinned host buffers on both ends.
        nthreads = 1
        d2h = a.nq * a.k * 12
        q_pin = torch.from_numpy(q_host).pin_memory()
        res_pin = [(torch.empty((a.nq, a.k), dtype=torch.int64).pin_memory(),
                    torch.empty((a.nq, a.k), dtype=torch.float32).pin_memory()) for _ in streams]

        def host_step(s):
            slot = s % len(streams)
            with torch.cuda.stream(streams[slot]):
                b = s % pool
                qin[slot].copy_(q_pin[b * a.nq:(b + 1) * a.nq], non_blocking=True)
                step_body(slot)
                res_pin[slot][0].copy_(merged[slot][0], non_blocking=True)
                res_pin[slot][1].copy_(merged[slot][1], non_blocking=True)

        for s in range(max(a.warmup, len(streams))):
            host_step(s)
        sync_all()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)
        t0 = time.perf_counter()
        for s in range(a.steps):
            host_step(a.warmup + s)
        sync_all()
        e2e_s = time.perf_counter() - t0
        e2e_thread_ms = e2e_s * 1e3
        e2e_api = "granne_b200.distributed.PartitionedGranne path (search_batch_device + all_gather + merge_topk)"
    else:
        hp = HostPool()
        hp.run(max(a.warmup, 2 * nthreads), 0)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)
        t0 = time.perf_counter()
        hp.run(a.steps, 3)
        torch.cuda.synchronize(dev)
        e2e_s = time.perf_counter() - t0
        e2e_thread_ms = max(hp.issue_s) * 1e3
        hp.close()
        e2e_api = "granne_b200.Granne.search_batch (granne_b200_search_batch)"
    if world > 1:
        t = torch.tensor([e2e_s], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_s = float(t.item())
    e2e_qps = job_queries / e2e_s

    if rank != 0:
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()
        return

    peak, peak_src = measured_peak_gbs()
    total_bytes = bytes_per_query * a.nq * a.steps  # this rank's launches in the timed region
    achieved = total_bytes / (ms / 1e3) / 1e9
    traffic = None
    tp = os.path.join(ROOT, "profiles", "dram_traffic.json")
    if os.path.exists(tp):
        try:
            for tj in json.load(open(tp)).get("captures", []):
                if (tj.get("kind"), tj.get("n"), tj.get("dim"), tj.get("queries_per_launch")) == (a.kind, n, a.dim, a.nq):
                    traffic = tj.get("dram_bytes_per_launch")
        except Exception:
            traffic = None
    cpu = None
    if want_cpu:
        cpu = cpu_baseline(a, index_bytes, cont, q_host, a.cpu_seconds)
    kern = {"angular": "DistF32<%d>" % (a.dim // 32), "angular_int": "DistI8", "embeddings": "DistSum"}[a.kind]
    line = {
        "metric": metric_name(a, n), "value": value, "unit": UNIT, "n_gpus": world, "steps": a.steps, "warmup": a.warmup,
        "ms_per_step": ms / a.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "i8" if a.kind == "angular_int" else "f32", "data": "synthetic (generated on the GPU)",
        "config": workload_config(a, "ours", n, world, prov),
        "recall_at_10": recall,
        "e2e": {"value": e2e_qps, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "host_threads": nthreads, "host_issue_ms_per_step": e2e_thread_ms / max(1, a.steps / nthreads),
                "cpu_affinity": cpus, "api": e2e_api},
        "gpu_launches": int(launches),
        "clocks": clocks,
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                     "traffic": traffic, "traffic_source": "ncu dram__bytes_read+write per launch "
                                                           "(profiles/dram_traffic.json)" if traffic else None,
                     "peak_source": peak_src,
                     "kernel": "search_kernel<%s,7> (1 launch per step; retry + slow passes exit at once)" % kern,
                     "algorithmic_bytes_per_query": bytes_per_query,
                     "algorithmic_bytes_per_launch": bytes_per_query * a.nq,
                     "n_dist_per_query": n_dist, "n_expand_per_query": n_expand,
                     "queries_beyond_fast_pass": retried,
                     "solo_launch_ms": solo_ms,
                     "solo_launch_gbs": bytes_per_query * a.nq / (solo_ms / 1e3) / 1e9},
        "cpu_baseline": cpu,
        "parity_checked": parity_checked,
        "setup_s": {"data+elements": t_data, "index(build or load)": t_build, "total": time.time() - t_all},
        "host_issue_ms_per_step": issue_ms / a.steps,
        "multi_gpu_gather": None if world == 1 else ("nccl all_gather + merge_topk_kernel" if partitioned else (
            "p2p peer stores fused into the search kernels" if fused is not None else "nccl all_gather")),
    }
    if last is not None:
        dump_outputs(a.dump_outputs, last)
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
