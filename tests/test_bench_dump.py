"""bench.py --dump-outputs: the files hold the table the timed path built, exactly (64-bit words as 32-bit halves),
the node sample does not depend on the order a build keeps its nodes in, and all files stay under 64 MB."""
import json
import os
import subprocess
import sys
import types

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench():
    import bench
    return bench


class _Handle:
    """Stands in for PregraphGPU: the three calls dump_outputs makes."""

    def __init__(self, pkg, nodes, W, checksum, n_instances, n_reads):
        self.nodes, self.W, self.checksum = nodes, W, np.asarray(checksum, dtype=np.uint64)
        self.n_instances, self.n_reads = n_instances, n_reads

    def stats(self):
        return types.SimpleNamespace(device_key_words=self.W, n_instances=self.n_instances, n_nodes=len(self.nodes), n_reads=self.n_reads)

    def export_nodes(self, thrd_num):
        return self.nodes.copy()

    def table_checksum(self):
        return self.checksum


def _load(d):
    return {f[:-4]: np.load(os.path.join(d, f)) for f in sorted(os.listdir(d))}


def _size(d):
    return sum(os.path.getsize(os.path.join(d, f)) for f in os.listdir(d))


@pytest.mark.parametrize("W,n", [(1, 1_500_000), (4, 300_000), (2, 0)])
def test_dump_is_exact_order_free_and_bounded(pkg, tmp_path, W, n):
    bench = _bench()
    rng = np.random.default_rng(W)
    nodes = np.zeros(n, dtype=pkg.NODE_DTYPE)
    nodes["key"][:, 4 - W:] = rng.integers(0, 2 ** 63, size=(n, W), dtype=np.uint64) * np.uint64(2) + np.uint64(1)
    nodes["count"] = rng.integers(1, 300, size=n)
    nodes["l_links"] = rng.integers(0, 2 ** 32, size=n, dtype=np.uint64).astype(np.uint32)
    nodes["ordinal"] = np.arange(n, dtype=np.uint64) * np.uint64(4099)      # leads a sampled row back to its node
    checksum = [2 ** 64 - 1, 12345, 2 ** 40 + 3, n]
    shapes = bench.dump_outputs(pkg, _Handle(pkg, nodes, W, checksum, 10 ** 10 + 7, 99), str(tmp_path / "a"))
    shuffled = nodes[rng.permutation(n)]
    bench.dump_outputs(pkg, _Handle(pkg, shuffled, W, checksum, 10 ** 10 + 7, 99), str(tmp_path / "b"))
    a, b = _load(tmp_path / "a"), _load(tmp_path / "b")
    assert {k: list(v.shape) for k, v in a.items()} == shapes
    for k in a:
        assert a[k].dtype in (np.float32, np.float64) and np.array_equal(a[k], b[k]), k
    assert _size(tmp_path / "a") <= 64_000_000
    assert a["stats"].tolist() == [10 ** 10 + 7, n, 99]
    assert [(int(h) << 32) | int(lo) for h, lo in a["table_checksum"]] == checksum
    m = len(a["nodes_count"])
    assert m == n if n * 8 * (2 * W + 4) < 50_000_000 else n // 2 < m < n
    # every sampled row is a distinct node of the table with its fields intact, and the rows are sorted by key
    key = a["nodes_key"].astype(np.uint64)
    words = np.stack([(key[:, 2 * q] << np.uint64(32)) | key[:, 2 * q + 1] for q in range(W)], axis=1) if m else None
    src = nodes[(a["nodes_ordinal"] / 4099).astype(np.int64)]
    assert len(np.unique(src["ordinal"])) == m
    if m:
        assert np.array_equal(words, src["key"][:, 4 - W:])
        assert np.array_equal(a["nodes_count"], src["count"]) and np.array_equal(a["nodes_l_links"], src["l_links"])
        assert np.array_equal(np.lexsort(tuple(words[:, q] for q in range(W - 1, -1, -1))), np.arange(m))


@pytest.mark.gpu
def test_bench_dump_matches_oracle(pkg, oracle, tmp_path):
    """A tiny C2-shaped run of bench.py: the dumped stats, fingerprint and node sample equal the oracle's table for the
    same seeded reads, and a second run writes the same files."""
    args = ["--pairs", "20000", "--transcripts", "200", "--steps", "2", "--warmup", "1", "--no-e2e", "--no-cpu-baseline"]
    for tag in ("a", "b"):
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args, "--dump-outputs", str(tmp_path / tag)],
                           capture_output=True, text=True, timeout=900)
        assert r.returncode == 0, r.stderr[-3000:]
        line = json.loads(r.stdout.strip().splitlines()[-1])
        assert line["steps"] == 2
    a, b = _load(tmp_path / "a"), _load(tmp_path / "b")
    for k in a:
        assert np.array_equal(a[k], b[k]), k

    cfg = dict(pkg.synth.CONFIGS["C2"], n_pairs=20000, n_transcripts=200)
    K, kw, L = cfg["K"], cfg["key_words"], cfg["read_len"]
    tr = pkg.synth.make_transcriptome(cfg["n_transcripts"], cfg["seed"], hot=cfg["hot"])
    reads, lens = pkg.synth.make_reads(tr, cfg["n_pairs"], L, cfg["seed"])
    ref = oracle.run_hashing(reads, lens, K, kw, 8, 0)
    W = 1
    nodes = np.zeros(ref.nodes, dtype=pkg.NODE_DTYPE)
    nodes["key"], nodes["count"], nodes["l_links"] = ref.records["key"], ref.records["count"], ref.records["l_links"]
    nodes["rword"], nodes["ordinal"] = ref.records["rword"], ref.first_ordinals
    h = _Handle(pkg, nodes, W, oracle.table_checksum(ref.records, W), ref.instances, len(reads))
    _bench().dump_outputs(pkg, h, str(tmp_path / "oracle"))
    o = _load(tmp_path / "oracle")
    for k in ("stats", "table_checksum", "nodes_key", "nodes_count", "nodes_l_links", "nodes_ordinal"):
        assert np.array_equal(a[k], o[k]), k
    # link bits of rword; the flags above them are set by finalize, which the oracle has run and the bench has not
    assert np.array_equal(np.mod(a["nodes_rword"], 2 ** 24), np.mod(o["nodes_rword"], 2 ** 24))
