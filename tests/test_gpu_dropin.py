"""End-to-end drop-in parity on the GPU: the reference binary with its hashing stage replaced by
host/prlHashReads_gpu.c + libsdtgpu.so (oracle/_ref/SOAPdenovo-Trans-*-gpu) must write the same
`pregraph` outputs as the stock binary, byte for byte: .kmerFreq, .edge.gz (decompressed),
.preArc, .vertex, .preGraphBasic — i.e. the k-mer table was handed back in the layout
node2edge.c / cutTipPreGraph.c / prlRead2path.c consume, including the order-dependent pruning.

Both binaries are linked from the reference's own objects (oracle/Makefile, host/Makefile), so they exist only where
the SOAPdenovo-Trans sources were at hand.  Elsewhere every test runs the drop-in's hashing stage through the same
library calls host/prlHashReads_gpu.c makes (_hashing_stage) on the same files, and compares what it hands the
reference at that seam (the KmerSets in their exact (set, slot) layout, the .kmerFreq histogram, the counter lines)
with the oracle, which tests/test_oracle.py pins bit for bit to the unmodified reference."""
import ctypes as C
import gzip
import os
import subprocess

import numpy as np
import pytest

from conftest import make_dataset

pytestmark = pytest.mark.gpu


def _run(exe, cfg, prefix, K, p, d, extra=(), devices=None, sliced_hint=0, direct=False):
    cmd = [exe, "pregraph", "-s", cfg, "-K", str(K), "-p", str(p), "-d", str(d), "-o", prefix, *extra]
    env = dict(os.environ)
    if devices:
        env["SDTGPU_DEVICES"] = devices
    if sliced_hint:
        env["SDTGPU_CAPACITY_HINT"] = str(sliced_hint)
    if direct:
        env["SDTGPU_DIRECT"] = "1"
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=1800, env=env)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-2000:]
    return r.stdout


def _outputs(prefix):
    out = {}
    for ext in ("kmerFreq", "preArc", "vertex", "preGraphBasic"):
        with open(f"{prefix}.{ext}", "rb") as f:
            out[ext] = f.read()
    with gzip.open(f"{prefix}.edge.gz", "rb") as f:
        out["edge"] = f.read()
    return out


def _binaries(oracle, build):
    stock = os.path.join(oracle.REF_DIR, f"SOAPdenovo-Trans-{build}")
    gpu = os.path.join(oracle.REF_DIR, f"SOAPdenovo-Trans-{build}-gpu")
    return (stock, gpu) if os.path.exists(stock) and os.path.exists(gpu) else None


def _hashing_stage(pkg, cfg, K, key_words, p, d, n_kmer=False, devices=(0,), hint=0, direct=False, batch_reads=1 << 20):
    """prlRead2HashTable of host/prlHashReads_gpu.c, call for call: the library's parser (sdtpack) over the config's
    files, every batch pushed from host buffers to every handle (each keeps the k-mers it owns when there are several),
    sync, finalize per handle with counters and histogram summed, then the hand-back: sdtgpu_export_kmersets on one
    handle, the handles' nodes merged and replayed by sdtgpu_build_kmersets on several.
    Returns (records in (set, slot) order, set_info, kmerFreq[257], {nodes, instances, removed, linear})."""
    keys = dict(line.strip().split("=", 1) for line in open(cfg) if "=" in line)
    L = int(keys["max_rd_len"])
    fastq = "q1" in keys
    path1, path2 = (keys["q1"], keys["q2"]) if fastq else (keys["f1"], keys["f2"])
    n = len(devices)
    lib = pkg.library()
    gs = [pkg.PregraphGPU(K, key_words, L, capacity_hint=(hint // n + hint // (8 * n) + 1) if hint else 0, device=dev,
                          n_kmer=n_kmer, sliced=not direct) for dev in devices]
    try:
        if n > 1:
            for b, g in enumerate(gs):
                g.set_owner(b, n)
        rd = pkg.ReadPacker(path1, path2, fastq=fastq)
        pushed = 0
        while True:
            packed, lens, nmask = rd.next(L, batch_reads, n_kmer=n_kmer)
            if not len(lens):
                break
            for g in gs:
                g.push_reads(packed, lens, nmask, n_reads=len(lens), stride_bytes=packed.shape[1], first_read_ordinal=pushed)
            pushed += len(lens)
        rd.close()
        freq, counts = np.zeros(257, np.int64), dict(nodes=0, instances=0, removed=0, linear=0)
        for g in gs:
            g.sync()
            f, st = g.finalize(d)
            freq += f
            for k, v in (("nodes", st.n_nodes), ("instances", st.n_instances), ("removed", st.n_removed), ("linear", st.n_linear)):
                counts[k] += int(v)
        if n == 1:
            rec, info = gs[0].export_kmersets(p)
        else:
            nodes = np.ascontiguousarray(np.concatenate([g.export_nodes(p) for g in gs]))
            last = np.zeros(p, np.uint64)
            rc = lib.sdtgpu_last_ordinals(gs[0].h, p, last.ctypes.data)
            assert rc in (0, 5), rc
            sets = (C.POINTER(pkg.pregraph.KmerSet) * p)()
            assert lib.sdtgpu_build_kmersets(nodes.ctypes.data, len(nodes), key_words, p, None if rc else last.ctypes.data, sets) == 0
            rec, info = pkg.read_kmersets(sets, p, key_words)
            lib.sdtgpu_free_kmersets(sets, p)
    finally:
        for g in gs:
            g.close()
    return rec, info, freq, counts


def _check_hashing_stage(pkg, oracle, cfg, reads, lens, build, K, p, d, n_kmer=False, **kw):
    """The drop-in's hand-back equals the oracle's table for the same reads: what the stock binary's later stages
    would read from it, and the stage's own output (.kmerFreq, "nodes allocated", "kmer in reads", "kmer removed",
    "linear nodes")."""
    key_words = 1 if build == "31mer" else 4
    rec, info, freq, counts = _hashing_stage(pkg, cfg, K, key_words, p, d, n_kmer=n_kmer, **kw)
    ref = oracle.run_hashing(reads, lens, K, key_words, p, d, n_kmer=int(n_kmer))
    assert counts == dict(nodes=ref.nodes, instances=ref.instances, removed=ref.removed, linear=ref.linear)
    assert np.array_equal(freq, ref.kmerfreq)
    assert np.array_equal(info, ref.set_info)
    assert np.array_equal(rec, ref.records)
    return counts


@pytest.mark.parametrize("direct", [False, True], ids=["sliced", "direct"])
@pytest.mark.parametrize("build,K,p,d,fastq,extra", [
    ("31mer", 25, 8, 0, False, ()),
    ("31mer", 31, 3, 2, True, ()),
    ("127mer", 63, 8, 1, False, ()),
    ("127mer", 127, 4, 0, False, ()),
    ("31mer", 25, 8, 0, False, ("-n",)),
])
def test_pregraph_outputs_identical(pkg, oracle, tmp_path, build, K, p, d, fastq, extra, direct):
    """The drop-in's default is the sliced build without any capacity hint; SDTGPU_DIRECT=1 is the single-pass insert."""
    L = 150 if K > 63 else 100
    tr = pkg.synth.make_transcriptome(60, 21)
    reads, lens = make_dataset(pkg, tr, 12000, L, 33 + K, ragged=30, n_rate=0.003 if extra else 0)
    cfg = pkg.synth.write_library(str(tmp_path / "in"), reads, lens, L, paired=True, fastq=fastq)
    if _binaries(oracle, build) is None:
        _check_hashing_stage(pkg, oracle, cfg, reads, lens, build, K, p, d, n_kmer="-n" in extra, direct=direct)
        return
    stock, gpu = _binaries(oracle, build)
    a = _run(stock, cfg, str(tmp_path / "ref"), K, p, d, extra)
    b = _run(gpu, cfg, str(tmp_path / "gpu"), K, p, d, extra, direct=direct)
    assert "GPU pregraph hashing" in b and "GPU pregraph hashing" not in a
    ra, rb = _outputs(str(tmp_path / "ref")), _outputs(str(tmp_path / "gpu"))
    for k in ra:
        assert ra[k] == rb[k], f"{k} differs ({len(ra[k])} vs {len(rb[k])} bytes)"
    assert len(ra["edge"]) > 1000 and len(ra["preArc"]) > 0
    # the reference's own conservation/consistency lines agree too
    for key in ("nodes allocated", "linear nodes", "kmer removed"):
        la = [l for l in a.splitlines() if key in l]
        lb = [l for l in b.splitlines() if key in l]
        assert la == lb, (la, lb)


@pytest.mark.parametrize("build,K,p,d", [("31mer", 31, 8, 1), ("127mer", 63, 5, 0)])
def test_pregraph_outputs_identical_sliced_build(pkg, oracle, tmp_path, build, K, p, d):
    """SDTGPU_CAPACITY_HINT: the sliced build with a hint (coarser chains); the hand-back and every pregraph
    output stay byte-identical."""
    tr = pkg.synth.make_transcriptome(60, 21)
    reads, lens = make_dataset(pkg, tr, 12000, 100, 5 + K, ragged=30)
    cfg = pkg.synth.write_library(str(tmp_path / "in"), reads, lens, 100, paired=True)
    if _binaries(oracle, build) is None:
        _check_hashing_stage(pkg, oracle, cfg, reads, lens, build, K, p, d, hint=4_000_000)
        return
    stock, gpu = _binaries(oracle, build)
    a = _run(stock, cfg, str(tmp_path / "ref"), K, p, d)
    b = _run(gpu, cfg, str(tmp_path / "gpu"), K, p, d, sliced_hint=4_000_000)
    ra, rb = _outputs(str(tmp_path / "ref")), _outputs(str(tmp_path / "gpu"))
    for k in ra:
        assert ra[k] == rb[k], f"{k} differs ({len(ra[k])} vs {len(rb[k])} bytes)"
    for key in ("nodes allocated", "linear nodes", "kmer removed"):
        pick = lambda t: [l for l in t.splitlines() if key in l and not l.startswith("time spent")]     # (wall-clock lines differ)
        assert pick(a) == pick(b)


@pytest.mark.parametrize("devices", ["0,0,0", "0,1"])
def test_pregraph_outputs_identical_sharded(pkg, oracle, tmp_path, devices):
    """SDTGPU_DEVICES: every table shard receives every batch and keeps the k-mers it owns; the
    shards' nodes are merged at hand-back.  "0,0,0" runs three shards on one GPU (always possible),
    "0,1" two GPUs.  Outputs must still equal the stock binary's byte for byte."""
    import torch
    if devices == "0,1" and torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    tr = pkg.synth.make_transcriptome(60, 21)
    reads, lens = make_dataset(pkg, tr, 12000, 100, 71, ragged=30)
    cfg = pkg.synth.write_library(str(tmp_path / "in"), reads, lens, 100, paired=True)
    if _binaries(oracle, "31mer") is None:
        _check_hashing_stage(pkg, oracle, cfg, reads, lens, "31mer", 27, 8, 1, devices=tuple(int(x) for x in devices.split(",")))
        return
    stock, gpu = _binaries(oracle, "31mer")
    a = _run(stock, cfg, str(tmp_path / "ref"), 27, 8, 1)
    b = _run(gpu, cfg, str(tmp_path / "gpu"), 27, 8, 1, devices=devices)
    assert f"on {len(devices.split(','))} device(s)" in b
    ra, rb = _outputs(str(tmp_path / "ref")), _outputs(str(tmp_path / "gpu"))
    for k in ra:
        assert ra[k] == rb[k], f"{k} differs"
    for key in ("nodes allocated", "linear nodes", "kmer removed"):
        pick = lambda t: [l for l in t.splitlines() if key in l and not l.startswith("time spent")]     # (wall-clock lines differ)
        assert pick(a) == pick(b)


def _compare(a, b, ra, rb):
    for k in ra:
        assert ra[k] == rb[k], f"{k} differs ({len(ra[k])} vs {len(rb[k])} bytes)"
    for key in ("nodes allocated", "linear nodes", "kmer removed", "kmer in reads"):
        pick = lambda t: [l for l in t.splitlines() if key in l and not l.startswith("time spent")]     # (wall-clock lines differ)
        assert pick(a) == pick(b)


def test_config_c1_as_stated(pkg, oracle, tmp_path):
    """BASELINE.json config 1 as stated: SOAPdenovo-Trans-31mer pregraph K=25 on 1 M synthetic 100 bp PE reads from 2 000
    random transcripts, -p 8 — the stock binary against the GPU drop-in (sliced build, no hint), all five outputs byte
    for byte, and the reference's counters (76 000 000 k-mers in reads)."""
    cfg_d = pkg.synth.CONFIGS["C1"]
    tr = pkg.synth.make_transcriptome(cfg_d["n_transcripts"], cfg_d["seed"])
    parts = [pkg.synth.make_reads(tr, 250_000, 100, cfg_d["seed"], first_pair=a)[0] for a in range(0, cfg_d["n_pairs"], 250_000)]
    reads = np.concatenate(parts)
    lens = np.full(len(reads), 100, np.uint32)
    cfg = pkg.synth.write_library(str(tmp_path / "in"), reads, lens, 100, paired=True)
    if _binaries(oracle, "31mer") is None:
        assert _check_hashing_stage(pkg, oracle, cfg, reads, lens, "31mer", 25, 8, 0)["instances"] == 76_000_000
        return
    stock, gpu = _binaries(oracle, "31mer")
    a = _run(stock, cfg, str(tmp_path / "ref"), 25, 8, 0)
    b = _run(gpu, cfg, str(tmp_path / "gpu"), 25, 8, 0)
    assert "76000000 kmer in reads" in a.replace(",", "") and "GPU pregraph hashing" in b
    _compare(a, b, _outputs(str(tmp_path / "ref")), _outputs(str(tmp_path / "gpu")))


def test_config_c5_flavour_d2_with_tip_pruning(pkg, oracle, tmp_path):
    """Config 5's shape through the drop-in: a few transcripts at 10^5 x depth (hot k-mers, slices that overflow by far
    and are cut into sub-slices), -d 2, and the order-dependent pruning after the hand-back."""
    tr = pkg.synth.make_transcriptome(200, 20261021, hot=3)
    reads, lens = make_dataset(pkg, tr, 150_000, 100, 77)
    cfg = pkg.synth.write_library(str(tmp_path / "in"), reads, lens, 100, paired=True)
    if _binaries(oracle, "31mer") is None:
        _check_hashing_stage(pkg, oracle, cfg, reads, lens, "31mer", 31, 8, 2)
        return
    stock, gpu = _binaries(oracle, "31mer")
    a = _run(stock, cfg, str(tmp_path / "ref"), 31, 8, 2)
    b = _run(gpu, cfg, str(tmp_path / "gpu"), 31, 8, 2)
    _compare(a, b, _outputs(str(tmp_path / "ref")), _outputs(str(tmp_path / "gpu")))
