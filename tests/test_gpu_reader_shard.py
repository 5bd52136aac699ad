"""Shard readers (include/sdtgpu.h sdtgpu_reader_open_shard / _summary / _plan / _tell): W ranks read one library
together, each parsing only its own byte range.  Here the W ranks are W readers in one process on device 0 with their
summaries passed in Python (the two-GPU test at the end plans over torch.distributed and over the library's NCCL).

Every run checks the whole contract: each rank returns exactly the records the byte-range rule gives it (computed
here from a restatement of the host parser's record rule), in ordinal order, each batch a run of consecutive ordinals
starting at tell(); put in ordinal order, the batches equal sdtpack_next (one thread) byte for byte; every ordinal comes
back once."""
import os
import random
import sys

import numpy as np
import pytest

from conftest import make_dataset
from test_gpu_reader import CHAR_RULES, CHUNKS, FASTA_CASES, FASTQ_CASES, UNEQUAL_1, UNEQUAL_2, _table, host_all, write
from test_gpu_reader import c1_library  # noqa: F401  (module fixture: the C1-sized pair)

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
pytestmark = pytest.mark.gpu
EINVAL, ESTATE = 1, 5


# ---- the rule, restated from host/sdt_readpack.c (find_header / index_range)
def header_offsets(data: bytes, fastq: bool):
    size = len(data)

    def next_line(p):
        e = data.find(b"\n", p)
        return size if e < 0 else e + 1

    def find_header(p):
        while p < size:
            if not fastq and data[p] == ord(">"):
                return p
            if fastq and data[p] == ord("@"):
                plus = next_line(next_line(p))
                if plus >= size or data[plus] == ord("+"):
                    return p
            p = next_line(p)
        return size

    out, p = [], find_header(0)
    while p < size:
        out.append(p)
        p = next_line(next_line(p))     # header and sequence line
        p = next_line(next_line(p)) if fastq else find_header(p)
    return out


def lo(S, r, W):
    return r * S // W


def expected_ordinals(d1, d2, fastq, W):
    """Per rank, the ordinals it returns, in order."""
    h1, S1 = header_offsets(d1, fastq), len(d1)
    if d2 is None:
        return [[k for k, o in enumerate(h1) if lo(S1, r, W) <= o < lo(S1, r + 1, W)] for r in range(W)]
    h2, S2 = header_offsets(d2, fastq), len(d2)
    m = min(len(h1), len(h2))
    c1 = [sum(o < lo(S1, r, W) for o in h1) for r in range(W + 1)]
    hl, sl = (h1, S1) if len(h1) >= len(h2) else (h2, S2)
    res = []
    for r in range(W):
        o = [x for i in range(min(m, c1[r]), min(m, c1[r + 1])) for x in (2 * i, 2 * i + 1)]
        o += [m + j for j in range(m, len(hl)) if lo(sl, r, W) <= hl[j] < lo(sl, r + 1, W)]
        res.append(o)
    return res


def open_ranks(pkg, p1, p2, fastq, W, chunk):
    return [pkg.DeviceReadPacker(p1, p2, fastq=fastq, device=0, chunk_bytes=chunk, rank=r, world=W) for r in range(W)]


def read_rank(rd, L, batch, n_kmer, reverse, stride, pairs_end):
    """[(tell before the call, packed, lens, nmask)] until the rank has nothing left.  pairs_end = 2 min (n1, n2):
    the records of a batch below that ordinal are whole pairs (the drain of the longer file may end on an odd count,
    as it does for a plain reader)."""
    import torch
    out = []
    while True:
        o = rd.tell()
        packed, lens, nmask = rd.next(L, batch, n_kmer=n_kmer, reverse=reverse, stride_bytes=stride)
        n = len(lens)
        assert n <= batch and max(0, min(o + n, pairs_end) - o) % 2 == 0, (o, n, pairs_end)
        if n == 0:
            break
        torch.cuda.synchronize()
        out.append((o, packed.cpu().numpy(), lens.cpu().numpy().view(np.uint32), nmask.cpu().numpy() if n_kmer else None))
    end = rd.tell()
    if out:
        assert end == out[-1][0] + len(out[-1][2])
    return out


def check_shard(pkg, p1, p2, fastq, L, W, n_kmer=False, reverse=False, stride=None, batch=1000, chunk=0):
    stride = stride or pkg.synth.stride_bytes(L)
    hp, hl, hm = host_all(pkg, p1, p2, fastq, L, n_kmer, reverse, stride)
    d1 = open(p1, "rb").read()
    d2 = open(p2, "rb").read() if p2 else None
    want = expected_ordinals(d1, d2, fastq, W)
    total = len(hl)
    rds = open_ranks(pkg, p1, p2, fastq, W, chunk)
    try:
        sums = [rd.summary() for rd in rds]
        P, Ln = np.zeros_like(hp), np.zeros_like(hl)
        M = np.zeros_like(hm) if n_kmer else None
        seen = np.zeros(total, np.int64)
        stats = []
        for r, rd in enumerate(rds):
            plan = rd.plan(sums)
            assert plan["library_records"] == total and plan["n1"] + plan["n2"] == total, (plan, total)
            assert plan["records"] == len(want[r]), (r, plan, want[r])
            got = []
            pairs_end = 2 * min(plan["n1"], plan["n2"]) if p2 else 0
            for o, packed, lens, nm in read_rank(rd, L, batch, n_kmer, reverse, stride, pairs_end):
                n = len(lens)
                got += range(o, o + n)
                P[o:o + n], Ln[o:o + n] = packed, lens
                if n_kmer:
                    M[o:o + n] = nm
            assert got == want[r], (W, r, got, want[r])
            np.add.at(seen, np.asarray(got, np.int64), 1)
            stats.append(rd.stats())
    finally:
        for rd in rds:
            rd.close()
    assert (seen == 1).all()
    assert np.array_equal(Ln, hl)
    assert np.array_equal(P, hp)
    if n_kmer:
        assert np.array_equal(M, hm)
    return stats


def widths(*sizes):
    return sorted({1, 2, 3, *(max(s, 1) for s in sizes)})


# ---- 1. exactness on the hand-written cases of test_gpu_reader.py; W = file size puts a boundary at every byte
OPTIONS = ((False, False, 1), (True, True, 2), (False, True, 3), (True, False, 1000))   # n_kmer, reverse, batch
CASES = [(False, k) for k in FASTA_CASES] + [(True, k) for k in FASTQ_CASES] + [(False, "char_rules")]


@pytest.mark.parametrize("chunk", CHUNKS)
@pytest.mark.parametrize("fastq,name", CASES)
def test_corner_cases(pkg, tmp_path, fastq, name, chunk):
    data = CHAR_RULES if name == "char_rules" else (FASTQ_CASES if fastq else FASTA_CASES)[name]
    L = 16 if name == "char_rules" else 5
    p = write(tmp_path, "x.fq" if fastq else "x.fa", data)
    other = write(tmp_path, "o.fq" if fastq else "o.fa", b"@o\nCCC\n+\nIII\n" if fastq else b">o\nCCC\n")
    for W in widths(len(data)):
        every_byte = W == len(data)     # W readers per run: one option set each there
        for i, (n_kmer, reverse, batch) in enumerate(OPTIONS):
            if not every_byte or i == CHUNKS.index(chunk):
                check_shard(pkg, p, None, fastq, L, W, n_kmer=n_kmer, reverse=reverse, batch=batch, chunk=chunk)
        # either side of a pair, with a shorter partner
        for p1, p2 in ((p, other), (other, p)):
            check_shard(pkg, p1, p2, fastq, L, W, batch=2, chunk=chunk)
            if not every_byte:
                check_shard(pkg, p1, p2, fastq, L, W, n_kmer=True, reverse=True, batch=1000, chunk=chunk)


@pytest.mark.parametrize("chunk", CHUNKS)
def test_unequal_pairs(pkg, tmp_path, chunk):
    a, b = write(tmp_path, "1.fa", UNEQUAL_1), write(tmp_path, "2.fa", UNEQUAL_2)
    for p1, p2 in ((a, b), (b, a)):
        for W in widths(len(UNEQUAL_1), len(UNEQUAL_2)):
            for batch in (2, 3, 4, 100):
                check_shard(pkg, p1, p2, False, 8, W, reverse=batch % 2 == 0, batch=batch, chunk=chunk)


@pytest.mark.parametrize("fastq", [False, True])
def test_empty_files(pkg, tmp_path, fastq):
    e = write(tmp_path, "e", b"")
    data = b"@a\nACGT\n+\nIIII\n@b\nGG\n+\nII\n" if fastq else b">a\nACGT\n>b\nGG\n"
    full = write(tmp_path, "f", data)
    for chunk in (7, 0):
        for W in widths(len(data)):
            check_shard(pkg, e, None, fastq, 8, W, chunk=chunk)
            check_shard(pkg, e, e, fastq, 8, W, chunk=chunk)
            check_shard(pkg, e, full, fastq, 8, W, batch=2, chunk=chunk)
            check_shard(pkg, full, e, fastq, 8, W, batch=2, chunk=chunk)


# ---- 2. the fuzz of test_gpu_reader.py with random W
def test_fuzz(pkg, tmp_path):
    rng = random.Random(20261022)
    alphabet = b"ACGTacgtNn.x-\r\n>@+"
    weights = [6, 6, 6, 6, 2, 2, 2, 2, 2, 1, 1, 1, 1, 2, 8, 3, 3, 3]

    def text():
        n = rng.choice((0, 1, 5, 40, 200, 600))
        return bytes(rng.choices(alphabet, weights, k=n))

    for case in range(200):
        fastq = rng.random() < 0.5
        paired = rng.random() < 0.4
        p1 = write(tmp_path, f"f{case}_1", text())
        p2 = write(tmp_path, f"f{case}_2", text()) if paired else None
        L = rng.choice((1, 5, 13, 37))
        stride = pkg.synth.stride_bytes(L) + rng.choice((0, 0, 4))
        check_shard(pkg, p1, p2, fastq, L, rng.randint(1, 64), n_kmer=rng.random() < 0.5, reverse=rng.random() < 0.5,
                    stride=stride, batch=rng.choice((2, 3, 1000)), chunk=rng.choice((7, 64, 4096)))


# ---- 3. synthetic ragged libraries with N
def _library(pkg, tr, d, fastq, paired, ragged=80, n_pairs=2000):
    reads, lens = make_dataset(pkg, tr, n_pairs, 100, 31, ragged=ragged, n_rate=0.01 if ragged else 0)
    pkg.synth.write_library(str(d), reads, lens, 100, paired=paired, fastq=fastq)
    ext = "fq" if fastq else "fa"
    if paired:
        return str(d / f"r1.{ext}"), str(d / f"r2.{ext}")
    return str(d / f"r.{ext}"), None


@pytest.mark.parametrize("paired", [False, True])
@pytest.mark.parametrize("fastq", [False, True])
def test_synthetic_library(pkg, tiny_transcriptome, tmp_path, fastq, paired):
    p1, p2 = _library(pkg, tiny_transcriptome, tmp_path, fastq, paired)
    for W in (2, 4, 7):
        for chunk, batch, n_kmer, reverse in ((4096, 1000, True, True), (65536, 2, False, False), (0, 1 << 20, True, False)):
            check_shard(pkg, p1, p2, fastq, 100, W, n_kmer=n_kmer, reverse=reverse, batch=batch, chunk=chunk)


# ---- 4. one rank is the plain reader, batch for batch
@pytest.mark.parametrize("paired", [False, True])
@pytest.mark.parametrize("fastq", [False, True])
def test_one_rank_is_the_plain_reader(pkg, tiny_transcriptome, tmp_path, fastq, paired):
    import torch
    p1, p2 = _library(pkg, tiny_transcriptome, tmp_path, fastq, paired)
    if paired:      # a longer file 2, so that the batches run from the pairs into the drain
        with open(p2, "ab") as f:
            f.write(b"@x\nACGT\n+\nIIII\n" * 5 if fastq else b">x\nACGT\n" * 5)
    for batch, chunk in ((2, 4096), (999, 65536)):
        plain = pkg.DeviceReadPacker(p1, p2, fastq=fastq, device=0, chunk_bytes=chunk)
        shard = pkg.DeviceReadPacker(p1, p2, fastq=fastq, device=0, chunk_bytes=chunk, rank=0, world=1)
        plan = shard.plan([shard.summary()])
        n = 0
        while True:
            assert plain.tell() == n and shard.tell() == n
            a, b = plain.next(100, batch, n_kmer=True), shard.next(100, batch, n_kmer=True)
            torch.cuda.synchronize()
            assert len(a[1]) == len(b[1])
            if len(a[1]) == 0:
                break
            for x, y in zip(a, b):
                assert torch.equal(x, y)
            n += len(a[1])
        assert n == plan["records"] == plan["library_records"]
        plain.close()
        shard.close()


# ---- 5. errors
def test_errors(pkg, tmp_path, tiny_transcriptome):
    p1, p2 = _library(pkg, tiny_transcriptome, tmp_path / "a", False, True, n_pairs=200)
    q1, _ = _library(pkg, tiny_transcriptome, tmp_path / "b", False, True, n_pairs=300)      # another file, another size
    same_size = str(tmp_path / "same_size.fa")      # another file of the same size
    d = bytearray(open(p1, "rb").read())
    d[-2] = ord("A") if d[-2] != ord("A") else ord("C")
    open(same_size, "wb").write(bytes(d))
    fq = str(tmp_path / "as_fastq.fa")
    open(fq, "wb").write(open(p1, "rb").read())

    def sums(a, b, W, fastq=False):
        rds = open_ranks(pkg, a, b, fastq, W, 4096)
        s = [rd.summary() for rd in rds]
        for rd in rds:
            rd.close()
        return s

    good = sums(p1, p2, 3)
    bad_sets = {
        "another file": [good[0], sums(q1, p2, 3)[1], good[2]],
        "same size, other contents": [good[0], good[1], sums(same_size, p2, 3)[2]],
        "another pair partner": [good[0], sums(p1, q1, 3)[1], good[2]],
        "single-ended": [good[0], sums(p1, None, 3)[1], good[2]],
        "fastq differs": [sums(fq, p2, 3, fastq=True)[0], good[1], good[2]],
        "wrong order": [good[1], good[0], good[2]],
        "another world": sums(p1, p2, 2) + [good[2]],
        "wrong count": good[:2],
    }
    rds = open_ranks(pkg, p1, p2, False, 3, 4096)
    for rd in rds:
        rd.summary()
    for name, s in bad_sets.items():
        for rd in rds:
            with pytest.raises(pkg.pregraph.SdtGpuError) as e:
                rd.plan(s)
            assert e.value.code == EINVAL, name
            with pytest.raises(pkg.pregraph.SdtGpuError) as e:      # a refused plan leaves the reader unplanned
                rd.next(100, 10)
            assert e.value.code == ESTATE, name
    with pytest.raises(pkg.pregraph.SdtGpuError) as e:          # a rank's own block must be the one it made
        rds[1].plan([good[0], sums(p1, p2, 3)[1][:-1] + b"\x01", good[2]])
    assert e.value.code == EINVAL
    assert [rd.plan(good)["records"] for rd in rds] == [rd.plan(good)["records"] for rd in rds]
    for rd in rds:
        rd.close()
    fresh = pkg.DeviceReadPacker(p1, p2, device=0, rank=1, world=3)
    with pytest.raises(pkg.pregraph.SdtGpuError) as e:
        fresh.next(100, 10)
    assert e.value.code == ESTATE
    with pytest.raises(pkg.pregraph.SdtGpuError) as e:
        fresh.tell()
    assert e.value.code == ESTATE
    fresh.plan(good)
    with pytest.raises(pkg.pregraph.SdtGpuError) as e:
        fresh.summary()
    assert e.value.code == ESTATE
    fresh.close()
    plain = pkg.DeviceReadPacker(p1, p2, device=0)
    with pytest.raises(pkg.pregraph.SdtGpuError) as e:
        plain.summary()
    assert e.value.code == ESTATE
    import ctypes as C
    assert plain.L.sdtgpu_reader_plan(plain.h, (C.c_uint8 * 256)(), (C.c_uint64 * 4)()) == ESTATE
    assert plain.tell() == 0
    plain.close()


# ---- 6. sharding shards: text uploaded per rank
@pytest.mark.parametrize("fastq", [False, True])
def test_each_rank_reads_about_its_range(pkg, tiny_transcriptome, tmp_path, fastq):
    p1, p2 = _library(pkg, tiny_transcriptome, tmp_path, fastq, True, ragged=0, n_pairs=20_000)   # both files laid out alike
    S1, S2 = os.path.getsize(p1), os.path.getsize(p2)
    assert S1 == S2
    chunk = 16384
    for W in (2, 4, 7):
        stats = check_shard(pkg, p1, p2, fastq, 100, W, batch=4096, chunk=chunk)
        for r, st in enumerate(stats):
            ranges = (lo(S1, r + 1, W) - lo(S1, r, W)) + (lo(S2, r + 1, W) - lo(S2, r, W))
            assert st["text_bytes"] <= 2 * ranges + 2 * 2 * chunk, (W, r, st, ranges)


# ---- 7. C1 end to end: four shard readers into one handle == the plain reader
def nodes_with_ordinals(nodes):
    order = np.lexsort((nodes["key"][:, 3], nodes["key"][:, 2], nodes["key"][:, 1], nodes["key"][:, 0]))
    n = nodes[order]
    return [n[f].copy() for f in ("key", "count", "l_links", "rword", "ordinal")]


def assert_same_nodes(a, b):
    for x, y in zip(nodes_with_ordinals(a), nodes_with_ordinals(b)):
        assert np.array_equal(x, y)


@pytest.mark.parametrize("fastq,sliced,n_kmer", [(False, True, False), (False, True, True), (False, False, False),
                                                 (False, False, True), (True, True, True)])
def test_c1_four_ranks_into_one_handle(pkg, c1_library, fastq, sliced, n_kmer):
    import torch
    c, d = c1_library
    K, kw, L = c["K"], c["key_words"], c["read_len"]
    ext = "fq" if fastq else "fa"
    p1, p2 = str(d / ext / f"r1.{ext}"), str(d / ext / f"r2.{ext}")
    stride = pkg.synth.stride_bytes(L)
    batch = 1 << 17
    dd = 2 if n_kmer else 0
    with pkg.PregraphGPU(K, kw, L, device=0, n_kmer=n_kmer, sliced=sliced) as g, \
            pkg.DeviceReadPacker(p1, p2, fastq=fastq, device=0, chunk_bytes=4 << 20) as rd:
        while True:
            first = rd.tell()
            packed, lens, nmask = rd.next(L, batch, n_kmer=n_kmer)
            if len(lens) == 0:
                break
            torch.cuda.current_stream().synchronize()
            g.push_reads(packed, lens, nmask, n_reads=len(lens), stride_bytes=stride, first_read_ordinal=first, device=True)
            g.sync()
        want = _table(pkg, g, dd)
        want_nodes = g.export_nodes(8)
    W = 4
    rds = open_ranks(pkg, p1, p2, fastq, W, 4 << 20)
    sums = [rd.summary() for rd in rds]
    plans = [rd.plan(sums) for rd in rds]
    assert sum(p["records"] for p in plans) == 1_000_000
    with pkg.PregraphGPU(K, kw, L, device=0, n_kmer=n_kmer, sliced=sliced) as g:
        pushes = []
        for rd in rds:
            while True:
                first = rd.tell()
                packed, lens, nmask = rd.next(L, batch, n_kmer=n_kmer)
                if len(lens) == 0:
                    break
                pushes.append((first, packed, lens, nmask))
        torch.cuda.current_stream().synchronize()
        for first, packed, lens, nmask in sorted(pushes, key=lambda x: x[0]):
            g.push_reads(packed, lens, nmask, n_reads=len(lens), stride_bytes=stride, first_read_ordinal=first, device=True)
            g.sync()
        got = _table(pkg, g, dd)
        got_nodes = g.export_nodes(8)
    for rd in rds:
        rd.close()
    assert got[0] == want[0]
    assert got[1] == want[1]
    assert np.array_equal(got[2], want[2])
    assert np.array_equal(got[3], want[3])
    assert_same_nodes(got_nodes, want_nodes)


# ---- two GPUs: each rank reads its share and builds with the super-k-mer exchange
def _worker(rank, world, port, K, kw, L, p1, p2, out_dir, how):
    sys.path.insert(0, ROOT)
    import torch
    import torch.distributed as dist
    import sdt_pkg
    pkg = sdt_pkg.load()
    from soapdenovo_trans_b200.exchange import SkmExchange, plan_reader
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    rd = pkg.DeviceReadPacker(p1, p2, device=rank, chunk_bytes=4 << 20, rank=rank, world=world)
    if how == "torch":
        plan = plan_reader(rd, dev)
    else:       # the library's communicator, its id carried by torch.distributed
        uid = torch.zeros(128, dtype=torch.uint8, device=dev)
        if rank == 0:
            uid.copy_(torch.frombuffer(bytearray(pkg.pregraph.SkmComm.unique_id()), dtype=torch.uint8))
        dist.broadcast(uid, src=0)
        comm = pkg.pregraph.SkmComm(rank, bytes(uid.cpu().numpy().tobytes()), rank, world)
        plan = rd.plan_exchange(comm)
        comm.close()
    # the same capacity hint on every rank, from the library's records (bench.py's rule on several GPUs)
    inst = plan["library_records"] * (L - K + 1)
    hint = int(min(inst + 1024.0, inst * (1.0 - 0.99 ** K) * 1.05 + 65536.0))
    g = pkg.PregraphGPU(K, kw, L, capacity_hint=hint, device=rank, sliced=True)
    ex = SkmExchange(pkg, g, world, rank, dev)
    stride = pkg.synth.stride_bytes(L)
    n = 0
    while True:
        first = rd.tell()
        packed, lens, _ = rd.next(L, 1 << 17)
        if len(lens) == 0:
            break
        torch.cuda.current_stream().synchronize()
        ex.round(g, packed, len(lens), 0, stride, first, d_lens=lens)
        g.sync()
        n += len(lens)
    assert n == plan["records"]
    ex.flush(g)
    g.sync()
    g.finalize(0)
    np.save(os.path.join(out_dir, f"nodes{rank}.npy"), g.export_nodes(8))
    rd.close()
    g.close()
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.parametrize("how", ["torch", "nccl"])
def test_two_gpu_sharded_read_build(pkg, c1_library, tmp_path, how):
    import torch
    import torch.multiprocessing as mp
    from test_gpu_multi import _free_port
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    c, d = c1_library
    K, kw, L = c["K"], c["key_words"], c["read_len"]
    p1, p2 = str(d / "fa" / "r1.fa"), str(d / "fa" / "r2.fa")
    stride = pkg.synth.stride_bytes(L)
    with pkg.PregraphGPU(K, kw, L, device=0, sliced=True) as g, pkg.DeviceReadPacker(p1, p2, device=0) as rd:
        while True:
            first = rd.tell()
            packed, lens, _ = rd.next(L, 1 << 17)
            if len(lens) == 0:
                break
            torch.cuda.current_stream().synchronize()
            g.push_reads(packed, lens, None, n_reads=len(lens), stride_bytes=stride, first_read_ordinal=first, device=True)
            g.sync()
        g.finalize(0)
        want = g.export_nodes(8)
    mp.spawn(_worker, args=(2, _free_port(), K, kw, L, p1, p2, str(tmp_path), how), nprocs=2, join=True)
    got = np.concatenate([np.load(tmp_path / f"nodes{r}.npy") for r in range(2)])
    assert_same_nodes(got, want)
