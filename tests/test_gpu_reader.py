"""The device FASTA/FASTQ reader (include/sdtgpu.h sdtgpu_reader_*, pregraph.DeviceReadPacker) against the host
parser: the concatenated device batches (packed rows, lens, nmask) must equal, byte for byte, the concatenated
output of sdtpack_next (one thread, batches as large as the input) for the same files and options.  Then reader +
push_reads_device against sdtpack + push_reads on a C1-sized library, for both insert paths."""
import random

import numpy as np
import pytest

from conftest import make_dataset

pytestmark = pytest.mark.gpu

CHAR_RULES = b">a\nacgtACGTnN..xx-ACGT\r\n>b desc\nACGTACGTACGTACGTACGT\nTTTTTTTT\n>c\n\n>d\nGATTACA"
UNEQUAL_1, UNEQUAL_2 = b">1\nAACCGGTT\n>2\nACGT\n>3\nGGGG\n", b">1\nTTTT\n"


def host_all(pkg, p1, p2, fastq, L, n_kmer, reverse, stride):
    """sdtpack_next with one thread and batches large enough for every record of the files (a pair may still
    come in two batches: when one file's window holds fewer records, the other gives the surplus back)."""
    import os
    max_reads = os.path.getsize(p1) + (os.path.getsize(p2) if p2 else 0) + 4
    rp = pkg.ReadPacker(p1, p2, fastq=fastq, n_threads=1)
    P, Ln, M = [], [], []
    while True:
        packed, lens, nmask = rp.next(L, max_reads, n_kmer=n_kmer, reverse=reverse, stride_bytes=stride)
        if len(lens) == 0:
            break
        P.append(packed.copy()); Ln.append(lens.copy())
        if n_kmer:
            M.append(nmask.copy())
    rp.close()
    if not P:
        return np.zeros((0, stride), np.uint8), np.zeros(0, np.uint32), (np.zeros((0, stride // 2), np.uint8) if n_kmer else None)
    return np.concatenate(P), np.concatenate(Ln), (np.concatenate(M) if n_kmer else None)


def device_all(pkg, p1, p2, fastq, L, n_kmer, reverse, stride, batch, chunk):
    import torch
    P, Ln, M = [], [], []
    with pkg.DeviceReadPacker(p1, p2, fastq=fastq, device=0, chunk_bytes=chunk) as rd:
        while True:
            packed, lens, nmask = rd.next(L, batch, n_kmer=n_kmer, reverse=reverse, stride_bytes=stride)
            assert len(lens) <= batch
            if len(lens) == 0:
                break
            torch.cuda.synchronize()
            P.append(packed.cpu().numpy()); Ln.append(lens.cpu().numpy().view(np.uint32))
            if n_kmer:
                M.append(nmask.cpu().numpy())
        stats = rd.stats()
        assert rd.next(L, batch, n_kmer=n_kmer, reverse=reverse, stride_bytes=stride)[1].numel() == 0
    if not P:
        return np.zeros((0, stride), np.uint8), np.zeros(0, np.uint32), (np.zeros((0, stride // 2), np.uint8) if n_kmer else None), stats
    return np.concatenate(P), np.concatenate(Ln), (np.concatenate(M) if n_kmer else None), stats


def check_same(pkg, p1, p2, fastq, L, n_kmer=False, reverse=False, stride=None, batch=1000, chunk=0):
    stride = stride or pkg.synth.stride_bytes(L)
    hp, hl, hm = host_all(pkg, p1, p2, fastq, L, n_kmer, reverse, stride)
    dp, dl, dm, stats = device_all(pkg, p1, p2, fastq, L, n_kmer, reverse, stride, batch, chunk)
    assert np.array_equal(dl, hl), (len(dl), len(hl))
    assert np.array_equal(dp, hp)
    if n_kmer:
        assert np.array_equal(dm, hm)
    assert stats["records"] == len(hl)
    return stats


def write(tmp_path, name, data: bytes) -> str:
    p = tmp_path / name
    p.write_bytes(data)
    return str(p)


# ---- synthetic libraries with ragged lengths and N
@pytest.mark.parametrize("chunk", [4096, 65536, 0])
@pytest.mark.parametrize("paired", [False, True])
@pytest.mark.parametrize("fastq", [False, True])
def test_synthetic_library(pkg, tiny_transcriptome, tmp_path, fastq, paired, chunk):
    reads, lens = make_dataset(pkg, tiny_transcriptome, 2000, 100, 31, ragged=80, n_rate=0.01)
    pkg.synth.write_library(str(tmp_path), reads, lens, 100, paired=paired, fastq=fastq)
    ext = "fq" if fastq else "fa"
    p1 = str(tmp_path / (f"r1.{ext}" if paired else f"r.{ext}"))
    p2 = str(tmp_path / f"r2.{ext}") if paired else None
    for batch, reverse, n_kmer in ((2, False, False), (1000, True, True), (4096, False, True), (1 << 20, True, False)):
        check_same(pkg, p1, p2, fastq, 100, n_kmer=n_kmer, reverse=reverse, batch=batch, chunk=chunk)
    # max_read_len not a multiple of 4, stride wider than it needs
    check_same(pkg, p1, p2, fastq, 37, n_kmer=True, reverse=True, stride=64, batch=999, chunk=chunk)


# ---- hand-written byte strings; chunks far smaller than a record included
CHUNKS = [7, 64, 4096, 0]


@pytest.mark.parametrize("chunk", CHUNKS)
def test_character_rules_truncation_and_n(pkg, tmp_path, chunk):
    p = write(tmp_path, "x.fa", CHAR_RULES)
    for n_kmer in (False, True):
        for reverse in (False, True):
            for batch in (1, 2, 100):
                check_same(pkg, p, None, False, 16, n_kmer=n_kmer, reverse=reverse, batch=batch, chunk=chunk)


@pytest.mark.parametrize("chunk", CHUNKS)
def test_reverse_seq_and_unequal_pairs(pkg, tmp_path, chunk):
    a, b = write(tmp_path, "1.fa", UNEQUAL_1), write(tmp_path, "2.fa", UNEQUAL_2)
    for p1, p2 in ((a, b), (b, a)):
        for batch in (2, 3, 4, 100):
            check_same(pkg, p1, p2, False, 8, reverse=True, batch=batch, chunk=chunk)
            check_same(pkg, p1, p2, False, 8, batch=batch, chunk=chunk)


FASTA_CASES = {
    "crlf_no_final_newline": b">r1\r\nACGTN\r\n>r2\r\nggcc\r\n>r3\r\nTTA",
    "empty_record": b">a\n\n>b\nACGT\n>c\n",
    "header_at_eof": b">a\nACGT\n>b",
    "multi_line_records": b">a\nACGT\nCCCC\nGGGG\n>b\nTT\nAA\n>c\nG\n",
    "runs_of_gt": b">1\nAC\n>2\n>3\nGG\n>4\n>5\n>6\nTT\n>7\n>8\n>9\n>10\nCA\n>11\n>12\n>13\n>14\n>15\nAAA\n",
    "junk_before_first_header": b"junk line\nACGTACGT\n\n+\n@x\n>h1\nACGT\n>h2\nGGTT\n",
    "only_junk": b"no header here\nACGT\n",
    "blank_lines": b"\n\n>a\n\n\n>b\nAC\n\n",
}
FASTQ_CASES = {
    "crlf_no_final_newline": b"@r1\r\nACGT\r\n+\r\nIIII\r\n@r2\r\nGGCA\r\n+\r\nIIII",
    "quality_starts_with_at_or_plus": b"@r1\nACGT\n+\n@III\n@r2\nGGTT\n+r2\n+III\n@r3\nAC\n+\n@@\n@r4\nTTTT\n+\n+@+@\n",
    "junk_before_first_header": b"junk\n@not a header\nACGT\nnot plus\n@r1\nACGT\n+\nIIII\n@r2\nCC\n+\nII\n",
    "trailing_incomplete_record": b"@r1\nACGT\n+\nIIII\n@r2\nGG",
    "header_only_at_eof": b"@r1\nACGT\n+\nIIII\n@r2\n",
    "first_header_decided_by_eof": b"junk\n@r1\nACGT",
    "empty_record": b"@r1\n\n+\n\n@r2\nAC\n+\nII\n",
}


@pytest.mark.parametrize("chunk", CHUNKS)
@pytest.mark.parametrize("fastq,name", [(False, k) for k in FASTA_CASES] + [(True, k) for k in FASTQ_CASES])
def test_corner_cases(pkg, tmp_path, fastq, name, chunk):
    data = (FASTQ_CASES if fastq else FASTA_CASES)[name]
    p = write(tmp_path, "x.fq" if fastq else "x.fa", data)
    for n_kmer, reverse in ((False, False), (True, True)):
        for batch in (1, 2, 1000):
            check_same(pkg, p, None, fastq, 5, n_kmer=n_kmer, reverse=reverse, batch=batch, chunk=chunk)
    # the same file as either side of a pair, with a shorter and a longer partner
    other = write(tmp_path, "o.fq" if fastq else "o.fa", b"@o\nCCC\n+\nIII\n" if fastq else b">o\nCCC\n")
    for p1, p2 in ((p, other), (other, p)):
        check_same(pkg, p1, p2, fastq, 5, batch=2, chunk=chunk)
        check_same(pkg, p1, p2, fastq, 5, n_kmer=True, batch=1000, chunk=chunk)


@pytest.mark.parametrize("fastq", [False, True])
def test_empty_files(pkg, tmp_path, fastq):
    e = write(tmp_path, "e", b"")
    full = write(tmp_path, "f", b"@a\nACGT\n+\nIIII\n@b\nGG\n+\nII\n" if fastq else b">a\nACGT\n>b\nGG\n")
    for chunk in (7, 0):
        check_same(pkg, e, None, fastq, 8, chunk=chunk)
        check_same(pkg, e, e, fastq, 8, chunk=chunk)
        check_same(pkg, e, full, fastq, 8, batch=2, chunk=chunk)
        check_same(pkg, full, e, fastq, 8, batch=2, chunk=chunk)


def test_junk_longer_than_a_chunk_does_not_grow(pkg, tmp_path):
    recs = b"".join(b">h%d\nACGTACGT\n" % i for i in range(50))
    data = b"J" * 100_000 + b"\n" + recs + b"x" * 50_000 + b"\n" + recs + b"more junk " * 20_000
    p = write(tmp_path, "j.fa", data)
    stats = check_same(pkg, p, None, False, 8, batch=7, chunk=4096)
    # two text slots, the block scratch, and newline + header lists for each slot: nothing grew
    assert stats["allocations"] <= 7, stats
    assert stats["text_bytes"] <= len(data)
    fq = b"".join(b"@h%d\nACGT\n+\nIIII\n" % i for i in range(50))
    p = write(tmp_path, "j.fq", b"J" * 100_000 + b"\n" + fq)
    stats = check_same(pkg, p, None, True, 8, batch=7, chunk=4096)
    assert stats["allocations"] <= 5, stats


@pytest.mark.parametrize("fastq", [False, True])
def test_line_longer_than_a_chunk_grows(pkg, tmp_path, fastq):
    long = b"ACGT" * 25_000
    if fastq:
        data = b"@a\nACGT\n+\nIIII\n@long\n" + long + b"\n+\n" + b"I" * len(long) + b"\n@b\nGG\n+\nII\n"
    else:
        data = b">a\nACGT\n>long\n" + long + b"\n>b\nGG\n"
    p = write(tmp_path, "l.fq" if fastq else "l.fa", data)
    for L, n_kmer in ((100, False), (37, True)):
        stats = check_same(pkg, p, None, fastq, L, n_kmer=n_kmer, batch=2, chunk=4096)
        assert stats["allocations"] > (5 if fastq else 7), stats
    check_same(pkg, p, None, fastq, 100, batch=1000, chunk=0)


def test_fuzz(pkg, tmp_path):
    rng = random.Random(20261021)
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
        check_same(pkg, p1, p2, fastq, L, n_kmer=rng.random() < 0.5, reverse=rng.random() < 0.5, stride=stride,
                   batch=rng.choice((2, 3, 1000)), chunk=rng.choice((7, 64, 4096)))


# ---- end to end at C1 size: reader + push_reads_device == sdtpack + push_reads
@pytest.fixture(scope="module")
def c1_library(pkg, tmp_path_factory):
    c = pkg.synth.CONFIGS["C1"]
    tr = pkg.synth.make_transcriptome(c["n_transcripts"], c["seed"])
    parts = [pkg.synth.make_reads(tr, 250_000, c["read_len"], c["seed"], first_pair=a, ragged=30) for a in (0, 250_000)]
    reads, lens = np.concatenate([p[0] for p in parts]), np.concatenate([p[1] for p in parts])
    rng = np.random.default_rng(c["seed"])
    reads[rng.random(reads.shape) < 0.002] = 4
    d = tmp_path_factory.mktemp("c1")
    for fastq in (False, True):
        pkg.synth.write_library(str(d / ("fq" if fastq else "fa")), reads, lens, c["read_len"], paired=True, fastq=fastq)
    return c, d


def _table(pkg, g, d):
    freq, st = g.finalize(d)
    return (st.n_instances, st.n_nodes, st.n_removed, st.n_linear, st.n_reads), g.table_checksum().tolist(), freq, \
        pkg.nodes_to_records(g.export_nodes(8))


@pytest.mark.parametrize("n_kmer", [False, True])
@pytest.mark.parametrize("sliced", [True, False])
@pytest.mark.parametrize("fastq", [False, True])
def test_c1_end_to_end(pkg, c1_library, fastq, sliced, n_kmer):
    import torch
    c, d = c1_library
    K, kw, L = c["K"], c["key_words"], c["read_len"]
    ext = "fq" if fastq else "fa"
    p1, p2 = str(d / ext / f"r1.{ext}"), str(d / ext / f"r2.{ext}")
    stride = pkg.synth.stride_bytes(L)
    batch = 1 << 17
    # host: sdtpack -> push_reads
    with pkg.PregraphGPU(K, kw, L, device=0, n_kmer=n_kmer, sliced=sliced) as g:
        rp = pkg.ReadPacker(p1, p2, fastq=fastq)
        pushed = 0
        while True:
            packed, lens, nmask = rp.next(L, batch, n_kmer=n_kmer)
            if len(lens) == 0:
                break
            g.push_reads(packed, lens, nmask, n_reads=len(lens), stride_bytes=stride, first_read_ordinal=pushed)
            pushed += len(lens)
        rp.close()
        want = _table(pkg, g, 2 if n_kmer else 0)
    # device: reader -> push_reads_device, here with chunks smaller than one batch of text
    with pkg.PregraphGPU(K, kw, L, device=0, n_kmer=n_kmer, sliced=sliced) as g, \
            pkg.DeviceReadPacker(p1, p2, fastq=fastq, device=0, chunk_bytes=4 << 20) as rd:
        pushed, allocs = 0, None
        while True:
            packed, lens, nmask = rd.next(L, batch, n_kmer=n_kmer)
            if len(lens) == 0:
                break
            torch.cuda.current_stream().synchronize()
            g.push_reads(packed, lens, nmask, n_reads=len(lens), stride_bytes=stride, first_read_ordinal=pushed, device=True)
            g.sync()        # the next batch overwrites nothing the push reads, but torch may reuse the memory
            pushed += len(lens)
            if allocs is None:
                allocs = rd.stats()["allocations"]
            assert rd.stats()["allocations"] == allocs
        got = _table(pkg, g, 2 if n_kmer else 0)
        st = rd.stats()
    assert pushed == 1_000_000 and st["records"] == pushed
    assert got[0] == want[0]
    assert got[1] == want[1]
    assert np.array_equal(got[2], want[2])
    assert np.array_equal(got[3], want[3])
