"""Pins the oracle (oracle/sdt_oracle.c) against the UNMODIFIED reference: the known-answer values
and table dumps in tests/golden/ were produced by tests/golden/make_golden.py through
oracle/_ref (the reference compiled from /root/reference/src).  Where oracle/_ref is present the
oracle is additionally compared live, record by record, against the reference binary."""
import hashlib
import importlib.util
import json
import os

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
GOLD = os.path.join(HERE, "golden")

with open(os.path.join(GOLD, "kat.json")) as f:
    KAT = json.load(f)
with open(os.path.join(GOLD, "dumps.json")) as f:
    DUMPS = json.load(f)


def _mg():
    spec = importlib.util.spec_from_file_location("make_golden", os.path.join(GOLD, "make_golden.py"))
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    return m


def _codes(seq):
    return np.array([{"A": 0, "C": 1, "T": 2, "G": 3}.get(c, 3) for c in seq], dtype=np.uint8)


@pytest.mark.parametrize("kw", [1, 4])
def test_known_answers_kmer_arithmetic_and_hash(oracle, kw):
    """fwd / reverse complement / KmerSmaller / hash_kmer for both builds (kmer.c, hashFunction.c)."""
    L = oracle.lib()
    for row in KAT[str(kw)]:
        K, seq = row["K"], row["seq"]
        assert [L.sdto_base2int(ord(c)) for c in seq] == list(oracle.encode(seq))
        fwd = oracle.kmer_from_codes(oracle.encode(seq))
        assert [f"{fwd.w[i]:016x}" for i in range(4)] == row["fwd"]
        rc = L.sdto_reverse_complement(fwd, K, kw)
        assert [f"{rc.w[i]:016x}" for i in range(4)] == row["rc"]
        assert L.sdto_kmer_smaller(fwd, rc) == row["smaller"]
        assert L.sdto_hash_kmer(fwd, kw) == row["hash_fwd"]
        assert L.sdto_hash_kmer(rc, kw) == row["hash_rc"]


def test_survey_known_answers(oracle):
    """The values SURVEY.md §8c lists (probe of the reference during the survey)."""
    L = oracle.lib()
    k = oracle.kmer_from_codes(oracle.encode("ACGTACGTACGTACGTACGTACGTA"))
    assert k.w[3] == 0x787878787878 and L.sdto_hash_kmer(k, 1) == 15503784 and L.sdto_hash_kmer(k, 4) == 9768184
    rc = L.sdto_reverse_complement(k, 25, 1)
    assert rc.w[3] == 0x21e1e1e1e1e1e and L.sdto_hash_kmer(rc, 1) == 9795150
    z = oracle.Kmer()
    assert L.sdto_hash_kmer(z, 1) == 12522122 and L.sdto_hash_kmer(z, 4) == 13012954
    import zlib
    assert (zlib.crc32((0x787878787878).to_bytes(8, "little")) & 0xFFFFFF) == 11165241 != 15503784  # not the standard CRC


def test_growth_sequence(oracle):
    """init_kmerset(1024,0.77f) + put_kmerset growth: sizes and max values (newhash.c:116-193, 293-350)."""
    sizes = [row[0] for row in KAT["grow"]]
    assert sizes[:5] == [1031, 2063, 4127, 8263, 16529]
    L = oracle.lib()
    n = 1031
    assert L.sdto_find_next_prime(1024) == 1031
    for want in sizes[1:]:
        n = L.sdto_find_next_prime(n * 2)
        assert n == want
    reads = np.random.default_rng(0).integers(0, 4, size=(3000, 100), dtype=np.uint8)
    r = oracle.run_hashing(reads, np.full(3000, 100, np.uint32), 31, 1, 1, 0)
    row = [g for g in KAT["grow"] if g[0] == int(r.set_info[0, 0])]
    assert row and row[0][1] == int(r.set_info[0, 2])


@pytest.mark.parametrize("name", sorted(DUMPS))
def test_table_dump_matches_reference_golden(oracle, name):
    """Whole hashing stage: (set, slot) layout, keys, counts, links, flags, kmerFreq — bit-exact."""
    g = DUMPS[name]
    spec = g["spec"]
    reads, lens = _mg().dataset(spec)
    if not spec["n"]:
        reads = np.where(reads == 4, 3, reads).astype(np.uint8)   # without -n the parser maps N to G (readseq1by1.c:151-160)
    r = oracle.run_hashing(reads, lens, spec["K"], spec["kw"], spec["p"], spec["d"], n_kmer=spec["n"])
    assert r.nodes == g["nodes"] and r.linear == g["linear"] and r.removed == g["deleted"]
    assert r.instances == g["count_sum"]
    assert r.set_info.tolist() == g["set_info"]
    assert r.kmerfreq[1:256].tolist() == g["kmerfreq"]
    assert hashlib.sha256(np.ascontiguousarray(r.records).tobytes()).hexdigest() == g["sha256"]
    assert hashlib.sha256(oracle.sorted_multiset(r.records).tobytes()).hexdigest() == g["multiset_sha256"]


def test_container_format_and_threads_do_not_change_the_multiset():
    """SURVEY §4: FASTA pair / FASTQ pair / single FASTA give the same table."""
    a, b, c = DUMPS["k31_31mer_ragged"], DUMPS["k31_31mer_fastq"], DUMPS["k31_31mer_single"]
    assert a["sha256"] == b["sha256"] == c["sha256"]
    assert DUMPS["k25_31mer_p8_d0"]["nodes"] == DUMPS["k25_31mer_p3_d2"]["nodes"]


@pytest.mark.parametrize("name", ["k25_31mer_p3_d2", "k63_127mer_d1", "k25_31mer_nkmer", "k127_127mer"])
def test_live_against_reference_binary(oracle, pkg, tmp_path, name):
    """Record-by-record against oracle/_ref; where the reference is not built, against the digest of the same
    reference run stored in tests/golden/dumps.json."""
    spec = DUMPS[name]["spec"]
    mg = _mg()
    reads, lens = mg.dataset(spec)
    r = oracle.run_hashing(reads, lens, spec["K"], spec["kw"], spec["p"], spec["d"], n_kmer=spec["n"])
    if oracle.ref_binary(spec["kw"]) is None:
        g = DUMPS[name]
        assert hashlib.sha256(np.ascontiguousarray(r.records).tobytes()).hexdigest() == g["sha256"]
        assert r.set_info.tolist() == g["set_info"]
        assert g["linear"] == r.linear and g["deleted"] == r.removed
        return
    cfg = mg.write_input(spec, reads, lens, str(tmp_path))
    info, rec, sinfo = oracle.run_reference(cfg, str(tmp_path / "out"), spec["K"], spec["kw"], spec["p"], spec["d"], spec["n"])
    assert np.array_equal(rec, r.records) and np.array_equal(sinfo, r.set_info)
    assert info["linear"] == r.linear and info["deleted"] == r.removed


def test_chop_rules_small_cases(oracle):
    """prev/next rules of chopKmer4read (SURVEY §8a-2) on a hand-checkable read, pure-Python check."""
    rng = np.random.default_rng(5)
    for K, kw in ((13, 1), (33, 4), (65, 4)):
        read = rng.integers(0, 4, size=K + 9, dtype=np.uint8)
        kmers, prev, nxt = oracle.chop_read(read, K, kw)
        n = len(read)
        assert len(kmers) == n - K + 1
        for j in range(n - K + 1):
            w = rc = 0
            for i in range(K):
                w = (w << 2) | int(read[j + i])
                rc |= (int(read[j + i]) ^ 2) << (2 * i)
            if w < rc:
                key, left, right = w, (read[j - 1] if j > 0 else 4), (read[j + K] if j < n - K else 4)
            else:
                key, left, right = rc, ((read[j + K] ^ 2) if j < n - K else 4), ((read[j - 1] ^ 2) if j > 0 else 4)
            got = (int(kmers[j, 0]) << 192) | (int(kmers[j, 1]) << 128) | (int(kmers[j, 2]) << 64) | int(kmers[j, 3])
            assert (got, int(prev[j]), int(nxt[j])) == (key, int(left), int(right))
    assert len(oracle.chop_read(np.zeros(13, np.uint8), 13, 1)[0]) == 0      # len < K+1: skipped
