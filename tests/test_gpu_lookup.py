"""GPU tests of the lookups in a finalized table (sdtgpu_lookup_kmers_device, sdtgpu_lookup_reads_device), through
the C ABI, bit-exact against the oracle: every hit's count, l_links and rword equal the oracle's record of the
canonical k-mer, FOUND exactly for the keys in the table, RC exactly for queries whose canonical key is their
reverse complement, status 0 for malformed keys and windows a read does not have.  Both insert paths (single-pass
insert and sliced build) feed the same index."""
import numpy as np
import pytest

from conftest import make_dataset
from test_gpu_parity import run_gpu

pytestmark = pytest.mark.gpu

KEY_CASES = [(25, 1), (31, 1), (33, 2), (63, 2), (63, 4), (127, 4)]


def key_int(k) -> int:
    return (int(k[0]) << 192) | (int(k[1]) << 128) | (int(k[2]) << 64) | int(k[3])


def int_key(v: int):
    return [(v >> (64 * (3 - q))) & 0xFFFFFFFFFFFFFFFF for q in range(4)]


def revcomp_keys(oracle, keys, K, kw):
    """sdto_reverse_complement of every row of keys (uint64 [n, 4])."""
    L = oracle.lib()
    out = np.empty_like(keys)
    m = oracle.Kmer()
    for i, k in enumerate(keys):
        for q in range(4):
            m.w[q] = int(k[q])
        r = L.sdto_reverse_complement(m, K, kw)
        out[i] = list(r.w)
    return out


def table_of(ref):
    """canonical key (int) -> (count, l_links, rword) of the oracle's records"""
    rec = ref.records
    return {key_int(k): (int(c), int(l), int(r)) for k, c, l, r in zip(rec["key"], rec["count"], rec["l_links"], rec["rword"])}


def hits_from(pkg, rows):
    return np.ascontiguousarray(np.array(rows, dtype=np.uint32).reshape(-1, 4)).view(pkg.HIT_DTYPE)[:, 0]


def assert_hits_equal(got, want, what=""):
    assert got.shape == want.shape, (what, got.shape, want.shape)
    bad = np.nonzero((got.view(np.uint32).reshape(got.shape + (4,)) != want.view(np.uint32).reshape(want.shape + (4,))).any(axis=-1))
    if len(bad[0]):
        first = tuple(int(b[0]) for b in bad)
        raise AssertionError(f"{what}: {len(bad[0])} hits differ; first at {first}: got {got[first]}, want {want[first]}")


def key_queries(pkg, oracle, ref, K, kw, rng):
    """-> (queries uint64 [n, 4], expected hits): present keys, their reverse complements, absent keys (canonical and
    reverse-complemented), malformed keys"""
    W, F, RC = pkg.HIT_WINDOW, pkg.HIT_FOUND, pkg.HIT_RC
    table = table_of(ref)
    keys = np.ascontiguousarray(ref.records["key"])
    vals = [table[key_int(k)] for k in keys]
    rcs = revcomp_keys(oracle, keys, K, kw)
    assert all(key_int(a) < key_int(b) for a, b in zip(keys[:1000], rcs[:1000]))      # the records hold canonical keys
    mask = (1 << (2 * K)) - 1
    absent = []
    while len(absent) < 2000:
        v = int.from_bytes(rng.bytes(32), "little") & mask
        absent.append(int_key(v))
    absent = np.array(absent, dtype=np.uint64)
    absent_rc = revcomp_keys(oracle, absent, K, kw)
    canon = np.array([a if key_int(a) < key_int(b) else b for a, b in zip(absent, absent_rc)], dtype=np.uint64)
    canon = canon[[key_int(k) not in table for k in canon]]
    canon_rc = revcomp_keys(oracle, canon, K, kw)
    # malformed: bit 2K set (for K = 127 that is bit 62 of key[0]); for keys of fewer than 4 device words, a non-zero
    # unused word; the all-ones word pattern of an empty slot
    src = keys[: min(len(keys), 300)]
    bad = []
    for k in src:
        b = k.copy()
        b[3 - (2 * K) // 64] |= np.uint64(1 << ((2 * K) % 64))
        bad.append(b)
        if 2 * K <= 192:
            b = k.copy()
            b[0] = np.uint64(1)
            bad.append(b)
    bad.append(np.full(4, 0xFFFFFFFFFFFFFFFF, dtype=np.uint64))
    bad.append(np.array([0, 0, 0, 1 << 63] if K < 32 else [1 << 63, 0, 0, 0], dtype=np.uint64))
    bad = np.array(bad, dtype=np.uint64)
    queries = np.concatenate([keys, rcs, canon, canon_rc, bad]).astype(np.uint64)
    rows = ([(c, l, r, W | F) for c, l, r in vals] + [(c, l, r, W | F | RC) for c, l, r in vals]
            + [(0, 0, 0, W)] * len(canon) + [(0, 0, 0, W | RC)] * len(canon_rc) + [(0, 0, 0, 0)] * len(bad))
    return queries, hits_from(pkg, rows)


@pytest.mark.parametrize("sliced", [False, True])
@pytest.mark.parametrize("K,kw", KEY_CASES)
def test_lookup_kmers_against_oracle(pkg, oracle, tiny_transcriptome, K, kw, sliced):
    import torch
    L = 150 if K > 63 else 100
    reads, lens = make_dataset(pkg, tiny_transcriptome, 1200, L, 31 + K, ragged=30)
    rng = np.random.default_rng(K)
    for d in (0, 2):
        ref = oracle.run_hashing(reads, lens, K, kw, 8, d)
        g, freq, st = run_gpu(pkg, reads, lens, K, kw, d=d, batches=2, hint=300_000 if sliced else 0, sliced=sliced)
        try:
            assert st.n_nodes == ref.nodes
            queries, want = key_queries(pkg, oracle, ref, K, kw, rng)
            got = g.lookup_kmers(queries)
            assert_hits_equal(got, want, f"K={K} kw={kw} d={d} sliced={sliced}")
            # a CUDA tensor in, a CUDA tensor out; the index is kept between calls
            got2 = g.lookup_kmers(torch.from_numpy(queries.view(np.int64)).cuda())
            assert got2.is_cuda and np.array_equal(pkg.hits_numpy(got2), got)
        finally:
            g.close()


def expected_read_hits(pkg, oracle, table, reads, lens, K, kw, max_read_len, n_kmer=False, uniform_len=None):
    """what every window of every read must give: the oracle's chop of the read (truncated to max_read_len)"""
    W, F, RC = pkg.HIT_WINDOW, pkg.HIT_FOUND, pkg.HIT_RC
    maxwin = max_read_len - K + 1
    want = np.zeros((len(reads), maxwin), dtype=pkg.HIT_DTYPE)
    mask = (1 << (2 * K)) - 1
    for r in range(len(reads)):
        ln = min(uniform_len if uniform_len is not None else int(lens[r]), max_read_len, reads.shape[1])
        codes = reads[r, :ln]
        kmers, _, _ = oracle.chop_read(codes, K, kw, int(n_kmer))
        assert len(kmers) == (ln - K + 1 if ln >= K + 1 else 0)
        if not len(kmers):
            continue
        has_n = np.concatenate([[0], np.cumsum(codes == 4)])
        v, row = 0, want[r]
        for i, c in enumerate(codes):
            v = ((v << 2) | (int(c) & 3)) & mask
            j = i - K + 1
            if j < 0:
                continue
            canon = key_int(kmers[j])
            n_win = n_kmer and has_n[i + 1] - has_n[j] > 0
            st = W | (RC if (not n_win and v != canon) else 0)
            if canon in table:
                c_, l_, r_ = table[canon]
                row[j] = (c_, l_, r_, st | F)
            else:
                row[j] = (0, 0, 0, st)
    return want


def lookup_reads_host(pkg, g, reads, lens, max_read_len, n_kmer=False, uniform_len=None):
    import torch
    synth = pkg.synth
    stride = synth.stride_bytes(max_read_len)
    packed = torch.from_numpy(synth.pack_reads(reads, lens, stride)).cuda()
    d_lens = None if uniform_len is not None else torch.from_numpy(lens.astype(np.int32)).cuda()
    nmask = torch.from_numpy(synth.nmask_reads(reads, stride)).cuda() if n_kmer else None
    out = g.lookup_reads(packed, d_lens, nmask, n_reads=len(reads), uniform_len=uniform_len or 0, stride_bytes=stride)
    assert out.shape == (len(reads), max_read_len - g.K + 1, 4)
    return pkg.hits_numpy(out)


@pytest.mark.parametrize("sliced", [False, True])
@pytest.mark.parametrize("K,kw", [(31, 1), (63, 2), (127, 4)])
def test_lookup_reads_against_oracle(pkg, oracle, tiny_transcriptome, K, kw, sliced):
    """Ragged reads with max_read_len > L (padding windows), then uniform lengths (one longer than max_read_len:
    truncated); the reads that built the table plus reads of another seed (absent windows)."""
    L = 150 if K > 63 else 100
    mrl = L + 13
    reads, lens = make_dataset(pkg, tiny_transcriptome, 800, L, 5 + K, ragged=40)
    other, olens = make_dataset(pkg, pkg.synth.make_transcriptome(20, 8), 200, L, 77, ragged=40)
    q, qlens = np.concatenate([reads, other]), np.concatenate([lens, olens])
    ref = oracle.run_hashing(reads, lens, K, kw, 8, 1, max_read_len=mrl)
    g, freq, st = run_gpu(pkg, reads, lens, K, kw, d=1, batches=2, hint=200_000 if sliced else 0, max_read_len=mrl, sliced=sliced)
    try:
        table = table_of(ref)
        want = expected_read_hits(pkg, oracle, table, q, qlens, K, kw, mrl)
        got = lookup_reads_host(pkg, g, q, qlens, mrl)
        assert_hits_equal(got, want, "ragged")
        found = (got["status"] & pkg.HIT_FOUND) != 0
        assert found[: len(reads)][want[: len(reads)]["status"] != 0].all() and not found[len(reads):].all()
    finally:
        g.close()
    # uniform lengths: a table of uniform reads, looked up with uniform_len = L and with uniform_len > max_read_len
    ureads, ulens = make_dataset(pkg, tiny_transcriptome, 600, L, 9 + K)
    ref = oracle.run_hashing(ureads, ulens, K, kw, 8, 0)
    g, freq, st = run_gpu(pkg, ureads, ulens, K, kw, d=0, uniform=True, hint=200_000 if sliced else 0, sliced=sliced)
    try:
        table = table_of(ref)
        q = np.concatenate([ureads, other[:, :L]])
        want = expected_read_hits(pkg, oracle, table, q, None, K, kw, L, uniform_len=L)
        assert_hits_equal(lookup_reads_host(pkg, g, q, np.full(len(q), L, np.uint32), L, uniform_len=L), want, "uniform")
        assert_hits_equal(lookup_reads_host(pkg, g, q, np.full(len(q), L, np.uint32), L, uniform_len=L + 7), want, "uniform, truncated")
    finally:
        g.close()


@pytest.mark.parametrize("sliced", [False, True])
def test_lookup_reads_n_kmer(pkg, oracle, tiny_transcriptome, sliced):
    """-n: a window that holds an N looks up key 0 without RC, as it was inserted."""
    for K, kw in ((25, 1), (63, 4)):
        L = 150 if K > 63 else 100
        reads, lens = make_dataset(pkg, tiny_transcriptome, 700, L, 21, ragged=20, n_rate=0.004)
        ref = oracle.run_hashing(reads, lens, K, kw, 8, 0, n_kmer=1)
        g, freq, st = run_gpu(pkg, reads, lens, K, kw, d=0, batches=2, n_kmer=True, hint=200_000 if sliced else 0, sliced=sliced)
        try:
            table = table_of(ref)
            assert 0 in table
            want = expected_read_hits(pkg, oracle, table, reads, lens, K, kw, L, n_kmer=True)
            got = lookup_reads_host(pkg, g, reads, lens, L, n_kmer=True)
            assert_hits_equal(got, want, f"-n K={K}")
            zero = table[0]
            n_windows = (got["status"] == pkg.HIT_WINDOW | pkg.HIT_FOUND) & (got["count"] == zero[0])
            assert n_windows.sum() >= 1
        finally:
            g.close()


@pytest.mark.parametrize("sliced", [False, True])
def test_lookup_state(pkg, oracle, tiny_transcriptome, sliced):
    """Before finalize: ESTATE.  Finalize -> lookup -> reset -> another read set -> finalize -> lookup: the second
    lookups see the second table.  An empty table and reads shorter than K+1: nothing found, no error."""
    import torch
    K, kw, L = 31, 1, 100
    synth = pkg.synth
    stride = synth.stride_bytes(L)
    a, alens = make_dataset(pkg, tiny_transcriptome, 600, L, 1)
    b, blens = make_dataset(pkg, pkg.synth.make_transcriptome(20, 9), 600, L, 2)
    ref_a, ref_b = oracle.run_hashing(a, alens, K, kw, 8, 0), oracle.run_hashing(b, blens, K, kw, 8, 0)
    keys_a, keys_b = np.ascontiguousarray(ref_a.records["key"]), np.ascontiguousarray(ref_b.records["key"])
    d_a = torch.from_numpy(synth.pack_reads(a, alens, stride)).cuda()
    with pkg.PregraphGPU(K, kw, L, capacity_hint=100_000 if sliced else 0, sliced=sliced) as g:
        for push in (False, True):
            if push:
                g.push_reads(synth.pack_reads(a, alens, stride), None, None, n_reads=len(a), uniform_len=L, stride_bytes=stride)
            with pytest.raises(pkg.SdtGpuError) as e:
                g.lookup_kmers(keys_a[:10])
            assert e.value.code == 5
            with pytest.raises(pkg.SdtGpuError) as e:
                g.lookup_reads(d_a, None, None, uniform_len=L)
            assert e.value.code == 5
        g.finalize(0)
        ha = g.lookup_kmers(keys_a)
        assert (ha["status"] == pkg.HIT_WINDOW | pkg.HIT_FOUND).all()
        assert np.array_equal(ha["count"], ref_a.records["count"])
        g.reset()
        with pytest.raises(pkg.SdtGpuError) as e:
            g.lookup_kmers(keys_a[:10])
        assert e.value.code == 5
        g.push_reads(synth.pack_reads(b, blens, stride), None, None, n_reads=len(b), uniform_len=L, stride_bytes=stride)
        g.finalize(0)
        hb = g.lookup_kmers(keys_b)
        assert (hb["status"] == pkg.HIT_WINDOW | pkg.HIT_FOUND).all()
        assert np.array_equal(hb["count"], ref_b.records["count"])
        assert np.array_equal(hb["l_links"], ref_b.records["l_links"]) and np.array_equal(hb["rword"], ref_b.records["rword"])
        only_a = np.array([k for k in keys_a if key_int(k) not in table_of(ref_b)], dtype=np.uint64)
        assert len(only_a) > 100
        assert (g.lookup_kmers(only_a)["status"] == pkg.HIT_WINDOW).all()
        want = expected_read_hits(pkg, oracle, table_of(ref_b), a, alens, K, kw, L)
        assert_hits_equal(pkg.hits_numpy(g.lookup_reads(d_a, None, None, uniform_len=L)), want, "after reset")
        assert len(g.lookup_kmers(np.zeros((0, 4), np.uint64))) == 0
    # an empty table; reads shorter than K+1
    with pkg.PregraphGPU(K, kw, L, sliced=sliced) as g:
        g.finalize(0)
        h = g.lookup_kmers(keys_a[:100])
        assert (h["status"] == pkg.HIT_WINDOW).all() and (h["count"] == 0).all()
        short = torch.from_numpy(np.full(len(a), K, np.int32)).cuda()
        out = g.lookup_reads(d_a, short, None, stride_bytes=stride)
        assert int(out.abs().sum()) == 0
        # every window is a window and nothing is found; RC still tells which windows are reverse complements
        full = pkg.hits_numpy(g.lookup_reads(d_a, None, None, uniform_len=L))
        assert_hits_equal(full, expected_read_hits(pkg, oracle, {}, a, alens, K, kw, L), "empty table")
        assert (full["status"] & pkg.HIT_WINDOW).all() and not (full["status"] & pkg.HIT_FOUND).any()


@pytest.mark.parametrize("K,kw", [(31, 1), (63, 2), (127, 4)])
def test_lookup_hot_kmers(pkg, oracle, K, kw):
    """Poly-A reads and one read repeated 20 000 times: counts in the tens of thousands, exact."""
    L = 150 if K > 63 else 100
    rng = np.random.default_rng(K)
    one = rng.integers(0, 4, size=L, dtype=np.uint8)
    reads = np.concatenate([np.zeros((600, L), np.uint8), np.tile(one, (20000, 1))])
    lens = np.full(len(reads), L, np.uint32)
    ref = oracle.run_hashing(reads, lens, K, kw, 8, 0)
    assert ref.records["count"].max() >= 20000
    for sliced in (False, True):
        g, freq, st = run_gpu(pkg, reads, lens, K, kw, d=0, batches=3, hint=10_000 if sliced else 0, sliced=sliced)
        try:
            keys = np.ascontiguousarray(ref.records["key"])
            h = g.lookup_kmers(keys)
            assert (h["status"] == pkg.HIT_WINDOW | pkg.HIT_FOUND).all()
            for f in ("count", "l_links", "rword"):
                assert np.array_equal(h[f], ref.records[f]), (f, sliced)
            want = expected_read_hits(pkg, oracle, table_of(ref), reads[598:603], lens[598:603], K, kw, L)
            assert_hits_equal(lookup_reads_host(pkg, g, reads[598:603], lens[598:603], L), want, f"hot reads sliced={sliced}")
        finally:
            g.close()


def test_lookup_reads_full_size_c1(pkg):
    """C1's 10^6 device-generated reads, sliced build without a hint: every one of the 7.6 x 10^7 windows is found, and
    the sum of the counts over all windows equals the sum over the nodes of count^2 (a node is hit once per instance)."""
    import torch
    from test_gpu_fullsize import _device_reads, _insert_all
    cfg = dict(pkg.synth.CONFIGS["C1"])
    K, kw, L = cfg["K"], cfg["key_words"], cfg["read_len"]
    dev = torch.device("cuda", 0)
    tr, d_packed, stride = _device_reads(pkg, cfg, cfg["n_pairs"], dev)
    n = d_packed.shape[0]
    with pkg.PregraphGPU(K, kw, L, sliced=True) as g:
        _insert_all(pkg, g, d_packed, L, stride, 1 << 22)
        freq, st = g.finalize(cfg["d"])
        assert st.n_instances == n * (L - K + 1)
        total, found = 0, 0
        for a in range(0, n, 1 << 18):
            b = min(a + (1 << 18), n)
            out = g.lookup_reads(d_packed[a:b], None, None, uniform_len=L, stride_bytes=stride)
            found += int(((out[..., 3] & pkg.HIT_FOUND) != 0).sum())
            total += int(out[..., 0].to(torch.int64).sum())
        nodes = g.export_nodes(8)
    assert found == st.n_instances
    assert total == int((nodes["count"].astype(np.uint64) ** 2).sum())
