"""GPU tests of the routed lookups on one device: 2 or 3 "ranks" are handles on device 0, each with its share of the
table, and the halves' buffers (sdtgpu_lookup_stage_* / _answer_buffer / _unstage_buffer) are moved between them
with torch device copies, as a transport between GPUs would move them.  The routed hits must be bit-identical to the
oracle's expectation and to sdtgpu_lookup_*_device on one unsharded handle of the same reads, for every sharding the
insert side has: the sliced build with sdtgpu_set_owner, the single-pass insert with sdtgpu_set_owner, and the
sliced build with the super-k-mer exchange (sdtgpu_skm_set_world)."""
import numpy as np
import pytest

from conftest import make_dataset
from test_gpu_lookup import assert_hits_equal, expected_read_hits, key_queries, table_of
from test_gpu_parity import run_gpu

pytestmark = pytest.mark.gpu

SHARDINGS = ["sliced_owner", "hashed_owner", "skm"]
HINT = 300_000


def _copy(dst: int, src: int, nbytes: int):
    """device memory owned by the library, copied with torch"""
    import torch
    from soapdenovo_trans_b200.exchange import _wrap
    if nbytes:
        dev = torch.device("cuda", 0)
        _wrap(dst, nbytes, dev).copy_(_wrap(src, nbytes, dev))


def build_ranks(pkg, reads, lens, K, kw, world, sharding, d, n_kmer=False, max_read_len=None):
    """world handles on device 0, each holding its share of the table of all reads, finalized with -d d"""
    import torch
    synth = pkg.synth
    L = reads.shape[1]
    mrl = max_read_len or L
    stride = synth.stride_bytes(mrl)
    packed = synth.pack_reads(reads, lens, stride)
    nmask = synth.nmask_reads(reads, stride) if n_kmer else None
    n = len(reads)
    gs = [pkg.PregraphGPU(K, kw, mrl, capacity_hint=HINT, n_kmer=n_kmer, sliced=sharding != "hashed_owner") for _ in range(world)]
    if sharding != "skm":       # replicated reads: every rank pushes all reads and keeps what it owns
        for r, g in enumerate(gs):
            g.set_owner(r, world)
            g.push_reads(packed, lens, nmask, n_reads=n, stride_bytes=stride)
    else:                       # every rank pushes its shard; the records travel to their slices' owners
        for r, g in enumerate(gs):
            g.skm_set_world(r, world)
            lo, hi = r * n // world, (r + 1) * n // world
            g.push_reads(np.ascontiguousarray(packed[lo:hi]), np.ascontiguousarray(lens[lo:hi]),
                         None if nmask is None else np.ascontiguousarray(nmask[lo:hi]), n_reads=hi - lo,
                         stride_bytes=stride, first_read_ordinal=lo)
            g.skm_set_ordinal_bound(n)
        staged = [g.skm_stage() for g in gs]
        rec = int(gs[0].slice_geometry()["record_bytes"])
        for dst, g in enumerate(gs):
            total = sum(s[2][dst] for s in staged)
            buf, off = g.skm_import_buffer(total), 0
            for ptr, starts, counts in staged:
                _copy(buf + off * rec, ptr + starts[dst] * rec, counts[dst] * rec)
                off += counts[dst]
            torch.cuda.synchronize()
            g.skm_import(total)
    for g in gs:
        g.finalize(d)
    return gs


def route(gs, stage, outs):
    """stage(r, g) -> (address, starts, counts) of rank r's staged queries; the hits go to outs[r]"""
    import torch
    world = len(gs)
    staged = [stage(r, g) for r, g in enumerate(gs)]
    qb = 8 * gs[0].lookup_route()["key_words"]
    replies = []
    for dst, g in enumerate(gs):        # every owner receives its queries, in source-rank order, and answers them
        total = sum(s[2][dst] for s in staged)
        q, rp = g.lookup_answer_buffer(total)
        off = 0
        for ptr, starts, counts in staged:
            _copy(q + off * qb, ptr + starts[dst] * qb, counts[dst] * qb)
            off += counts[dst]
        torch.cuda.synchronize()
        g.lookup_answer(total)
        replies.append(rp)
    for src, g in enumerate(gs):        # the hits back into the asker's unstage buffer, in staged order
        back = g.lookup_unstage_buffer()
        _, starts, counts = staged[src]
        for dst in range(world):
            before = sum(staged[s][2][dst] for s in range(src))
            _copy(back + starts[dst] * 16, replies[dst] + before * 16, counts[dst] * 16)
        torch.cuda.synchronize()
        g.lookup_unstage(outs[src])
    return outs


def route_kmers(pkg, gs, parts):
    """parts[r]: rank r's keys (uint64 [n_r, 4]) -> the routed hits of every rank, concatenated"""
    import torch
    keys = [torch.from_numpy(np.ascontiguousarray(p, dtype=np.uint64).view(np.int64)).cuda() for p in parts]
    outs = [torch.full((len(p), 4), -1, dtype=torch.int32, device="cuda") for p in parts]
    route(gs, lambda r, g: g.lookup_stage_kmers(keys[r]), outs)
    return np.concatenate([pkg.hits_numpy(o) for o in outs])


def route_reads(pkg, gs, reads, lens, max_read_len, bounds, n_kmer=False, uniform_len=None):
    """rank r looks up every window of reads[bounds[r]:bounds[r + 1]] -> hits [n_reads, maxwin] of all ranks (bounds
    are multiples of 4, so that every rank's reads start 16-byte aligned)"""
    import torch
    synth = pkg.synth
    stride = synth.stride_bytes(max_read_len)
    packed = torch.from_numpy(synth.pack_reads(reads, lens, stride)).cuda()
    d_lens = None if uniform_len is not None else torch.from_numpy(lens.astype(np.int32)).cuda()
    nmask = torch.from_numpy(synth.nmask_reads(reads, stride)).cuda() if n_kmer else None
    maxwin = max_read_len - gs[0].K + 1
    outs = [torch.full((b - a, maxwin, 4), -1, dtype=torch.int32, device="cuda") for a, b in zip(bounds[:-1], bounds[1:])]

    def stage(r, g):
        a, b = bounds[r], bounds[r + 1]
        return g.lookup_stage_reads(packed[a:b], None if d_lens is None else d_lens[a:b], None if nmask is None else nmask[a:b],
                                    n_reads=b - a, uniform_len=uniform_len or 0, stride_bytes=stride)
    route(gs, stage, outs)
    return np.concatenate([pkg.hits_numpy(o) for o in outs])


def close_all(gs):
    for g in gs:
        g.close()


@pytest.mark.parametrize("K,kw", [(25, 1), (63, 2), (127, 4)])
@pytest.mark.parametrize("sharding", SHARDINGS)
def test_owner_agrees_with_build(pkg, oracle, tiny_transcriptome, sharding, K, kw):
    """Staging rank r's exported nodes puts every one of them in region r, and the shares add up to the table."""
    import torch
    L = 150 if K > 63 else 100
    reads, lens = make_dataset(pkg, tiny_transcriptome, 1200, L, 3 + K, ragged=30)
    ref = oracle.run_hashing(reads, lens, K, kw, 8, 0)
    for world in (2, 3):
        gs = build_ranks(pkg, reads, lens, K, kw, world, sharding, 0)
        try:
            total = 0
            for r, g in enumerate(gs):
                route_info = g.lookup_route()
                assert (route_info["rank"], route_info["world"]) == (r, world)
                nodes = g.export_nodes(8)
                keys = torch.from_numpy(np.ascontiguousarray(nodes["key"]).view(np.int64)).cuda()
                _, starts, counts = g.lookup_stage_kmers(keys)
                assert counts == [len(nodes) if q == r else 0 for q in range(world)], (sharding, K, world, r)
                total += len(nodes)
            assert total == ref.nodes
        finally:
            close_all(gs)


@pytest.mark.parametrize("K,kw", [(25, 1), (63, 2), (127, 4)])
@pytest.mark.parametrize("sharding", SHARDINGS)
def test_routed_kmers(pkg, oracle, tiny_transcriptome, sharding, K, kw):
    """Present keys, their reverse complements, absent and malformed keys, split unevenly over 3 ranks (one asks
    nothing): the routed hits equal the oracle's and one unsharded handle's, with -d 0 and 2."""
    L = 150 if K > 63 else 100
    reads, lens = make_dataset(pkg, tiny_transcriptome, 1200, L, 31 + K, ragged=30)
    rng = np.random.default_rng(K)
    for d in (0, 2):
        ref = oracle.run_hashing(reads, lens, K, kw, 8, d)
        queries, want = key_queries(pkg, oracle, ref, K, kw, rng)
        perm = rng.permutation(len(queries))
        queries, want = queries[perm], want[perm]
        n = len(queries)
        parts = [queries[:0], queries[: n // 5], queries[n // 5:]]
        gs = build_ranks(pkg, reads, lens, K, kw, 3, sharding, d)
        try:
            got = route_kmers(pkg, gs, parts)
        finally:
            close_all(gs)
        assert_hits_equal(got, want, f"{sharding} K={K} d={d}")
        one, _, _ = run_gpu(pkg, reads, lens, K, kw, d=d, hint=HINT if sharding != "hashed_owner" else 0, sliced=sharding != "hashed_owner")
        try:
            assert_hits_equal(got, one.lookup_kmers(queries), f"{sharding} K={K} d={d} vs one handle")
        finally:
            one.close()


@pytest.mark.parametrize("sharding", SHARDINGS)
def test_routed_reads(pkg, oracle, tiny_transcriptome, sharding):
    """Ragged reads with max_read_len > L, reads of another transcriptome (absent windows), uniform lengths (one
    longer than max_read_len: truncated) and -n reads with N-runs: the routed hits equal expected_read_hits and the
    unsharded handle's lookup_reads."""
    import torch
    synth = pkg.synth
    for K, kw in ((31, 1), (127, 4)):
        L = 150 if K > 63 else 100
        mrl = L + 13
        reads, lens = make_dataset(pkg, tiny_transcriptome, 800, L, 5 + K, ragged=40)
        other, olens = make_dataset(pkg, synth.make_transcriptome(20, 8), 200, L, 77, ragged=40)
        q, qlens = np.concatenate([reads, other]), np.concatenate([lens, olens])
        ref = oracle.run_hashing(reads, lens, K, kw, 8, 1, max_read_len=mrl)
        want = expected_read_hits(pkg, oracle, table_of(ref), q, qlens, K, kw, mrl)
        n = len(q)
        gs = build_ranks(pkg, reads, lens, K, kw, 2, sharding, 1, max_read_len=mrl)
        try:
            got = route_reads(pkg, gs, q, qlens, mrl, [0, n // 12 * 4, n])
        finally:
            close_all(gs)
        assert_hits_equal(got, want, f"ragged {sharding} K={K}")
        one, _, _ = run_gpu(pkg, reads, lens, K, kw, d=1, hint=HINT, max_read_len=mrl, sliced=sharding != "hashed_owner")
        try:
            stride = synth.stride_bytes(mrl)
            packed = torch.from_numpy(synth.pack_reads(q, qlens, stride)).cuda()
            d_lens = torch.from_numpy(qlens.astype(np.int32)).cuda()
            assert_hits_equal(got, pkg.hits_numpy(one.lookup_reads(packed, d_lens, None, stride_bytes=stride)), f"ragged {sharding} K={K} vs one handle")
        finally:
            one.close()
        # uniform lengths, and uniform_len beyond max_read_len (truncated); 3 ranks, the first asks nothing
        ureads, ulens = make_dataset(pkg, tiny_transcriptome, 600, L, 9 + K)
        ref = oracle.run_hashing(ureads, ulens, K, kw, 8, 0)
        uq = np.concatenate([ureads, other[:, :L]])
        want = expected_read_hits(pkg, oracle, table_of(ref), uq, None, K, kw, L, uniform_len=L)
        gs = build_ranks(pkg, ureads, ulens, K, kw, 3, sharding, 0)
        try:
            full = np.full(len(uq), L, np.uint32)
            for ul in (L, L + 7):
                got = route_reads(pkg, gs, uq, full, L, [0, 0, len(uq) // 8 * 4, len(uq)], uniform_len=ul)
                assert_hits_equal(got, want, f"uniform_len={ul} {sharding} K={K}")
        finally:
            close_all(gs)
    # -n: windows that hold an N look up key 0 without RC
    K, kw, L = 25, 1, 100
    reads, lens = make_dataset(pkg, tiny_transcriptome, 700, L, 21, ragged=20, n_rate=0.004)
    ref = oracle.run_hashing(reads, lens, K, kw, 8, 0, n_kmer=1)
    table = table_of(ref)
    assert 0 in table
    want = expected_read_hits(pkg, oracle, table, reads, lens, K, kw, L, n_kmer=True)
    gs = build_ranks(pkg, reads, lens, K, kw, 3, sharding, 0, n_kmer=True)
    try:
        got = route_reads(pkg, gs, reads, lens, L, [0, 100, 900, len(reads)], n_kmer=True)
    finally:
        close_all(gs)
    assert_hits_equal(got, want, f"-n {sharding}")
    assert ((got["status"] == pkg.HIT_WINDOW | pkg.HIT_FOUND) & (got["count"] == table[0][0])).sum() >= 1


@pytest.mark.parametrize("sharding", SHARDINGS)
def test_routed_hot_kmers(pkg, oracle, sharding):
    """Poly-A reads and one read repeated 20 000 times: one owner receives most of the queries."""
    K, kw, L = 31, 1, 100
    rng = np.random.default_rng(5)
    one = rng.integers(0, 4, size=L, dtype=np.uint8)
    reads = np.concatenate([np.zeros((600, L), np.uint8), np.tile(one, (20000, 1))])
    lens = np.full(len(reads), L, np.uint32)
    ref = oracle.run_hashing(reads, lens, K, kw, 8, 0)
    gs = build_ranks(pkg, reads, lens, K, kw, 2, sharding, 0)
    try:
        keys = np.ascontiguousarray(ref.records["key"])
        h = route_kmers(pkg, gs, [keys[:3], keys[3:]])
        assert (h["status"] == pkg.HIT_WINDOW | pkg.HIT_FOUND).all()
        for f in ("count", "l_links", "rword"):
            assert np.array_equal(h[f], ref.records[f]), f
        q = reads[590:4000]
        want = expected_read_hits(pkg, oracle, table_of(ref), q, lens[590:4000], K, kw, L)
        assert_hits_equal(route_reads(pkg, gs, q, lens[590:4000], L, [0, 8, len(q)]), want, f"hot reads {sharding}")
    finally:
        close_all(gs)


def test_routed_state(pkg, oracle, tiny_transcriptome):
    """Before finalize and after reset: ESTATE; unstage without a stage: ESTATE; after reset, push and finalize the
    routed hits see the new table."""
    import torch
    K, kw, L = 31, 1, 100
    synth = pkg.synth
    stride = synth.stride_bytes(L)
    a, alens = make_dataset(pkg, tiny_transcriptome, 600, L, 1)
    b, blens = make_dataset(pkg, synth.make_transcriptome(20, 9), 600, L, 2)
    ref_b = oracle.run_hashing(b, blens, K, kw, 8, 0)
    keys = torch.from_numpy(np.ascontiguousarray(ref_b.records["key"]).view(np.int64)).cuda()
    out = torch.empty((len(keys), 4), dtype=torch.int32, device="cuda")

    def estate(fn):
        with pytest.raises(pkg.SdtGpuError) as e:
            fn()
        assert e.value.code == 5

    gs = [pkg.PregraphGPU(K, kw, L, capacity_hint=HINT, sliced=True) for _ in range(2)]
    try:
        for r, g in enumerate(gs):
            g.set_owner(r, 2)
            g.push_reads(synth.pack_reads(a, alens, stride), None, None, n_reads=len(a), uniform_len=L, stride_bytes=stride)
            estate(lambda: g.lookup_stage_kmers(keys))
            estate(lambda: g.lookup_answer_buffer(10))
            estate(lambda: g.lookup_unstage(out))
            g.finalize(0)
            estate(lambda: g.lookup_unstage_buffer())
            estate(lambda: g.lookup_unstage(out))
        route_kmers(pkg, gs, [ref_b.records["key"][:0], ref_b.records["key"]])
        for g in gs:
            estate(lambda: g.lookup_unstage(out))         # the stage was used up
            g.lookup_stage_kmers(keys)
            g.reset()
            estate(lambda: g.lookup_unstage(out))
            estate(lambda: g.lookup_stage_kmers(keys))
            estate(lambda: g.lookup_answer(0))
        for g in gs:
            g.push_reads(synth.pack_reads(b, blens, stride), None, None, n_reads=len(b), uniform_len=L, stride_bytes=stride)
            g.finalize(0)
        rk = np.ascontiguousarray(ref_b.records["key"])
        h = route_kmers(pkg, gs, [rk[:100], rk[100:]])
        assert (h["status"] == pkg.HIT_WINDOW | pkg.HIT_FOUND).all()
        for f in ("count", "l_links", "rword"):
            assert np.array_equal(h[f], ref_b.records[f]), f
    finally:
        close_all(gs)


def test_exchange_world_of_one(pkg, oracle, tiny_transcriptome):
    """A communicator of one rank on device 0: lookup_*_exchange equals lookup_* for both insert paths, also with no
    queries; a handle sharded for two ranks is refused with EINVAL."""
    import torch
    K, kw, L = 31, 1, 100
    synth = pkg.synth
    reads, lens = make_dataset(pkg, tiny_transcriptome, 600, L, 4, ragged=30)
    ref = oracle.run_hashing(reads, lens, K, kw, 8, 0)
    rng = np.random.default_rng(1)
    queries, want = key_queries(pkg, oracle, ref, K, kw, rng)
    stride = synth.stride_bytes(L)
    packed = torch.from_numpy(synth.pack_reads(reads, lens, stride)).cuda()
    d_lens = torch.from_numpy(lens.astype(np.int32)).cuda()
    comm = pkg.pregraph.SkmComm(0, pkg.pregraph.SkmComm.unique_id(), 0, 1)
    try:
        for sliced in (False, True):
            g, _, _ = run_gpu(pkg, reads, lens, K, kw, hint=HINT if sliced else 0, sliced=sliced)
            try:
                got = g.lookup_kmers_exchange(comm, queries)
                assert_hits_equal(got, want, f"world 1 sliced={sliced}")
                assert_hits_equal(got, g.lookup_kmers(queries), f"world 1 sliced={sliced} vs lookup_kmers")
                assert g.last_collective_ms >= 0
                assert len(g.lookup_kmers_exchange(comm, np.zeros((0, 4), np.uint64))) == 0
                rr = g.lookup_reads_exchange(comm, packed, d_lens, None, stride_bytes=stride)
                assert torch.equal(rr, g.lookup_reads(packed, d_lens, None, stride_bytes=stride))
                assert g.lookup_reads_exchange(comm, packed[:0], d_lens[:0], None, stride_bytes=stride).shape[0] == 0
            finally:
                g.close()
        with pkg.PregraphGPU(K, kw, L) as g:
            g.set_owner(0, 2)
            g.push_reads(synth.pack_reads(reads, lens, stride), lens, None, n_reads=len(reads), stride_bytes=stride)
            g.finalize(0)
            with pytest.raises(pkg.SdtGpuError) as e:
                g.lookup_kmers_exchange(comm, queries)
            assert e.value.code == 1
    finally:
        comm.close()
