"""GPU tests of the read paths (sdtgpu_edges_map_reads, sdtgpu_arcs_*) against a model stated here in Python.

The model takes the device's records once check_edges (test_gpu_edges.py) has validated them against the oracle: every
step s_i of every record goes into a dict as (record, i, 0), and its reverse complement as (record, i, 1) unless that
key is already there, which only a palindromic record may cause.  A read window's step is dict.get of the read's
(K+1)-mer; an arc is a vertex window between two mapped steps, read in the vertex's + orientation."""
import collections

import numpy as np
import pytest
import torch

from conftest import make_dataset
from test_gpu_edges import KEY_CASES, canon, check_edges, hand_cases, model_table, rand_codes, rc, reads_of
from test_gpu_parity import run_gpu

pytestmark = pytest.mark.gpu

LINEAR, DELETED = 1 << 24, 1 << 25


def records_of(pkg, g, K):
    edges, seq = g.edges()
    return edges, ["".join(map(str, pkg.edge_codes(edges, seq, i, K))) for i in range(len(edges))]


def model_steps(pkg, edges, seqs, K):
    d = {}
    for r, (e, s) in enumerate(zip(edges, seqs)):
        m, cyc = int(e["length"]), int(e["flags"]) & pkg.EDGE_CYCLE
        word = (s[:m] * ((K + 1) // m + 2)) if cyc else s
        steps = [word[i: i + K + 1] for i in range(m)]
        for i, st in enumerate(steps):
            assert st not in d, ("a step of two records", st, d[st], r)
            d[st] = (r, i, 0)
        for i, st in enumerate(steps):
            k = rc(st)
            if k in d:
                assert d[k][0] == r and int(e["flags"]) & pkg.EDGE_PALINDROME, ("collision", k, d[k], r)
            else:
                d[k] = (r, i, 1)
    return d


def read_strings(reads, lens):
    return ["".join(map(str, reads[i, : int(lens[i])])) for i in range(len(reads))]


def model_map(d, t, strs, K, maxwin, pal):
    """-> (expected steps int64 [n, maxwin, 3], Counter of arcs (from, to) -> count)"""
    want = np.full((len(strs), maxwin, 3), -1, dtype=np.int64)
    arcs = collections.Counter()
    for r, s in enumerate(strs):
        n = len(s) - K
        got = [d.get(s[j: j + K + 1]) for j in range(max(n, 0))]
        for j, st in enumerate(got):
            if st is not None:
                want[r, j] = st
        for j in range(n - 1):
            if got[j] is None or got[j + 1] is None:
                continue
            v, o = canon(s[j + 1: j + 1 + K])
            if t[v][2] & (LINEAR | DELETED):
                continue
            a, b = int(s[j]), int(s[j + K + 1])
            left, right = (a, b) if o == 0 else (b ^ 2, a ^ 2)
            to, fr = d[v + str(right)], d[rc(v) + str(left ^ 2)]
            arcs[(fr[0] << 1 | (0 if pal[fr[0]] else fr[2] ^ 1), to[0] << 1 | to[2])] += 1
    return want, arcs


def device_map(pkg, g, reads, lens, n_kmer=False, batches=1, count_arcs=True):
    synth = pkg.synth
    stride = synth.stride_bytes(g.max_read_len)
    packed = torch.from_numpy(synth.pack_reads(reads, lens, stride)).cuda()
    d_lens = torch.from_numpy(lens.astype(np.int32)).cuda()
    nmask = torch.from_numpy(synth.nmask_reads(reads, stride)).cuda() if n_kmer else None
    n = len(reads)
    outs = []
    cuts = [(n * i // batches) & ~3 for i in range(batches)] + [n]      # (batches start 16-byte aligned)
    for a, b in zip(cuts[:-1], cuts[1:]):
        outs.append(g.map_reads(packed[a:b], d_lens[a:b], None if nmask is None else nmask[a:b], n_reads=b - a,
                                stride_bytes=stride, count_arcs=count_arcs))
    return pkg.steps_numpy(torch.cat(outs))


def device_arcs(g):
    res = g.arcs_build()
    a = g.arcs()
    assert len(a) == res["arcs"] and int(a["count"].sum()) == res["crossings"] and (a["unused"] == 0).all()
    assert (a["count"] > 0).all()
    return a, res


def arc_counter(a):
    return collections.Counter({(int(x["from"]), int(x["to"])): int(x["count"]) for x in a}) if len(a) else collections.Counter()


def check_paths(pkg, g, ref, reads, lens, K, n_kmer=False, what=""):
    """edges checked against the oracle's table, then steps and arcs against the model; -> (steps, arcs)"""
    check_edges(pkg, g, ref, K, what)
    edges, seqs = records_of(pkg, g, K)
    d = model_steps(pkg, edges, seqs, K)
    t = model_table(ref, K)
    pal = [bool(int(e["flags"]) & pkg.EDGE_PALINDROME) for e in edges]
    maxwin = g.max_read_len - K + 1
    want, want_arcs = model_map(d, t, read_strings(reads, lens), K, maxwin, pal)
    got = device_map(pkg, g, reads, lens, n_kmer=n_kmer)
    bad = np.argwhere((got != want).any(axis=-1))
    assert len(bad) == 0, (what, len(bad), [(tuple(x), got[tuple(x)].tolist(), want[tuple(x)].tolist()) for x in bad[:5]])
    a, res = device_arcs(g)
    assert len(a) == len(arc_counter(a)), (what, "an arc key twice")
    assert arc_counter(a) == want_arcs, what
    return got, a


def build_and_check(pkg, oracle, reads, lens, K, kw, d=0, sliced=False, n_kmer=False, what=""):
    ref = oracle.run_hashing(reads, lens, K, kw, 8, d, n_kmer=int(n_kmer))
    g, _, _ = run_gpu(pkg, reads, lens, K, kw, d=d, batches=2, sliced=sliced, n_kmer=n_kmer)
    try:
        return check_paths(pkg, g, ref, reads, lens, K, n_kmer=n_kmer, what=what)
    finally:
        g.close()


@pytest.mark.parametrize("sliced", [False, True])
@pytest.mark.parametrize("K,kw", KEY_CASES)
def test_paths_against_model(pkg, oracle, tiny_transcriptome, K, kw, sliced):
    L = 150 if K > 63 else 100
    reads, lens = make_dataset(pkg, tiny_transcriptome, 800, L, 31 + K, ragged=30)
    for d in (0, 2):
        steps, arcs = build_and_check(pkg, oracle, reads, lens, K, kw, d=d, sliced=sliced, what=f"K={K} kw={kw} d={d} sliced={sliced}")
        assert (steps[..., 0] >= 0).any()
        if d == 0:     # every (K+1)-mer of every read is a step of the graph
            n_win = np.maximum(lens.astype(np.int64) - K, 0)
            assert int((steps[..., 0] >= 0).sum()) == int(n_win.sum())


def test_paths_hot_kmers(pkg, oracle):
    """k-mers shared between transcripts: vertices inside reads, so arcs to check against the model"""
    tr = pkg.synth.make_transcriptome(30, 21, hot=3)
    reads, lens = make_dataset(pkg, tr, 1500, 100, 9, ragged=20)
    for sliced in (False, True):
        for d in (0, 2):
            _, arcs = build_and_check(pkg, oracle, reads, lens, 31, 1, d=d, sliced=sliced, what=f"hot d={d} sliced={sliced}")
            assert len(arcs) > 0 and int(arcs["count"].max()) > 1


@pytest.mark.parametrize("K,kw", [(25, 1), (63, 2), (99, 4)])
def test_paths_n_kmer(pkg, oracle, tiny_transcriptome, K, kw):
    L = 150 if K > 63 else 100
    reads, lens = make_dataset(pkg, tiny_transcriptome, 800, L, 5 + K, ragged=20, n_rate=0.002)
    for sliced in (False, True):
        build_and_check(pkg, oracle, reads, lens, K, kw, sliced=sliced, n_kmer=True, what=f"-n K={K} sliced={sliced}")


@pytest.mark.parametrize("K,kw", [(25, 1), (33, 2), (127, 4)])
@pytest.mark.parametrize("case", ["hairpin", "two_hairpins", "poly_a", "circle", "tandem", "snp", "one_edge", "short"])
def test_paths_hand_made(pkg, oracle, K, kw, case):
    rng = np.random.default_rng(K * 1000 + len(case))
    strings = hand_cases(K, rng)[case]
    reads, lens = reads_of(strings, width=max(max(map(len, strings)), K + 8))
    for sliced in (False, True):
        steps, arcs = build_and_check(pkg, oracle, reads, lens, K, kw, sliced=sliced, what=f"{case} K={K} sliced={sliced}")
        mapped = steps[steps[..., 0] >= 0]
        if case in ("hairpin", "two_hairpins"):    # the palindromic record reports strand 0 only
            assert len(mapped) and (mapped[:, 2] == 0).any()
        if case in ("poly_a", "circle"):            # steps on a cycle, no vertex to cross
            assert len(mapped) == int(np.maximum(lens.astype(np.int64) - K, 0).sum()) and len(arcs) == 0
        if case == "snp":                            # a bubble: each branch entered once and left once
            assert len(arcs) == 4 and (arcs["count"] == 1).all()
        if case == "tandem" and K < 100:             # the read goes round the repeat's loop several times
            assert int(arcs["count"].max()) >= 2
        if case == "short":
            assert len(mapped) == 0 and len(arcs) == 0


def test_paths_short_reads(pkg, oracle):
    K = 25
    rng = np.random.default_rng(3)
    strings = [rand_codes(rng, 80) for _ in range(20)] + [rand_codes(rng, n) for n in (1, K - 1, K, K + 1)]
    reads, lens = reads_of(strings, width=80)
    steps, _ = build_and_check(pkg, oracle, reads, lens, K, 1, what="short reads")
    assert (steps[20:23, :, 0] == -1).all()
    assert steps[23, 0, 0] >= 0 and (steps[23, 1:, 0] == -1).all()


def test_paths_invariance(pkg, tiny_transcriptome):
    """batches, count_arcs = 0, arcs_clear, repeated builds, and the two insert paths"""
    K = 31
    reads, lens = make_dataset(pkg, tiny_transcriptome, 2000, 100, 78, ragged=20)
    per_path = []
    for sliced in (False, True):
        g, _, _ = run_gpu(pkg, reads, lens, K, 1, d=1, batches=3, sliced=sliced)
        try:
            g.edges_build()
            s1 = device_map(pkg, g, reads, lens)
            a1, r1 = device_arcs(g)
            assert r1["arcs"] > 0
            a1b, _ = device_arcs(g)
            assert a1.tobytes() == a1b.tobytes()
            s_nc = device_map(pkg, g, reads, lens, count_arcs=False)
            assert np.array_equal(s_nc, s1)
            assert device_arcs(g)[0].tobytes() == a1.tobytes()      # count_arcs=0 left the counters alone
            g.arcs_clear()
            assert device_arcs(g)[1]["arcs"] == 0
            s3 = device_map(pkg, g, reads, lens, batches=3)
            assert np.array_equal(s3, s1)
            assert device_arcs(g)[0].tobytes() == a1.tobytes()
            g.arcs_clear()
            stride = pkg.synth.stride_bytes(100)
            packed = torch.from_numpy(pkg.synth.pack_reads(reads, lens, stride)).cuda()
            d_lens = torch.from_numpy(lens.astype(np.int32)).cuda()
            g._ck(g.L.sdtgpu_edges_map_reads(g.h, packed.data_ptr(), d_lens.data_ptr(), None, len(reads), 0, stride, None, 1))
            g.sync()
            assert device_arcs(g)[0].tobytes() == a1.tobytes()      # d_out = NULL with count_arcs
            edges, seqs = records_of(pkg, g, K)
            strand = lambda x: seqs[x >> 1] if x & 1 == 0 else rc(seqs[x >> 1])
            per_path.append(sorted((strand(int(x["from"])), strand(int(x["to"])), int(x["count"])) for x in a1))
        finally:
            g.close()
    assert per_path[0] == per_path[1]


def test_paths_states_and_sharding(pkg, tiny_transcriptome):
    reads, lens = make_dataset(pkg, tiny_transcriptome, 600, 100, 13)
    stride = pkg.synth.stride_bytes(100)
    packed = torch.from_numpy(pkg.synth.pack_reads(reads, lens, stride)).cuda()
    d_lens = torch.from_numpy(lens.astype(np.int32)).cuda()

    def estate(fn):
        with pytest.raises(pkg.SdtGpuError) as e:
            fn()
        assert e.value.code == 5

    g = pkg.PregraphGPU(25, 1, 100)
    try:
        g.push_reads(packed.cpu().numpy(), lens, None, n_reads=len(reads), stride_bytes=stride)
        g.finalize(0)
        estate(lambda: g.map_reads(packed, d_lens))
        estate(g.arcs_build)
        estate(g.arcs_clear)
        g.edges_build()
        estate(g.arcs)
        s1 = pkg.steps_numpy(g.map_reads(packed, d_lens))
        r1 = g.arcs_build()
        a1 = g.arcs()
        assert r1["arcs"] > 0
        g.edges_build()                                  # a new build: no arcs, counters zeroed, stamps made again
        estate(g.arcs)
        assert g.arcs_build()["arcs"] == 0
        assert np.array_equal(pkg.steps_numpy(g.map_reads(packed, d_lens)), s1)
        g.arcs_build()
        assert g.arcs().tobytes() == a1.tobytes()
        g.reset()
        estate(lambda: g.map_reads(packed, d_lens))
        estate(g.arcs_build)
        estate(g.arcs)
    finally:
        g.close()
    g = pkg.PregraphGPU(25, 1, 100)
    try:
        g.set_owner(0, 2)
        g.push_reads(packed.cpu().numpy(), lens, None, n_reads=len(reads), stride_bytes=stride)
        g.finalize(0)
        with pytest.raises(pkg.SdtGpuError):
            g.edges_build()
        estate(lambda: g.map_reads(packed, d_lens))
    finally:
        g.close()


def test_paths_c1_without_a_python_walk(pkg):
    """C1 size at -d 0: every read (K+1)-mer maps; consecutive steps through a linear k-mer advance on one record (+1
    on strand 0, -1 on strand 1, modulo m on a cycle); the arc total equals the vertex crossings counted from hits."""
    synth = pkg.synth
    cfg = synth.CONFIGS["C1"]
    K, L = cfg["K"], cfg["read_len"]
    tr = synth.make_transcriptome(cfg["n_transcripts"], cfg["seed"])
    reads, lens = synth.make_reads(tr, cfg["n_pairs"], L, cfg["seed"])
    stride = synth.stride_bytes(L)
    packed = torch.from_numpy(synth.pack_reads(reads, lens, stride)).cuda()
    codes = torch.from_numpy(reads[:, :L].astype(np.int64)).cuda()
    g = pkg.PregraphGPU(K, cfg["key_words"], L, sliced=True)
    try:
        n = len(reads)
        B = 1 << 18
        for a in range(0, n, B):
            b = min(a + B, n)
            g.push_reads(packed[a:b], None, None, n_reads=b - a, uniform_len=L, stride_bytes=stride, first_read_ordinal=a, device=True)
        g.finalize(0)
        g.edges_build()
        edges, _ = g.edges()
        length = torch.from_numpy(edges["length"].astype(np.int64)).cuda()
        cyc = torch.from_numpy((edges["flags"] & pkg.EDGE_CYCLE) != 0).cuda()
        want_cross = 0
        for a in range(0, n, B):
            b = min(a + B, n)
            st = g.map_reads(packed[a:b], None, None, n_reads=b - a, uniform_len=L, stride_bytes=stride)
            hits = g.lookup_reads(packed[a:b], None, None, n_reads=b - a, uniform_len=L, stride_bytes=stride)
            rec = st[..., 0].long() & 0xFFFFFFFF
            pos = st[..., 1].long() & 0xFFFFFFFF
            none = rec == 0xFFFFFFFF
            assert not none[:, :-1].any() and none[:, -1].all()
            rec, idx, strand = rec[:, :-1], pos[:, :-1] >> 1, pos[:, :-1] & 1
            rword = hits[..., 2].long() & 0xFFFFFFFF
            lin = (rword & LINEAR) != 0
            # step j -> j+1 through window j+1, linear
            thru = lin[:, 1:-1]
            same = rec[:, :-1] == rec[:, 1:]
            assert bool(same[thru].all())
            assert bool((strand[:, :-1] == strand[:, 1:])[thru].all())
            m = length[rec[:, :-1]]
            step = torch.where(strand[:, :-1] == 0, 1, -1)
            nxt = idx[:, :-1] + step
            nxt = torch.where(cyc[rec[:, :-1]], (nxt + m) % m, nxt)
            assert bool((nxt == idx[:, 1:])[thru].all())
            # crossings: windows 1 .. maxwin-2 at a vertex with both link bases' counters non-zero
            w = torch.arange(1, L - K, device="cuda")
            h = hits[:, 1:-1]
            lw = h[..., 1].long() & 0xFFFFFF
            rw = rword[:, 1:-1] & 0xFFFFFF
            isrc = (h[..., 3] & pkg.HIT_RC) != 0
            c = codes[a:b]
            prev, nextb = c[:, w - 1], c[:, w + K]
            left = torch.where(isrc, nextb ^ 2, prev)
            right = torch.where(isrc, prev ^ 2, nextb)
            vert = ((h[..., 3] & pkg.HIT_FOUND) != 0) & ~lin[:, 1:-1] & ((rword[:, 1:-1] & DELETED) == 0)
            ok = vert & (((lw >> (6 * left)) & 63) > 0) & (((rw >> (6 * right)) & 63) > 0)
            want_cross += int(ok.sum())
        res = g.arcs_build()
        assert res["arcs"] > 0 and res["crossings"] == want_cross
    finally:
        g.close()
