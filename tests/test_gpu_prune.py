"""GPU tests of pruning (sdtgpu_prune) against a model of the definition of include/sdtgpu.h stated here in Python.

The model works on the oracle's finalized table as test_gpu_edges.py reads it (k-mers as strings of base codes).  A
round decides from the table as it is at its start and applies every cut together: minor branches (one round), single
tips (one round), minor tips (rounds until one cuts nothing).  Removing a node zeroes its counters and their
reciprocals in its neighbours; after a prune a node without a non-zero counter is deleted.  The device's export must
equal the model's table exactly, and its eight counts the model's."""
import collections
import ctypes
import hashlib
import types

import numpy as np
import pytest
import torch

from conftest import make_dataset
from test_gpu_edges import KEY_CASES, canon, check_edges, model_table, rand_codes, rc, reads_of
from test_gpu_parity import run_gpu
from test_gpu_paths import check_paths

pytestmark = pytest.mark.gpu

LINEAR, DELETED, SINGLE = 1 << 24, 1 << 25, 1 << 27
S, M = 1, 2                                   # PRUNE_SINGLE_TIPS, PRUNE_MINOR_TIPS
ESTATE, EINVAL = 5, 1
M64 = (1 << 64) - 1


def nnz(w):
    return sum(1 for x in range(4) if (w >> (6 * x)) & 63)


def model_prune(t, K, minor_pct, flags):
    """t: model_table of a finalized table -> (the pruned table in model_table's form, the eight counts)"""
    T = {s: [c, L, rw & 0xFFFFFF] for s, (c, L, rw) in t.items()}
    counts = collections.Counter()

    def outs(s, o):                           # (counter index, appended base) of the out-links of (s, o)
        w = T[s][2] if o == 0 else T[s][1]
        return [(x, x if o == 0 else x ^ 2) for x in range(4) if (w >> (6 * x)) & 63]

    def hop(kk, y):                           # -> successor, its orientation, the reciprocal's bit, the oriented k-mer
        f, nk = int(kk[0]), kk[1:] + str(y)
        u, o = canon(nk)
        return u, o, (4 + (f ^ 2) if o else f), nk

    def linear(s):
        return nnz(T[s][1]) == 1 and nnz(T[s][2]) == 1

    def apply(marked, phase):
        clear = collections.Counter()
        for s in marked:
            for o in (0, 1):
                for _, y in outs(s, o):
                    u, _, bit, _ = hop(rc(s) if o else s, y)
                    clear[u] |= 1 << bit
        for s, v in T.items():
            had = v[1] | v[2]
            if s in marked:
                v[1] = v[2] = 0
            for b in range(4):
                if (clear[s] >> b) & 1:
                    v[1] &= ~(63 << (6 * b))
                if (clear[s] >> (4 + b)) & 1:
                    v[2] &= ~(63 << (6 * b))
            counts[phase] += bool(had) and not (v[1] | v[2])

    def minor_branches():
        marked = set()
        for s in T:
            for o in (0, 1):
                ls = outs(s, o)
                if len(ls) < 2:
                    continue
                nb = [hop(rc(s) if o else s, y)[0] for _, y in ls]
                mx = max(T[u][0] for u in nb)
                marked.update(u for u in nb if 100 * T[u][0] < minor_pct * mx)
        apply(marked, 0)

    def tips_round(phase):
        marked, tips = set(), 0
        for s in T:
            if nnz(T[s][1]) + nnz(T[s][2]) != 1:
                continue
            o = 0 if nnz(T[s][2]) else 1
            kk, ((_, y),) = (rc(s) if o else s), outs(s, o)
            path, single, found = [s], T[s][0] == 1, False
            for _ in range(2 * K):
                u, o, bit, kk = hop(kk, y)
                if not linear(u):
                    found = True
                    break
                single &= T[u][0] == 1
                path.append(u)
                ((_, y),) = outs(u, o)
            if not found:
                continue
            side = T[u][2] if bit >= 4 else T[u][1]
            back = (side >> (6 * (bit & 3))) & 63
            isolated = nnz(T[u][1]) + nnz(T[u][2]) == 1
            if isolated or (single if phase == 1 else back < max((side >> (6 * x)) & 63 for x in range(4))):
                tips += not isolated or s <= u
                marked.update(path)
                if isolated:
                    marked.add(u)
        counts["tips"] += tips
        apply(marked, phase)
        return tips

    if minor_pct:
        minor_branches()
    if flags & S:
        tips_round(1)
    rounds = 0
    if flags & M:
        while True:
            rounds += 1
            if not tips_round(2):
                break
    out = {}
    for s, (c, L, R) in T.items():
        rw = R | (LINEAR if nnz(L) == 1 and nnz(R) == 1 else 0) | (DELETED if L == 0 and R == 0 else 0) | (SINGLE if c == 1 else 0)
        out[s] = (c, L, rw)
    live = sum(1 for v in T.values() if v[1] | v[2])
    lin = sum(1 for v in out.values() if v[2] & LINEAR)
    res = dict(minor_branches=counts[0], single_tips=counts[1], minor_tips=counts[2], tips=counts["tips"], rounds=rounds,
               live=live, linear=lin, vertices=live - lin)
    return out, res


def records_of_model(t):
    """a model table as oracle-like records (what check_edges and check_paths read)"""
    rec = np.zeros(len(t), dtype=[("key", "<u8", (4,)), ("count", "<u4"), ("l_links", "<u4"), ("rword", "<u4")])
    for i, (s, (c, L, rw)) in enumerate(sorted(t.items())):
        v = int(s, 4)
        rec[i] = ([(v >> 192) & M64, (v >> 128) & M64, (v >> 64) & M64, v & M64], c, L, rw)
    return types.SimpleNamespace(records=rec)


def device_table(pkg, g, K):
    return model_table(types.SimpleNamespace(records=pkg.nodes_to_records(g.export_nodes(8))), K)


def prune_and_check(pkg, g, t, K, minor_pct, flags, what=""):
    """prunes g and checks export and counts against the model of t -> (model table after, counts)"""
    want_t, want_n = model_prune(t, K, minor_pct, flags)
    res = g.prune(minor_pct, single_tips=bool(flags & S), minor_tips=bool(flags & M))
    assert {k: v for k, v in res.items() if k != "ms"} == want_n, (what, res, want_n)
    got = device_table(pkg, g, K)
    assert got.keys() == want_t.keys(), what
    bad = [(s, got[s], want_t[s]) for s in want_t if got[s] != want_t[s]]
    assert not bad, (what, len(bad), bad[:3])
    return want_t, res


SETTINGS = [(0, S), (0, M), (5, 0), (5, S | M)]


@pytest.mark.parametrize("sliced", [False, True])
@pytest.mark.parametrize("K,kw", KEY_CASES)
def test_prune_against_model(pkg, oracle, tiny_transcriptome, K, kw, sliced):
    L = 150 if K > 63 else 100
    reads, lens = make_dataset(pkg, tiny_transcriptome, 1500, L, 29 + K, ragged=30)
    for d in (0, 2):
        ref = oracle.run_hashing(reads, lens, K, kw, 8, d)
        t = model_table(ref, K)
        for pct, flags in SETTINGS:
            what = f"K={K} d={d} sliced={sliced} pct={pct} flags={flags}"
            g, _, _ = run_gpu(pkg, reads, lens, K, kw, d=d, batches=2, sliced=sliced)
            try:
                want_t, res = prune_and_check(pkg, g, t, K, pct, flags, what)
                if (pct, flags) == (5, S | M):
                    assert res["tips"] > 0 and res["minor_branches"] + res["single_tips"] + res["minor_tips"] > 0, what
                    e = check_edges(pkg, g, records_of_model(want_t), K, what)
                    assert e["vertices"] == res["vertices"] and e["linear_on_edges"] + e["linear_on_cycles"] == res["linear"]
            finally:
                g.close()


@pytest.mark.parametrize("K,kw", [(25, 1), (99, 4)])
def test_prune_n_kmer(pkg, oracle, tiny_transcriptome, K, kw):
    L = 150 if K > 63 else 100
    reads, lens = make_dataset(pkg, tiny_transcriptome, 1500, L, 5 + K, ragged=20, n_rate=0.002)
    ref = oracle.run_hashing(reads, lens, K, kw, 8, 0, n_kmer=1)
    t = model_table(ref, K)
    for sliced in (False, True):
        g, _, _ = run_gpu(pkg, reads, lens, K, kw, d=0, batches=2, sliced=sliced, n_kmer=True)
        try:
            prune_and_check(pkg, g, t, K, 5, S | M, f"-n K={K} sliced={sliced}")
        finally:
            g.close()


# ---- hand-made graphs: a backbone read `cov` times, branches hanging off it
def kmers(s, K):
    return [canon(s[i: i + K])[0] for i in range(len(s) - K + 1)]


def branch(rng, backbone, at, n, K):
    """a read that leaves the backbone after its k-mer at `at` and runs n bases more (n new k-mers)"""
    nxt = int(backbone[at + K])
    x = str((nxt + 1 + int(rng.integers(0, 3))) % 4) + rand_codes(rng, n - 1)
    return backbone[at: at + K] + x, x


def hand_check(pkg, oracle, strings, K, kw, minor_pct, flags, sliced, what):
    reads, lens = reads_of(strings, width=max(max(map(len, strings)), K + 8))
    ref = oracle.run_hashing(reads, lens, K, kw, 8, 0)
    g, _, _ = run_gpu(pkg, reads, lens, K, kw, d=0, batches=1, sliced=sliced)
    try:
        want_t, res = prune_and_check(pkg, g, model_table(ref, K), K, minor_pct, flags, what)
        return g, want_t, res
    except BaseException:
        g.close()
        raise


def alive(t, kms):
    return [bool(t[k][1] or t[k][2] & 0xFFFFFF) for k in kms]


HAND = [(25, 1), (63, 2), (127, 4)]


@pytest.mark.parametrize("sliced", [False, True])
@pytest.mark.parametrize("K,kw", HAND)
def test_prune_tip_length_limit(pkg, oracle, K, kw, sliced):
    """a weak tip of 2K k-mers is cut, one of 2K + 1 is not; the removed k-mers look up as deleted"""
    rng = np.random.default_rng(K)
    bb = rand_codes(rng, 9 * K)
    r1, x1 = branch(rng, bb, 3 * K, 2 * K, K)
    r2, x2 = branch(rng, bb, 6 * K, 2 * K + 1, K)
    g, t, res = hand_check(pkg, oracle, [bb] * 5 + [r1, r2], K, kw, 0, M, sliced, f"length K={K}")
    try:
        gone, kept = kmers(r1, K)[1:], kmers(r2, K)[1:]
        assert not any(alive(t, gone)) and all(alive(t, kept))
        assert res["tips"] == 1 and res["rounds"] == 2 and res["minor_tips"] == 2 * K
        keys = np.array([[(int(k, 4) >> s) & M64 for s in (192, 128, 64, 0)] for k in gone + kept], dtype=np.uint64)
        hits = g.lookup_kmers(keys)
        assert (hits["status"] & pkg.HIT_FOUND).all()
        dele = (hits["rword"] & DELETED) != 0
        assert dele[: len(gone)].all() and not dele[len(gone):].any()
    finally:
        g.close()


@pytest.mark.parametrize("K,kw", HAND)
def test_prune_tip_at_the_maximum(pkg, oracle, K, kw):
    """a tip whose junction counter equals the largest is no minor tip, but goes as a single tip when all its k-mers
    have count 1"""
    rng = np.random.default_rng(K + 1)
    bb = rand_codes(rng, 8 * K)
    r, x = branch(rng, bb, 4 * K, K, K)
    gone = kmers(r, K)[1:]
    g, t, res = hand_check(pkg, oracle, [bb, r], K, kw, 0, M, False, "at max, minor")
    g.close()
    assert all(alive(t, gone)) and res["tips"] == 0 and res["rounds"] == 1
    g, t, res = hand_check(pkg, oracle, [bb, r], K, kw, 0, S, True, "at max, single")
    g.close()
    assert not any(alive(t, gone)) and res["single_tips"] == K and res["tips"] == 1


@pytest.mark.parametrize("sliced", [False, True])
@pytest.mark.parametrize("K,kw", HAND)
def test_prune_isolated_chains_and_hairpins(pkg, oracle, K, kw, sliced):
    """short isolated chains and a short hairpin tip are removed whole by either tip phase; a chain of 2K + 2 k-mers
    and a long hairpin are not"""
    rng = np.random.default_rng(K + 2)
    h = (K + 1) // 2
    u, w = rand_codes(rng, h), rand_codes(rng, h)
    short, long_ = rand_codes(rng, K + 5), rand_codes(rng, 3 * K + 1)
    hp_short, hp_long = rand_codes(rng, 5) + u + rc(u), rand_codes(rng, 2 * K) + w + rc(w)
    strings = [short, long_, hp_short, hp_long] * 2
    for flags in (S, M):
        g, t, res = hand_check(pkg, oracle, strings, K, kw, 0, flags, sliced, f"isolated K={K} flags={flags}")
        g.close()
        assert not any(alive(t, kmers(short, K) + kmers(hp_short, K)))
        assert all(alive(t, kmers(long_, K) + kmers(hp_long, K)))
        assert res["tips"] == 2


@pytest.mark.parametrize("K,kw", HAND)
def test_prune_two_tips_one_round(pkg, oracle, K, kw):
    rng = np.random.default_rng(K + 3)
    bb = rand_codes(rng, 8 * K)
    at = 4 * K
    nxt = int(bb[at + K])
    x1 = str((nxt + 1) % 4) + rand_codes(rng, K)
    x2 = str((nxt + 2) % 4) + rand_codes(rng, K + 3)
    r1, r2 = bb[at: at + K] + x1, bb[at: at + K] + x2
    g, t, res = hand_check(pkg, oracle, [bb] * 5 + [r1, r2], K, kw, 0, M, True, "two tips")
    g.close()
    assert not any(alive(t, kmers(r1, K)[1:] + kmers(r2, K)[1:]))
    assert res["tips"] == 2 and res["rounds"] == 2
    assert t[canon(bb[at: at + K])[0]][2] & LINEAR


@pytest.mark.parametrize("K,kw", HAND)
def test_prune_tip_uncovered_by_a_first_round(pkg, oracle, K, kw):
    """a branch ends in a fork of a strong and a weak tip: the first round cuts the weak tip, which makes the branch
    with the strong tip a tip of the backbone, cut in the second round"""
    rng = np.random.default_rng(K + 4)
    bb = rand_codes(rng, 8 * K)
    at = 4 * K
    s = str((int(bb[at + K]) + 1) % 4) + rand_codes(rng, K // 2)
    p = bb[at: at + K] + s
    c = int(rng.integers(0, 4))
    t1, t2 = str(c) + rand_codes(rng, K // 2), str((c + 1) % 4) + rand_codes(rng, K // 2)
    strings = [bb] * 5 + [p + t1] * 3 + [p + t2]
    g, t, res = hand_check(pkg, oracle, strings, K, kw, 0, M, False, "uncovered")
    g.close()
    assert not any(alive(t, kmers(p + t1, K)[1:] + kmers(p + t2, K)[1:]))
    assert res["tips"] == 2 and res["rounds"] == 3


@pytest.mark.parametrize("K,kw", HAND)
def test_prune_snp_bubble(pkg, oracle, K, kw):
    """the minor branch of a SNP bubble goes at 1:30 (100 < 150) and stays at 1:20 (exactly 5 %)"""
    rng = np.random.default_rng(K + 5)
    snp = rand_codes(rng, 5 * K)
    mid = len(snp) // 2
    alt = snp[:mid] + str((int(snp[mid]) + 1) % 4) + snp[mid + 1:]
    own = [k for k in kmers(alt, K) if k not in set(kmers(snp, K))]
    for cov, goes in ((30, True), (20, False)):
        g, t, res = hand_check(pkg, oracle, [snp] * cov + [alt], K, kw, 5, 0, cov == 30, f"snp 1:{cov}")
        g.close()
        a = alive(t, own)
        if goes:
            assert not a[0] and not a[-1] and res["minor_branches"] >= 2
        else:
            assert all(a) and res["minor_branches"] == 0


@pytest.mark.parametrize("K,kw", HAND)
def test_prune_poly_a(pkg, oracle, K, kw):
    """a poly-A run links its k-mer to itself: the short arms on both sides go as minor tips, the self-linked node
    stays, linear"""
    rng = np.random.default_rng(K + 6)
    arm1, arm2 = rand_codes(rng, K // 2) + "1", "3" + rand_codes(rng, K // 2)
    read = arm1 + "0" * (K + 10) + arm2
    g, t, res = hand_check(pkg, oracle, [read] * 2, K, kw, 5, S | M, False, "poly-A")
    try:
        pa = "0" * K
        assert t[pa][2] & LINEAR and alive(t, [pa]) == [True]
        assert sum(alive(t, sorted(set(kmers(read, K))))) == 1
        e = g.edges_build()
        assert e["cycles"] == 1 and e["edges"] == 1 and e["dangling"] == 0
    finally:
        g.close()


def test_prune_graph_and_paths(pkg, oracle, tiny_transcriptome):
    """after a prune the edge, path and arc calls wait for a new edge build, which builds the pruned graph; the read
    paths then follow the model of test_gpu_paths.py"""
    K = 25
    reads, lens = make_dataset(pkg, tiny_transcriptome, 800, 100, 41, ragged=20)
    ref = oracle.run_hashing(reads, lens, K, 1, 8, 0)
    g, _, _ = run_gpu(pkg, reads, lens, K, 1, d=0, batches=2)
    try:
        g.edges_build()
        stride = pkg.synth.stride_bytes(100)
        packed = torch.from_numpy(pkg.synth.pack_reads(reads, lens, stride)).cuda()
        g.map_reads(packed, torch.from_numpy(lens.astype(np.int32)).cuda(), stride_bytes=stride)
        g.arcs_build()
        want_t, _ = prune_and_check(pkg, g, model_table(ref, K), K, 5, S | M, "paths")
        for fn in (g.edges, g.arcs, g.arcs_build, g.arcs_clear, lambda: g.map_reads(packed, None, n_reads=4, uniform_len=100, stride_bytes=stride)):
            with pytest.raises(pkg.SdtGpuError) as e:
                fn()
            assert e.value.code == ESTATE
        check_paths(pkg, g, records_of_model(want_t), reads, lens, K, what="pruned")
    finally:
        g.close()


def test_prune_noop(pkg, tiny_transcriptome):
    reads, lens = make_dataset(pkg, tiny_transcriptome, 800, 100, 43)
    g, _, st = run_gpu(pkg, reads, lens, 31, 1, d=2)
    try:
        before, ck = pkg.nodes_to_records(g.export_nodes(8)), g.table_checksum()
        res = g.prune(0, single_tips=False, minor_tips=False)
        assert pkg.nodes_to_records(g.export_nodes(8)).tobytes() == before.tobytes()
        assert np.array_equal(g.table_checksum(), ck)
        assert {k: res[k] for k in ("minor_branches", "single_tips", "minor_tips", "tips", "rounds")} == dict.fromkeys(
            ("minor_branches", "single_tips", "minor_tips", "tips", "rounds"), 0)
        assert res["live"] == st.n_nodes - st.n_removed and res["linear"] == st.n_linear
        assert res["vertices"] == res["live"] - res["linear"]
    finally:
        g.close()


def test_prune_c1_order_free(pkg):
    """C1-sized, no Python walk: the single-pass insert and the sliced build give the same pruned table, and the
    accounting holds"""
    synth = pkg.synth
    cfg = synth.CONFIGS["C1"]
    K, L = cfg["K"], cfg["read_len"]
    tr = synth.make_transcriptome(cfg["n_transcripts"], cfg["seed"])
    reads, lens = synth.make_reads(tr, cfg["n_pairs"], L, cfg["seed"])
    stride = synth.stride_bytes(L)
    packed = torch.from_numpy(synth.pack_reads(reads, lens, stride)).cuda()
    n = len(reads)
    out = []
    for sliced in (False, True):
        g = pkg.PregraphGPU(K, cfg["key_words"], L, sliced=sliced)
        try:
            for a in range(0, n, 1 << 18):
                b = min(a + (1 << 18), n)
                g.push_reads(packed[a:b], None, None, n_reads=b - a, uniform_len=L, stride_bytes=stride, first_read_ordinal=a, device=True)
            _, st = g.finalize(cfg["d"])
            before = g.edges_build()
            res = g.prune()
            nodes = pkg.nodes_to_records(g.export_nodes(8))
            deleted = int(((nodes["rword"] & DELETED) != 0).sum())
            live_before = before["vertices"] + st.n_linear
            assert res["live"] == st.n_nodes - deleted == live_before - res["minor_branches"] - res["single_tips"] - res["minor_tips"]
            assert res["vertices"] == res["live"] - res["linear"] and res["tips"] > 0 and res["rounds"] >= 2
            assert res["linear"] == int(((nodes["rword"] & LINEAR) != 0).sum())
            after = g.edges_build()
            assert after["dangling"] == 0 and after["vertices"] == res["vertices"]
            assert after["linear_on_edges"] + after["linear_on_cycles"] == res["linear"]
            out.append((hashlib.sha256(nodes.tobytes()).hexdigest(), g.table_checksum().tolist(),
                        {k: v for k, v in res.items() if k != "ms"}, {k: v for k, v in after.items() if k != "ms"}))
        finally:
            g.close()
    assert out[0] == out[1]


def test_prune_states_and_sharding(pkg, tiny_transcriptome):
    reads, lens = make_dataset(pkg, tiny_transcriptome, 800, 100, 12)
    stride = pkg.synth.stride_bytes(100)
    packed = pkg.synth.pack_reads(reads, lens, stride)
    g = pkg.PregraphGPU(25, 1, 100)
    try:
        with pytest.raises(pkg.SdtGpuError) as e:
            g.prune()
        assert e.value.code == ESTATE                  # before finalize
        g.push_reads(packed[:800], lens[:800], None, n_reads=800, stride_bytes=stride)
        g.finalize(0)
        out, ms = (ctypes.c_uint64 * 8)(), ctypes.c_double()
        for pct, flags in ((-1, 3), (101, 3), (5, 4)):
            assert g.L.sdtgpu_prune(g.h, pct, flags, out, ctypes.byref(ms)) == EINVAL, (pct, flags)
        g.edges_build()
        g.prune()                                      # a refused call did not mark the table pruned
        with pytest.raises(pkg.SdtGpuError) as e:
            g.prune()
        assert e.value.code == ESTATE                  # a table is pruned once
        with pytest.raises(pkg.SdtGpuError) as e:
            g.edges()
        assert e.value.code == ESTATE
        g.edges_build()
        g.edges()
        g.reset()
        with pytest.raises(pkg.SdtGpuError) as e:
            g.prune()
        assert e.value.code == ESTATE                  # after reset
        g.push_reads(packed[800:], lens[800:], None, n_reads=len(reads) - 800, stride_bytes=stride)
        g.finalize(0)
        assert g.lookup_route()["deLowKmer"] == 0
        g.prune()
    finally:
        g.close()
    g = pkg.PregraphGPU(25, 1, 100)
    try:
        g.set_owner(0, 2)
        g.push_reads(packed, lens, None, n_reads=len(reads), stride_bytes=stride)
        g.finalize(0)
        with pytest.raises(pkg.SdtGpuError) as e:
            g.prune()
        assert e.value.code == EINVAL
    finally:
        g.close()
    g = pkg.PregraphGPU(25, 1, 100, capacity_hint=100_000, sliced=True)
    try:
        g.skm_set_world(1, 2)
        with pytest.raises(pkg.SdtGpuError) as e:
            g.prune()
        assert e.value.code == EINVAL
    finally:
        g.close()
