"""GPU tests of the edge build (sdtgpu_edges_build, sdtgpu_edges_buffers) against a model stated here in Python.

The model reads the oracle's records: k-mers are strings of base codes ('0'..'3', A C T G), so that string order is
the order of the keys as integers and the reverse complement is a reversal plus a translation.  It follows the
definition of include/sdtgpu.h: out-links of (v,+) are the right counters, out-links of (v,-) the left counters
(base appended comp(x)); an edge is a walk from a vertex through linear nodes to a vertex, kept iff its first (K+1)-mer
<= the reverse complement of its last; the linear nodes no kept edge visits form cycles.  Edges must equal the
device's exactly (sequence, length, flags, count_sum, link); cycles are compared in canonical rotation and strand."""
import numpy as np
import pytest

from conftest import make_dataset
from test_gpu_parity import run_gpu

pytestmark = pytest.mark.gpu

KEY_CASES = [(25, 1), (31, 1), (33, 2), (63, 2), (63, 4), (127, 4)]
COMP = str.maketrans("0123", "2301")
HEX2 = {f"{i:x}": f"{i >> 2}{i & 3}" for i in range(16)}
LINEAR, DELETED = 1 << 24, 1 << 25


def rc(s: str) -> str:
    return s[::-1].translate(COMP)


def canon(s: str):
    r = rc(s)
    return (s, 0) if s < r else (r, 1)


def key_str(k, K: int) -> str:
    v = (int(k[0]) << 192) | (int(k[1]) << 128) | (int(k[2]) << 64) | int(k[3])
    return "".join(HEX2[c] for c in format(v, "064x"))[-K:]


def model_table(ref, K):
    rec = ref.records
    return {key_str(k, K): (int(c), int(l) & 0xFFFFFF, int(r)) for k, c, l, r in
            zip(rec["key"], rec["count"], rec["l_links"], rec["rword"])}


def out_links(t, s: str, o: int):
    """(counter value, appended base) of every out-link of (s, o)"""
    L, rw = t[s][1], t[s][2]
    w = (rw & 0xFFFFFF) if o == 0 else L
    return [((w >> (6 * x)) & 63, x if o == 0 else x ^ 2) for x in range(4) if (w >> (6 * x)) & 63]


def model_edges(t, K):
    """-> (edges as (sequence, m, flags, count_sum, link) sorted, cycles as (canonical circular word, m, flags,
    count_sum) sorted, counts dict)"""
    linear = {s for s, v in t.items() if v[2] & LINEAR}
    vertices = [s for s, v in t.items() if not v[2] & (LINEAR | DELETED)]
    edges, seen, dangling = [], set(), 0
    lin_edges = pal = bases = 0
    for v in vertices:
        for o in (0, 1):
            kk = rc(v) if o else v
            for link, y in out_links(t, v, o):
                seq, m, csum, visited = [kk, str(y)], 1, 0, []
                u, ou = canon(kk[1:] + str(y))
                while u in linear:
                    csum += t[u][0]
                    visited.append(u)
                    ok_ = rc(u) if ou else u
                    (_, z), = out_links(t, u, ou)
                    seq.append(str(z))
                    u, ou = canon(ok_[1:] + str(z))
                    m += 1
                if u not in t:
                    dangling += 1
                    continue
                s = "".join(seq)
                first, last = s[: K + 1], rc(s[-(K + 1):])
                if first <= last:
                    flags = 1 if first == last else 0
                    edges.append((s, m, flags, csum, link))
                    seen.update(visited)
                    pal += flags
                    bases += m + K
                    lin_edges += (m - 1) // 2 if flags else m - 1
    cycles, lin_cyc = [], 0
    for p in sorted(linear - seen):
        if p in seen:
            continue
        cu, co, m, csum, word, nodes, is_pal = p, 0, 0, 0, [], set(), False
        while True:
            cur = rc(cu) if co else cu
            word.append(cur[0])
            csum += t[cu][0]
            nodes.add(cu)
            m += 1
            (_, z), = out_links(t, cu, co)
            cu, co = canon(cur[1:] + str(z))
            if cu == p and co == 1:
                is_pal = True
            if cu == p and co == 0:
                break
        seen.update(nodes)
        w = "".join(word)
        cycles.append((canon_circular(w), m, 2 | (1 if is_pal else 0), csum))
        pal += is_pal
        bases += m + K - 1
        lin_cyc += m // 2 if is_pal else m
    counts = dict(edges=len(edges) + len(cycles), palindromes=pal, cycles=len(cycles), bases=bases,
                  vertices=len(vertices), linear_on_edges=lin_edges, linear_on_cycles=lin_cyc, dangling=dangling)
    return sorted(edges), sorted(cycles), counts


def canon_circular(w: str) -> str:
    r = rc(w)
    return min(min(w[i:] + w[:i] for i in range(len(w))), min(r[i:] + r[:i] for i in range(len(r))))


def device_edges(pkg, g, K):
    edges, seq = g.edges()
    got_e, got_c = [], []
    for i in range(len(edges)):
        e = edges[i]
        s = "".join(map(str, pkg.edge_codes(edges, seq, i, K)))
        assert int(e["seq"]) % 32 == 0 and int(e["unused"]) == 0
        if int(e["flags"]) & pkg.EDGE_CYCLE:
            m = int(e["length"])
            assert len(s) == m + K - 1 and s[m:] == s[: K - 1]
            got_c.append((canon_circular(s[:m]), m, int(e["flags"]), int(e["count_sum"])))
        else:
            assert not got_c, "cycles follow the edges"
            got_e.append((s, int(e["length"]), int(e["flags"]), int(e["count_sum"]), int(e["link"])))
    return sorted(got_e), sorted(got_c), edges, seq


def check_edges(pkg, g, ref, K, what=""):
    """the device's edges against the model of the oracle's table; -> the build's counts"""
    t = model_table(ref, K)
    want_e, want_c, want_n = model_edges(t, K)
    res = g.edges_build()
    got_e, got_c, _, _ = device_edges(pkg, g, K)
    assert res["dangling"] == 0, what
    assert len(got_e) == len(want_e), (what, len(got_e), len(want_e))
    for a, b in zip(got_e, want_e):
        assert a == b, (what, a, b)
    assert got_c == want_c, what
    assert {k: res[k] for k in want_n} == want_n, (what, res, want_n)
    return res


def reads_of(strings, width=None):
    """code strings (or lists) -> (reads uint8 [n, width], lens)"""
    width = width or max(len(s) for s in strings)
    reads = np.zeros((len(strings), width), dtype=np.uint8)
    lens = np.zeros(len(strings), dtype=np.uint32)
    for i, s in enumerate(strings):
        a = np.array([int(c) for c in s], dtype=np.uint8)
        reads[i, : len(a)] = a
        lens[i] = len(a)
    return reads, lens


def rand_codes(rng, n):
    return "".join(map(str, rng.integers(0, 4, n)))


def build_and_check(pkg, oracle, reads, lens, K, kw, d=0, sliced=False, n_kmer=False, what=""):
    ref = oracle.run_hashing(reads, lens, K, kw, 8, d, n_kmer=int(n_kmer))
    g, freq, st = run_gpu(pkg, reads, lens, K, kw, d=d, batches=2, hint=0, sliced=sliced, n_kmer=n_kmer)
    try:
        assert st.n_nodes == ref.nodes
        res = check_edges(pkg, g, ref, K, what)
        assert res["vertices"] == st.n_nodes - st.n_linear - st.n_removed
        assert res["linear_on_edges"] + res["linear_on_cycles"] == st.n_linear
        return res
    finally:
        g.close()


@pytest.mark.parametrize("sliced", [False, True])
@pytest.mark.parametrize("K,kw", KEY_CASES)
def test_edges_against_model(pkg, oracle, tiny_transcriptome, K, kw, sliced):
    L = 150 if K > 63 else 100
    reads, lens = make_dataset(pkg, tiny_transcriptome, 1500, L, 17 + K, ragged=30)
    for d in (0, 2):
        res = build_and_check(pkg, oracle, reads, lens, K, kw, d=d, sliced=sliced, what=f"K={K} kw={kw} d={d} sliced={sliced}")
        assert res["edges"] > 0


@pytest.mark.parametrize("K,kw", [(25, 1), (63, 2), (99, 4)])
def test_edges_n_kmer(pkg, oracle, tiny_transcriptome, K, kw):
    L = 150 if K > 63 else 100
    reads, lens = make_dataset(pkg, tiny_transcriptome, 1500, L, 3 + K, ragged=20, n_rate=0.002)
    for sliced in (False, True):
        build_and_check(pkg, oracle, reads, lens, K, kw, d=0, sliced=sliced, n_kmer=True, what=f"-n K={K}")


def hand_cases(K, rng):
    h = (K + 1) // 2
    u, w = rand_codes(rng, h), rand_codes(rng, h)
    circle = rand_codes(rng, 300)
    unit = rand_codes(rng, 40)
    snp = rand_codes(rng, 3 * K)
    alt = snp[: len(snp) // 2] + str((int(snp[len(snp) // 2]) + 1) % 4) + snp[len(snp) // 2 + 1:]
    return {
        "hairpin": [rand_codes(rng, 40) + u + rc(u)],
        "two_hairpins": [rc(u) + u + rand_codes(rng, 60) + w + rc(w)],
        "poly_a": ["0" * (K + 20)],
        "circle": [(circle * 2)[i: i + 2 * K + 10] for i in range(0, 300, 10)],
        "tandem": [rand_codes(rng, 30) + unit * 5 + rand_codes(rng, 30)],
        "snp": [snp, alt],
        "one_edge": [rand_codes(rng, K + 1)],
        "short": [rand_codes(rng, K), rand_codes(rng, K - 3)],
    }


@pytest.mark.parametrize("K,kw", [(25, 1), (33, 2), (127, 4)])
@pytest.mark.parametrize("case", ["hairpin", "two_hairpins", "poly_a", "circle", "tandem", "snp", "one_edge", "short"])
def test_edges_hand_made(pkg, oracle, K, kw, case):
    rng = np.random.default_rng(K * 1000 + len(case))
    strings = hand_cases(K, rng)[case]
    reads, lens = reads_of(strings, width=max(max(map(len, strings)), K + 8))
    for sliced in (False, True):
        res = build_and_check(pkg, oracle, reads, lens, K, kw, sliced=sliced, what=f"{case} K={K}")
        if case == "hairpin":
            assert res["edges"] == 1 and res["palindromes"] == 1 and res["cycles"] == 0
        elif case == "two_hairpins":
            assert res["edges"] == 1 and res["cycles"] == 1 and res["palindromes"] == 1
        elif case == "poly_a":
            assert res["cycles"] == 1 and res["edges"] == 1 and res["bases"] == K
        elif case == "circle":
            assert res["cycles"] == 1 and res["edges"] == 1 and res["linear_on_cycles"] == 300
        elif case == "one_edge":
            assert res["edges"] == 1 and res["bases"] == K + 1 and res["vertices"] == 2
        elif case == "short":
            assert res == dict(res, edges=0, vertices=0, bases=0)


def test_edges_everything_deleted(pkg, oracle):
    rng = np.random.default_rng(5)
    reads, lens = reads_of([rand_codes(rng, 100) for _ in range(20)])
    res = build_and_check(pkg, oracle, reads, lens, 25, 1, d=2, what="deleted")
    assert res["edges"] == 0 and res["vertices"] == 0


def test_edges_hot_kmers(pkg, oracle):
    tr = pkg.synth.make_transcriptome(30, 21, hot=3)
    reads, lens = make_dataset(pkg, tr, 3000, 100, 9)
    for sliced in (False, True):
        res = build_and_check(pkg, oracle, reads, lens, 31, 1, d=2, sliced=sliced, what="hot")
        assert res["edges"] > 0


def test_edges_same_for_both_insert_paths_and_rebuild(pkg, tiny_transcriptome):
    reads, lens = make_dataset(pkg, tiny_transcriptome, 3000, 100, 77, ragged=20)
    out = []
    for sliced in (False, True):
        g, _, _ = run_gpu(pkg, reads, lens, 31, 1, d=1, batches=3, sliced=sliced)
        try:
            r1 = g.edges_build()
            e1, s1 = g.edges()
            r2 = g.edges_build()
            e2, s2 = g.edges()
            assert {k: v for k, v in r1.items() if k != "ms"} == {k: v for k, v in r2.items() if k != "ms"}
            assert e1.tobytes() == e2.tobytes() and s1.tobytes() == s2.tobytes()
            out.append(device_edges(pkg, g, 31)[:2])
        finally:
            g.close()
    assert out[0] == out[1]


def test_edges_reset_state_and_sharding(pkg, oracle, tiny_transcriptome):
    reads, lens = make_dataset(pkg, tiny_transcriptome, 800, 100, 12)
    stride = pkg.synth.stride_bytes(100)
    packed = pkg.synth.pack_reads(reads, lens, stride)
    g = pkg.PregraphGPU(25, 1, 100)
    try:
        with pytest.raises(pkg.SdtGpuError) as e:
            g.edges_build()
        assert e.value.code == 5                       # ESTATE before finalize
        g.push_reads(packed[:800], lens[:800], None, n_reads=800, stride_bytes=stride)
        g.finalize(0)
        g.edges_build()
        g.reset()
        with pytest.raises(pkg.SdtGpuError) as e:
            g.edges()
        assert e.value.code == 5                       # the buffers went with reset
        g.push_reads(packed[800:], lens[800:], None, n_reads=len(reads) - 800, stride_bytes=stride)
        g.finalize(0)
        ref = oracle.run_hashing(reads[800:], lens[800:], 25, 1, 8, 0)
        check_edges(pkg, g, ref, 25, "after reset")
    finally:
        g.close()
    g = pkg.PregraphGPU(25, 1, 100)
    try:
        g.set_owner(0, 2)
        g.push_reads(packed, lens, None, n_reads=len(reads), stride_bytes=stride)
        g.finalize(0)
        with pytest.raises(pkg.SdtGpuError) as e:
            g.edges_build()
        assert e.value.code == 1
    finally:
        g.close()
    g = pkg.PregraphGPU(25, 1, 100, capacity_hint=100_000, sliced=True)
    try:
        g.skm_set_world(1, 2)
        with pytest.raises(pkg.SdtGpuError) as e:
            g.edges_build()
        assert e.value.code == 1
    finally:
        g.close()


def test_edges_c1_accounting_and_lookups(pkg):
    """C1-sized (no Python walk): the counts add up to the table's, and a sample of edges looked up k-mer by k-mer
    finds every k-mer, linear inside and not linear at the ends, with count_sum the sum of the inner counts."""
    import torch
    synth = pkg.synth
    cfg = synth.CONFIGS["C1"]
    K, L = cfg["K"], cfg["read_len"]
    tr = synth.make_transcriptome(cfg["n_transcripts"], cfg["seed"])
    reads, lens = synth.make_reads(tr, cfg["n_pairs"], L, cfg["seed"])
    stride = synth.stride_bytes(L)
    packed = torch.from_numpy(synth.pack_reads(reads, lens, stride)).cuda()
    g = pkg.PregraphGPU(K, cfg["key_words"], L, sliced=True)
    try:
        n = len(reads)
        for a in range(0, n, 1 << 18):
            b = min(a + (1 << 18), n)
            g.push_reads(packed[a:b], None, None, n_reads=b - a, uniform_len=L, stride_bytes=stride, first_read_ordinal=a, device=True)
        _, st = g.finalize(cfg["d"])
        res = g.edges_build()
        edges, seq = g.edges()
        assert res["dangling"] == 0 and len(edges) == res["edges"] > 0
        pal = (edges["flags"] & pkg.EDGE_PALINDROME) != 0
        cyc = (edges["flags"] & pkg.EDGE_CYCLE) != 0
        m = edges["length"].astype(np.int64)
        inner = np.where(cyc, m, m - 1)
        assert int(np.where(pal, inner // 2, inner).sum()) == st.n_linear
        assert res["linear_on_edges"] + res["linear_on_cycles"] == st.n_linear
        assert res["vertices"] == st.n_nodes - st.n_linear - st.n_removed
        assert res["bases"] == int((m + K - cyc).sum()) and res["cycles"] == int(cyc.sum())
        rng = np.random.default_rng(1)
        pick = rng.choice(np.nonzero(~cyc)[0], size=min(10_000, int((~cyc).sum())), replace=False)
        keys, owner = [], []
        for i in pick:
            s = pkg.edge_codes(edges, seq, int(i), K)
            v = 0
            for j, b in enumerate(s):
                v = ((v << 2) | int(b)) & ((1 << (2 * K)) - 1)
                if j >= K - 1:
                    keys.append([0, 0, 0, v])
                    owner.append(int(i))
        hits = g.lookup_kmers(np.array(keys, dtype=np.uint64))
        assert (hits["status"] & pkg.HIT_FOUND).all()
        owner = np.array(owner)
        starts = np.concatenate([[0], np.nonzero(np.diff(owner))[0] + 1])
        ends = np.concatenate([starts[1:], [len(owner)]])
        lin = (hits["rword"] & (1 << 24)) != 0
        for a, b in zip(starts, ends):
            i = owner[a]
            assert not lin[a] and not lin[b - 1], i
            assert lin[a + 1: b - 1].all(), i
            assert int(hits["count"][a + 1: b - 1].sum()) == int(edges["count_sum"][i]), i
    finally:
        g.close()
