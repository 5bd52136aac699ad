"""Reads mapped onto the edge graph on one GPU (sdtgpu_edges_map_reads, sdtgpu_arcs_build).

  python tools/map_bench.py [--config C2] [--pairs P] [--device 0] [--repeats 3]

C2 as bench.py defines it (K = 31, 5 x 10^7 reads of 100 bp, generated on the device).  The sliced build without a
capacity hint, finalize(d) and edges_build make the graph.  Then, each timed by CUDA events on the handle's stream
(class 7 of sdtgpu_phase_times):
  stamps    the first map call after the build with no reads, which only stamps the graph;
  mapping   every read in batches of 2^22 into one reused step buffer, arcs counted; reported as windows/s, a window
            being one of the max_read_len - K + 1 positions of a read (the last one has no (K+1)-mer);
  arcs      arcs_build, --repeats times (the ms it reports).
Memory added: device memory in use after the arcs minus before the first map call, as cudaMemGetInfo reports it.

Checks on the result: at -d 0 every (K+1)-mer of every read maps and the last window of every read does not; the arc
counts add up to the vertex crossings counted independently from lookup_reads hits (a window 1 .. maxwin - 2 that is
found, neither linear nor deleted, with the counters of both its link bases non-zero); two arcs_build calls give
byte-identical buffers.  Prints one JSON line with the card's name and power limit as NVML reports them (read only;
nothing is changed)."""
import argparse
import ctypes as C
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

BATCH = 1 << 22
LINEAR, DELETED = 1 << 24, 1 << 25


def lookup_ms(g) -> float:
    """device ms of class 7 of sdtgpu_phase_times (lookups, stamps, mapping) since the last call"""
    ms = (C.c_double * 8)()
    g._ck(g.L.sdtgpu_phase_times(g.h, 1, ms, None))
    return ms[7]


def crossings(torch, pkg, packed, hits, K, L):
    """vertex crossings of a batch of uniform reads of length L, from their lookup hits"""
    pos = torch.arange(L, device=packed.device)
    codes = ((packed[:, pos // 4].long() >> (6 - 2 * (pos % 4))) & 3)
    w = torch.arange(1, L - K, device=packed.device)
    h = hits[:, 1:-1].long() & 0xFFFFFFFF
    lw, rword, status = h[..., 1] & 0xFFFFFF, h[..., 2], h[..., 3]
    rw = rword & 0xFFFFFF
    isrc = (status & pkg.HIT_RC) != 0
    prev, nxt = codes[:, w - 1], codes[:, w + K]
    left = torch.where(isrc, nxt ^ 2, prev)
    right = torch.where(isrc, prev ^ 2, nxt)
    vert = ((status & pkg.HIT_FOUND) != 0) & ((rword & (LINEAR | DELETED)) == 0)
    return int((vert & (((lw >> (6 * left)) & 63) > 0) & (((rw >> (6 * right)) & 63) > 0)).sum())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--config", default="C2")
    ap.add_argument("--pairs", type=int, default=0, help="read pairs (default: the config's)")
    ap.add_argument("--device", type=int, default=0)
    ap.add_argument("--repeats", type=int, default=3)
    args = ap.parse_args()
    import torch
    import sdt_pkg
    from lookup_bench import card
    pkg = sdt_pkg.load()
    synth = pkg.synth
    cfg = dict(synth.CONFIGS[args.config])
    K, kw, L = cfg["K"], cfg["key_words"], cfg["read_len"]
    n_pairs = args.pairs or cfg["n_pairs"]
    dev = torch.device("cuda", args.device)
    torch.cuda.set_device(dev)
    info = card(args.device)

    tr = synth.make_transcriptome(cfg["n_transcripts"], cfg["seed"], hot=cfg["hot"])
    tr_dev = dict(bases=torch.from_numpy(tr.bases).to(dev), starts=torch.from_numpy(tr.starts.astype(np.int64)).to(dev),
                  lengths=torch.from_numpy(tr.lengths.astype(np.int32)).to(dev),
                  cum=torch.from_numpy(tr.cum.astype(np.int64)).to(dev), n=len(tr.lengths))
    stride = synth.stride_bytes(L)
    n = 2 * n_pairs
    d_packed = torch.empty((n, stride), dtype=torch.uint8, device=dev)
    pkg.pregraph.synth_reads_device(tr_dev, cfg["seed"], 0, n_pairs, L, stride, d_packed, device=args.device)
    torch.cuda.synchronize()

    g = pkg.PregraphGPU(K, kw, L, capacity_hint=0, device=args.device, sliced=True)
    for a in range(0, n, BATCH):
        b = min(a + BATCH, n)
        g.push_reads(d_packed[a:b], None, None, n_reads=b - a, uniform_len=L, stride_bytes=stride, first_read_ordinal=a, device=True)
    freq, st = g.finalize(cfg["d"])
    ed = g.edges_build()
    maxwin = L - K + 1
    out = torch.empty((BATCH, maxwin, 2), dtype=torch.int32, device=dev)
    torch.cuda.synchronize()
    free0, _ = torch.cuda.mem_get_info(dev)

    lookup_ms(g)
    g.map_reads(d_packed[:0], None, None, n_reads=0, uniform_len=L, stride_bytes=stride, out=out)
    stamp_ms = lookup_ms(g)

    t0 = time.perf_counter()
    for a in range(0, n, BATCH):
        b = min(a + BATCH, n)
        g.map_reads(d_packed[a:b], None, None, n_reads=b - a, uniform_len=L, stride_bytes=stride, out=out)
    map_wall = time.perf_counter() - t0
    map_ms = lookup_ms(g)
    windows = n * maxwin

    runs = [g.arcs_build() for _ in range(args.repeats)]
    a1 = g.arcs().tobytes()
    g.arcs_build()
    a2 = g.arcs()
    free1, _ = torch.cuda.mem_get_info(dev)

    # checks: every (K+1)-mer maps (at -d 0), and the crossings counted from the hits
    all_map, want_cross = True, 0
    for a in range(0, n, BATCH):
        b = min(a + BATCH, n)
        s = g.map_reads(d_packed[a:b], None, None, n_reads=b - a, uniform_len=L, stride_bytes=stride, count_arcs=False, out=out)[: b - a]
        none = s[..., 0] == -1
        all_map &= bool((~none[:, :-1]).all()) and bool(none[:, -1].all())
        hits = g.lookup_reads(d_packed[a:b], None, None, n_reads=b - a, uniform_len=L, stride_bytes=stride)
        want_cross += crossings(torch, pkg, d_packed[a:b], hits, K, L)
        del hits
    res_arcs = runs[-1]
    checks = dict(
        every_step_maps=all_map if cfg["d"] == 0 else None,
        arcs_equal_crossings=res_arcs["crossings"] == want_cross,
        arcs_sum=int(a2["count"].sum()) == res_arcs["crossings"],
        arcs_repeatable=a1 == a2.tobytes() and all({k: v for k, v in r.items() if k != "ms"} == {k: v for k, v in res_arcs.items() if k != "ms"} for r in runs),
    )
    arcs_ms = [r["ms"] for r in runs]
    res = dict(config=args.config, K=K, reads=n, nodes=int(st.n_nodes), records=ed["edges"], vertices=ed["vertices"],
               stamp_ms=round(stamp_ms, 3), map_ms=round(map_ms, 3), map_wall_ms=round(map_wall * 1e3, 3),
               windows=windows, windows_per_s=round(windows / (map_ms * 1e-3), 1),
               arcs=res_arcs["arcs"], crossings=res_arcs["crossings"], arcs_ms=round(min(arcs_ms), 3),
               arcs_ms_all=[round(x, 3) for x in arcs_ms], memory_added_bytes=int(free0 - free1),
               checks=checks, ok=all(v is not False for v in checks.values()), **info)
    g.close()
    print(json.dumps(res))
    return 0 if res["ok"] else 1


if __name__ == "__main__":
    sys.exit(main())
