"""Pruning on one GPU: a config's table pruned of minor branches and tips (sdtgpu_prune) with the reference's defaults.

  python tools/prune_bench.py [--config C2] [--pairs P] [--device 0] [--repeats 2]

The config as bench.py defines it (reads generated on the device).  Each repeat builds the table afresh (sliced build
without a capacity hint, finalize(d)), because a table is pruned once; runs edges_build once for the counts before;
prunes with -i 5, single tips when d = 0 and minor tips (as call_pregraph does), timed by the library's CUDA events
(the ms it reports) and by a host clock around the call (which includes its host reads between rounds); and runs
edges_build again for the counts after.  The first edges_build also builds the lookup index, so the prune does not.

Checks: no dangling link after the prune; live = nodes - deleted by finalize - removed by the prune (the configs' reads
have no N, so at d = 0 every node has a counter); vertices after = live - linear, as the edge build counts them; the
linear nodes on edges and cycles add up to the prune's linear count; the repeats agree on every count and on
table_checksum.  Prints one JSON line with the card's name and power limit as NVML reports them (read only)."""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

BATCH = 1 << 22


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--config", default="C2")
    ap.add_argument("--pairs", type=int, default=0, help="read pairs (default: the config's)")
    ap.add_argument("--device", type=int, default=0)
    ap.add_argument("--repeats", type=int, default=2)
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
    runs = []
    for _ in range(args.repeats):
        d_packed = torch.empty((n, stride), dtype=torch.uint8, device=dev)
        pkg.pregraph.synth_reads_device(tr_dev, cfg["seed"], 0, n_pairs, L, stride, d_packed, device=args.device)
        torch.cuda.synchronize()
        g = pkg.PregraphGPU(K, kw, L, capacity_hint=0, device=args.device, sliced=True)
        try:
            for a in range(0, n, BATCH):
                b = min(a + BATCH, n)
                g.push_reads(d_packed[a:b], None, None, n_reads=b - a, uniform_len=L, stride_bytes=stride, first_read_ordinal=a, device=True)
            _, st = g.finalize(cfg["d"])
            del d_packed
            torch.cuda.empty_cache()
            before = g.edges_build()
            t0 = time.perf_counter()
            res = g.prune()
            wall = (time.perf_counter() - t0) * 1e3
            after = g.edges_build()
            runs.append(dict(st=st, before=before, res=res, wall=wall, after=after, checksum=g.table_checksum().tolist()))
        finally:
            g.close()
        torch.cuda.empty_cache()
    r = runs[-1]
    st, res, after = r["st"], r["res"], r["after"]
    counts = {k: v for k, v in res.items() if k != "ms"}
    removed = res["minor_branches"] + res["single_tips"] + res["minor_tips"]
    strip = lambda x: {k: v for k, v in x.items() if k != "ms"}  # noqa: E731
    checks = dict(
        no_dangling=after["dangling"] == 0,
        live_adds_up=res["live"] == st.n_nodes - st.n_removed - removed,
        vertices_add_up=after["vertices"] == res["vertices"] == res["live"] - res["linear"],
        linear_adds_up=after["linear_on_edges"] + after["linear_on_cycles"] == res["linear"],
        repeatable=all(strip(x["res"]) == counts and x["checksum"] == r["checksum"] and strip(x["after"]) == strip(after)
                       for x in runs),
    )
    ms = [x["res"]["ms"] for x in runs]
    out = dict(config=args.config, K=K, d=cfg["d"], reads=n, nodes=int(st.n_nodes), deleted_by_finalize=int(st.n_removed),
               prune_ms=round(min(ms), 3), prune_ms_all=[round(x, 3) for x in ms],
               wall_ms=[round(x["wall"], 3) for x in runs], **counts,
               edges_before=r["before"]["edges"], vertices_before=r["before"]["vertices"], edges_after=after["edges"],
               vertices_after=after["vertices"], checks=checks, ok=all(checks.values()), **info)
    print(json.dumps(out))
    return 0 if out["ok"] else 1


if __name__ == "__main__":
    sys.exit(main())
