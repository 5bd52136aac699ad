"""Edge build on one GPU: a config's table compacted into edges between junction k-mers (sdtgpu_edges_build).

  python tools/edges_bench.py [--config C2] [--pairs P] [--device 0] [--repeats 3]

C2 as bench.py defines it (K = 31, 5 x 10^7 reads of 100 bp, generated on the device).  The sliced build without a
capacity hint and finalize(d) make the table; one edges_build is a warm-up (module load, the lookup index, the first
allocation of the edge buffers), then --repeats builds are timed by the library's CUDA events (the ms it reports) and
by a host clock around each call (which includes its host waits for the sizes).  Memory added: device memory in use
after the builds minus before the first, as cudaMemGetInfo reports it (lookup index included).

Accounting checks on the result (the definition of include/sdtgpu.h): no dangling link; the linear nodes on edges and
cycles add up to the table's linear nodes; vertices = nodes - linear - deleted; two builds give the same counts.
Prints one JSON line with the card's name and power limit as NVML reports them (read only; nothing is changed)."""
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
    del d_packed
    torch.cuda.empty_cache()
    torch.cuda.synchronize()
    free0, total = torch.cuda.mem_get_info(dev)

    warm = g.edges_build()
    runs, walls = [], []
    for _ in range(args.repeats):
        t0 = time.perf_counter()
        r = g.edges_build()
        walls.append((time.perf_counter() - t0) * 1e3)
        runs.append(r)
    free1, _ = torch.cuda.mem_get_info(dev)
    counts = {k: v for k, v in runs[-1].items() if k != "ms"}
    checks = dict(
        no_dangling=counts["dangling"] == 0,
        linear_adds_up=counts["linear_on_edges"] + counts["linear_on_cycles"] == st.n_linear,
        vertices_add_up=counts["vertices"] == st.n_nodes - st.n_linear - st.n_removed,
        repeatable=all({k: v for k, v in x.items() if k != "ms"} == counts for x in runs + [warm]),
    )
    ms = [x["ms"] for x in runs]
    res = dict(config=args.config, K=K, reads=n, nodes=int(st.n_nodes), linear=int(st.n_linear),
               deleted=int(st.n_removed), edges_ms=round(min(ms), 3), edges_ms_all=[round(x, 3) for x in ms],
               wall_ms=[round(x, 3) for x in walls], **counts,
               memory_added_bytes=int(free0 - free1), checks=checks, ok=all(checks.values()), **info)
    g.close()
    print(json.dumps(res))
    return 0 if res["ok"] else 1


if __name__ == "__main__":
    sys.exit(main())
