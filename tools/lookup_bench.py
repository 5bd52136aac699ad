"""Lookup rate on one GPU: every window of a config's reads looked up in the table those reads built.

  python tools/lookup_bench.py [--config C2] [--pairs P] [--device 0]

C2 as bench.py defines it (K = 31, 5 x 10^7 reads of 100 bp, generated on the device).  The sliced build without a
capacity hint and finalize(0) make the table; the first lookup of one key builds the index (its time: that call
minus a second call of one key, CUDA events on the handle's stream); then sdtgpu_lookup_reads_device runs over
all reads in batches of 2^22 reads into one reused output buffer, each call between CUDA events on the handle's
stream.  Every window was inserted, so the found fraction must be exactly 1.  Prints one JSON line with the card's
name and power limit as NVML reports them (read only; nothing is changed).

The ceiling quoted beside the rate: a hit costs about two cold-line requests (index entry, then the slot), and a
B200 completes 36.65 G such requests/s (DESIGN.md §4.1)."""
import argparse
import ctypes as C
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

REQUESTS_PER_S = 36.65e9
BATCH = 1 << 22


def card(index: int) -> dict:
    import pynvml
    import torch
    pynvml.nvmlInit()
    pr = torch.cuda.get_device_properties(index)
    try:
        h = pynvml.nvmlDeviceGetHandleByPciBusId(f"{getattr(pr, 'pci_domain_id', 0):08X}:{pr.pci_bus_id:02X}:{pr.pci_device_id:02X}.0".encode())
    except Exception:
        h = pynvml.nvmlDeviceGetHandleByIndex(index)
    name = pynvml.nvmlDeviceGetName(h)
    return {"gpu": name.decode() if isinstance(name, bytes) else name,
            "power_limit_w": pynvml.nvmlDeviceGetEnforcedPowerLimit(h) / 1000.0}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--config", default="C2")
    ap.add_argument("--pairs", type=int, default=0, help="read pairs (default: the config's)")
    ap.add_argument("--device", type=int, default=0)
    args = ap.parse_args()
    import torch
    import sdt_pkg
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
    nodes = int(st.n_nodes)

    lib, h = g.L, g.h
    s = torch.cuda.ExternalStream(g.stream, device=dev)
    ms = (C.c_double * 8)()
    nl = (C.c_uint64 * 8)()
    g._ck(lib.sdtgpu_phase_times(h, 1, ms, nl))

    def timed(fn):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(s)
        g._ck(fn())
        e1.record(s)
        e1.synchronize()
        return e0.elapsed_time(e1)

    key = torch.zeros((1, 4), dtype=torch.int64, device=dev)
    hit = torch.zeros((1, 4), dtype=torch.int32, device=dev)
    torch.cuda.synchronize()
    first = timed(lambda: lib.sdtgpu_lookup_kmers_device(h, key.data_ptr(), 1, hit.data_ptr()))
    second = timed(lambda: lib.sdtgpu_lookup_kmers_device(h, key.data_ptr(), 1, hit.data_ptr()))
    g._ck(lib.sdtgpu_phase_times(h, 1, ms, nl))
    index_device_ms = ms[7]      # memset + index_build_kernel + the two one-key lookups

    maxwin = L - K + 1
    out = torch.empty((min(BATCH, n), maxwin, 4), dtype=torch.int32, device=dev)
    torch.cuda.synchronize()

    def lookup(a, b):
        return lambda: lib.sdtgpu_lookup_reads_device(h, d_packed[a:b].data_ptr(), None, None, b - a, L, stride, out.data_ptr())

    timed(lookup(0, min(BATCH, n)))          # warm-up: module load of the kernel
    total_ms, found, windows = 0.0, 0, 0
    for a in range(0, n, BATCH):
        b = min(a + BATCH, n)
        total_ms += timed(lookup(a, b))
        found += int(((out[: b - a, :, 3] & pkg.HIT_FOUND) != 0).sum())
        windows += (b - a) * maxwin
    rate = windows / (total_ms * 1e-3)
    ceiling = REQUESTS_PER_S / 2
    res = dict(config=args.config, K=K, reads=n, windows=windows, nodes=nodes, batch_reads=BATCH,
               lookup_ms=round(total_ms, 3), windows_per_s=rate, ceiling_windows_per_s=ceiling,
               fraction_of_ceiling=round(rate / ceiling, 4), found_fraction=found / windows,
               index_build_ms=round(first - second, 3), index_build_device_ms=round(index_device_ms, 3),
               index_bytes=max(1024, 2 * nodes) * 8, **info)
    g.close()
    print(json.dumps(res))
    if found != windows:
        sys.exit(f"lookup_bench: {windows - found} of {windows} windows not found")


if __name__ == "__main__":
    main()
