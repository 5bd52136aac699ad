"""FASTA pair on disk -> table counters, two ways, on one GPU:
  (a) host   sdtpack_next (all cores) -> pinned batches -> sdtgpu_push_reads            (bench.py's e2e_from_files)
  (b) device sdtgpu_reader_next (text chunks to the GPU, parsed and packed there) -> sdtgpu_push_reads_device
Both end with sdtgpu_get_stats on a sliced-build handle without a capacity hint.  The library is C2-shaped
(K = 31, 100 bp, synthetic reads of synth.CONFIGS["C2"], --pairs pairs, default all 25 M) and written to a
temporary directory first; one untimed read of both files warms the page cache, then the paths run alternately
--repeats times each.  Asserts equal n_instances, n_nodes and sdtgpu_table_checksum, prints one JSON line.

    python tools/parse_bench.py [--pairs N] [--batch-reads N] [--chunk-bytes N] [--repeats N]
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        name, power = [x.strip() for x in q.split(",")]
        return name, power
    except Exception as e:  # noqa: BLE001
        return f"unknown ({e})", "unknown"


def write_library(pkg, torch, cfg, n_pairs, d, piece=1 << 20):
    """f_1.fa / f_2.fa: the layout of bench.py's write_fasta_pair (">f" + 10-digit number, one sequence line),
    generated on the device piece by piece."""
    synth, dev = pkg.synth, torch.device("cuda", 0)
    L = cfg["read_len"]
    stride = synth.stride_bytes(L)
    tr = synth.make_transcriptome(cfg["n_transcripts"], cfg["seed"], hot=cfg["hot"])
    tr_dev = dict(bases=torch.from_numpy(tr.bases).to(dev), starts=torch.from_numpy(tr.starts.astype(np.int64)).to(dev),
                  lengths=torch.from_numpy(tr.lengths.astype(np.int32)).to(dev),
                  cum=torch.from_numpy(tr.cum.astype(np.int64)).to(dev), n=len(tr.lengths))
    lut = torch.tensor(list(b"ACTG"), dtype=torch.uint8, device=dev)
    shifts = torch.tensor([6, 4, 2, 0], dtype=torch.uint8, device=dev)
    paths = [os.path.join(d, "f_1.fa"), os.path.join(d, "f_2.fa")]
    files = [open(p, "wb") for p in paths]
    hdr = 13
    total = 0
    for a in range(0, n_pairs, piece):
        n = min(piece, n_pairs - a)
        packed = torch.empty((2 * n, stride), dtype=torch.uint8, device=dev)
        pkg.pregraph.synth_reads_device(tr_dev, cfg["seed"], a, n, L, stride, packed)
        codes = ((packed[:, :, None] >> shifts) & 3).reshape(2 * n, 4 * stride)[:, :L].long()
        for mate in (0, 1):
            rows = torch.empty((n, hdr + L + 1), dtype=torch.uint8, device=dev)
            rows[:, 0], rows[:, 1], rows[:, 12], rows[:, -1] = ord(">"), ord("f"), 10, 10
            idx = torch.arange(a, a + n, dtype=torch.int64, device=dev)
            for k in range(10):
                rows[:, 11 - k] = (48 + (idx // 10 ** k) % 10).to(torch.uint8)
            rows[:, hdr:hdr + L] = lut[codes[mate::2]]
            buf = rows.cpu().numpy()
            buf.tofile(files[mate])
            total += buf.size
    for f in files:
        f.close()
    return paths, total


def path_host(pkg, paths, cfg, batch):
    lib = pkg.library()
    L = cfg["read_len"]
    stride = pkg.synth.stride_bytes(L)
    bufs = []
    for _ in range(2):
        p, ln = C.c_void_p(), C.c_void_p()
        assert lib.sdtgpu_host_alloc(C.byref(p), batch * stride) == 0 and lib.sdtgpu_host_alloc(C.byref(ln), batch * 4) == 0
        bufs.append((p, ln))
    try:
        with pkg.PregraphGPU(cfg["K"], cfg["key_words"], L, capacity_hint=0, device=0, sliced=True) as g:
            t0 = time.perf_counter()
            rd = pkg.ReadPacker(paths[0], paths[1], fastq=False)
            pushed, cur = 0, 0
            while True:
                p, ln = bufs[cur]
                n = lib.sdtpack_next(rd.h, L, 0, 0, p, ln, None, batch, stride)
                assert n >= 0
                if n == 0:
                    break
                g._ck(lib.sdtgpu_push_reads(g.h, p, ln, None, n, 0, stride, pushed))
                pushed += n
                cur ^= 1
            rd.close()
            st = g.stats()
            dt = time.perf_counter() - t0
            return dt, pushed, st, g.table_checksum().tolist(), None
    finally:
        for p, ln in bufs:
            lib.sdtgpu_host_free(p)
            lib.sdtgpu_host_free(ln)


def path_device(pkg, torch, paths, cfg, batch, chunk):
    lib = pkg.library()
    L = cfg["read_len"]
    stride = pkg.synth.stride_bytes(L)
    dev = torch.device("cuda", 0)
    bufs = [(torch.empty((batch, stride), dtype=torch.uint8, device=dev), torch.empty(batch, dtype=torch.int32, device=dev))
            for _ in range(2)]
    torch.cuda.synchronize()
    with pkg.PregraphGPU(cfg["K"], cfg["key_words"], L, capacity_hint=0, device=0, sliced=True) as g:
        t0 = time.perf_counter()
        rd = pkg.DeviceReadPacker(paths[0], paths[1], fastq=False, device=0, chunk_bytes=chunk)
        pushed, cur, n = 0, 0, C.c_uint64()
        while True:
            p, ln = bufs[cur]
            # packs go on the handle's stream, so each push is ordered after the pack that feeds it
            rc = lib.sdtgpu_reader_next(rd.h, g.stream, L, 0, 0, p.data_ptr(), ln.data_ptr(), None, batch, stride, C.byref(n))
            assert rc == 0, lib.sdtgpu_reader_last_error(rd.h)
            if n.value == 0:
                break
            g._ck(lib.sdtgpu_push_reads_device(g.h, p.data_ptr(), ln.data_ptr(), None, n.value, 0, stride, pushed))
            pushed += n.value
            cur ^= 1
        st = g.stats()
        dt = time.perf_counter() - t0
        rstats = rd.stats()
        rd.close()
        return dt, pushed, st, g.table_checksum().tolist(), rstats


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--pairs", type=int, default=25_000_000)
    ap.add_argument("--batch-reads", type=int, default=1 << 22)
    ap.add_argument("--chunk-bytes", type=int, default=0, help="device reader upload size (0: its default)")
    ap.add_argument("--repeats", type=int, default=2)
    ap.add_argument("--out", default="", help="also write the JSON line to this file")
    args = ap.parse_args()
    import torch
    import sdt_pkg
    pkg = sdt_pkg.load()
    cfg = pkg.synth.CONFIGS["C2"]
    name, power = card()
    nwin = cfg["read_len"] - cfg["K"] + 1
    with tempfile.TemporaryDirectory() as d:
        t0 = time.perf_counter()
        paths, text_bytes = write_library(pkg, torch, cfg, args.pairs, d)
        t_write = time.perf_counter() - t0
        for p in paths:        # page cache
            with open(p, "rb") as f:
                while f.read(1 << 26):
                    pass
        runs = {"host": [], "device": []}
        res = {}
        for _ in range(args.repeats):
            for which in ("host", "device"):
                if which == "host":
                    dt, n, st, ck, rs = path_host(pkg, paths, cfg, args.batch_reads)
                else:
                    dt, n, st, ck, rs = path_device(pkg, torch, paths, cfg, args.batch_reads, args.chunk_bytes)
                runs[which].append(dt)
                res[which] = (n, int(st.n_instances), int(st.n_nodes), ck, rs)
    h, dv = res["host"], res["device"]
    assert h[0] == dv[0] == 2 * args.pairs, (h[0], dv[0])
    assert h[1] == dv[1] and h[2] == dv[2] and h[3] == dv[3], "the two paths built different tables"
    out = {"card": name, "power_limit": power, "pairs": args.pairs, "reads": h[0], "text_bytes": text_bytes,
           "n_instances": h[1], "n_nodes": h[2], "table_checksum": [str(x) for x in h[3]], "checksums_equal": True,
           "batch_reads": args.batch_reads, "write_s": round(t_write, 2)}
    assert h[1] == h[0] * nwin
    for which in ("host", "device"):
        s = min(runs[which])
        out[which] = {"seconds": round(s, 4), "all_seconds": [round(x, 4) for x in runs[which]],
                      "G_instances_per_s": round(h[1] / s / 1e9, 3), "M_reads_per_s": round(h[0] / s / 1e6, 2),
                      "text_GB_per_s": round(text_bytes / s / 1e9, 3)}
    out["device"]["reader_stats"] = dict(dv[4])
    out["host"]["what"] = "sdtpack_next (all cores) -> pinned -> sdtgpu_push_reads -> get_stats"
    out["device"]["what"] = "sdtgpu_reader_next -> sdtgpu_push_reads_device -> get_stats"
    line = json.dumps(out)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
