"""One FASTA pair read by N GPUs together, each rank parsing only its own byte range, into the multi-GPU build.

  python tools/shard_read_bench.py [--gpus N] [--pairs P] [--batch-reads 4194304] [--chunk-bytes 0]

Writes a C2-shaped pair (tools/parse_bench.write_library: ">f" + 10-digit number, one sequence line) to a temporary
directory and reads it once, untimed, to warm the page cache.  Then N processes, one per GPU (spawned and joined as in
tools/lookup_exchange_bench.py); every rank:
  1. open_shard + summary (a device pass over its byte range), then plan over torch.distributed
     (exchange.plan_reader: an all-gather of the 256-byte summaries, then host arithmetic);
  2. sdtgpu_reader_next in a loop on the handle's stream, each batch into sdtgpu_push_reads_device of a sliced handle
     set up with skm_set_world, its first ordinal from sdtgpu_reader_tell; the capacity hint is the same on every rank,
     from the plan's records of the library x (L - K + 1) in bench.py's closed form;
  3. sdtgpu_skm_exchange (the super-k-mer exchange inside the library), then sync.
Each phase is timed on the host clock and ends in a device synchronise.  Then, in the same invocation, one GPU builds
the same files with a plain reader; the ranks' node counts and table checksums (sdtgpu_table_checksum, summed over the
ranks) must equal it.

Prints one JSON line: seconds per phase (the slowest rank), text bytes uploaded and records returned per rank, the
node count and checksum check, and the card's name and power limit (nvidia-smi, read only)."""
import argparse
import ctypes as C
import json
import os
import socket
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _hint(records, K, L):
    inst = records * (L - K + 1)
    return int(min(inst + 1024.0, inst * (1.0 - 0.99 ** K) * 1.05 + 65536.0))      # bench.py's rule on several GPUs


def _worker(rank, world, port, args, paths, out_dir):
    sys.path.insert(0, ROOT)
    import torch
    import torch.distributed as dist
    import sdt_pkg
    pkg = sdt_pkg.load()
    from soapdenovo_trans_b200.exchange import SkmExchange, plan_reader
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    lib = pkg.library()
    cfg = pkg.synth.CONFIGS["C2"]
    K, kw, L = cfg["K"], cfg["key_words"], cfg["read_len"]
    stride = pkg.synth.stride_bytes(L)
    batch = args.batch_reads
    bufs = [(torch.empty((batch, stride), dtype=torch.uint8, device=dev), torch.empty(batch, dtype=torch.int32, device=dev))
            for _ in range(2)]
    torch.cuda.synchronize()
    dist.barrier()
    t = {}
    t0 = time.perf_counter()
    rd = pkg.DeviceReadPacker(paths[0], paths[1], device=rank, chunk_bytes=args.chunk_bytes, rank=rank, world=world)
    rd.summary()
    torch.cuda.synchronize()
    t["summary"] = time.perf_counter() - t0
    t0 = time.perf_counter()
    plan = plan_reader(rd, dev)
    torch.cuda.synchronize()
    t["plan"] = time.perf_counter() - t0
    g = pkg.PregraphGPU(K, kw, L, capacity_hint=_hint(plan["library_records"], K, L), device=rank, sliced=True)
    ex = SkmExchange(pkg, g, world, rank, dev, native=True)      # skm_set_world, and the library's communicator
    after_summary = rd.stats()["text_bytes"]
    g.sync()
    dist.barrier()
    t0 = time.perf_counter()
    cur, n, pushed, reads_end = 0, C.c_uint64(), 0, 0
    while True:
        first = rd.tell()
        p, ln = bufs[cur]
        # packs go on the handle's stream, so each push is ordered after the pack that feeds it
        rc = lib.sdtgpu_reader_next(rd.h, g.stream, L, 0, 0, p.data_ptr(), ln.data_ptr(), None, batch, stride, C.byref(n))
        assert rc == 0, lib.sdtgpu_reader_last_error(rd.h)
        if n.value == 0:
            break
        g._ck(lib.sdtgpu_push_reads_device(g.h, p.data_ptr(), ln.data_ptr(), None, n.value, 0, stride, first))
        pushed += n.value
        reads_end = first + n.value
        cur ^= 1
    g.sync()
    t["read_push"] = time.perf_counter() - t0
    dist.barrier()
    t0 = time.perf_counter()
    g.skm_exchange(ex.comm, reads_end)
    g.sync()
    t["exchange_build"] = time.perf_counter() - t0
    st = g.stats()
    ck = g.table_checksum()
    rs = rd.stats()
    mine = torch.tensor([t["summary"], t["plan"], t["read_push"], t["exchange_build"], rs["text_bytes"], after_summary,
                         pushed, plan["records"], st.n_nodes, st.n_instances, *[float(x) for x in ck[:3] % (1 << 40)],
                         *[float(x >> np.uint64(40)) for x in ck[:3]]], dtype=torch.float64, device=dev)
    allv = torch.empty((world, mine.numel()), dtype=torch.float64, device=dev)
    dist.all_gather_into_tensor(allv.view(-1), mine)
    if rank == 0:
        np.save(os.path.join(out_dir, "ranks.npy"), allv.cpu().numpy())
        with open(os.path.join(out_dir, "plan.json"), "w") as f:
            json.dump(plan, f)
    rd.close()
    g.close()
    ex.comm.close()
    dist.barrier()
    dist.destroy_process_group()


def one_gpu(pkg, torch, paths, batch, records):
    """The same files through a plain reader on one GPU: node count and table checksum."""
    lib = pkg.library()
    cfg = pkg.synth.CONFIGS["C2"]
    K, kw, L = cfg["K"], cfg["key_words"], cfg["read_len"]
    stride = pkg.synth.stride_bytes(L)
    dev = torch.device("cuda", 0)
    p, ln = torch.empty((batch, stride), dtype=torch.uint8, device=dev), torch.empty(batch, dtype=torch.int32, device=dev)
    with pkg.PregraphGPU(K, kw, L, capacity_hint=_hint(records, K, L), device=0, sliced=True) as g, \
            pkg.DeviceReadPacker(paths[0], paths[1], device=0) as rd:
        n, pushed = C.c_uint64(), 0
        while True:
            rc = lib.sdtgpu_reader_next(rd.h, g.stream, L, 0, 0, p.data_ptr(), ln.data_ptr(), None, batch, stride, C.byref(n))
            assert rc == 0, lib.sdtgpu_reader_last_error(rd.h)
            if n.value == 0:
                break
            g._ck(lib.sdtgpu_push_reads_device(g.h, p.data_ptr(), ln.data_ptr(), None, n.value, 0, stride, pushed))
            pushed += n.value
        st = g.stats()
        return pushed, int(st.n_nodes), [int(x) for x in g.table_checksum()]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=0, help="processes, one per GPU (default: every visible GPU)")
    ap.add_argument("--pairs", type=int, default=25_000_000, help="read pairs of the library (default: all of C2)")
    ap.add_argument("--batch-reads", type=int, default=1 << 22)
    ap.add_argument("--chunk-bytes", type=int, default=0, help="reader upload size (0: its default)")
    args = ap.parse_args()
    import torch
    import torch.multiprocessing as mp
    import sdt_pkg
    from tools.parse_bench import card, write_library
    world = args.gpus or torch.cuda.device_count()
    if world < 1 or world > torch.cuda.device_count():
        sys.exit(f"shard_read_bench: {world} GPUs asked, {torch.cuda.device_count()} visible")
    pkg = sdt_pkg.load()
    name, power = card()
    with tempfile.TemporaryDirectory() as d:
        paths, text_bytes = write_library(pkg, torch, pkg.synth.CONFIGS["C2"], args.pairs, d)
        torch.cuda.empty_cache()
        for p in paths:        # page cache
            with open(p, "rb") as f:
                while f.read(1 << 26):
                    pass
        mp.spawn(_worker, args=(world, _free_port(), args, paths, d), nprocs=world, join=True)
        v = np.load(os.path.join(d, "ranks.npy"))
        with open(os.path.join(d, "plan.json")) as f:
            plan = json.load(f)
        ref_reads, ref_nodes, ref_ck = one_gpu(pkg, torch, paths, args.batch_reads, plan["library_records"])
    ck = [(sum(int(x) for x in v[:, 10 + i]) + (sum(int(x) for x in v[:, 13 + i]) << 40)) % (1 << 64) for i in range(3)]
    nodes = int(v[:, 8].sum())
    ok = nodes == ref_nodes and ck == [x % (1 << 64) for x in ref_ck[:3]] and int(v[:, 6].sum()) == ref_reads
    phases = ("summary", "plan", "read_push", "exchange_build")
    out = {"card": name, "power_limit": power, "gpus": world, "pairs": args.pairs, "text_bytes": text_bytes,
           "chunk_bytes": args.chunk_bytes, "batch_reads": args.batch_reads,
           "seconds": {k: round(float(v[:, i].max()), 4) for i, k in enumerate(phases)},
           "seconds_per_rank": {k: [round(float(x), 4) for x in v[:, i]] for i, k in enumerate(phases)},
           "text_bytes_per_rank": [int(x) for x in v[:, 4]], "summary_text_bytes_per_rank": [int(x) for x in v[:, 5]],
           "records_per_rank": [int(x) for x in v[:, 6]], "library_records": plan["library_records"],
           "n_instances": int(v[:, 9].sum()), "n_nodes": nodes, "one_gpu_n_nodes": ref_nodes,
           "table_checksum": [str(x) for x in ck], "one_gpu_table_checksum": [str(x) for x in ref_ck[:3]],
           "table_check": "pass" if ok else "FAIL"}
    print(json.dumps(out))
    if not ok:
        sys.exit("shard_read_bench: the sharded build differs from the one-GPU build")


if __name__ == "__main__":
    main()
