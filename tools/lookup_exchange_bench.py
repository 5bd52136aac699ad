"""Routed lookup rate on N GPUs: every rank looks up every window of its own reads in the table all ranks built.

  python tools/lookup_exchange_bench.py [--gpus N] [--config C2] [--pairs P] [--batch-reads 1048576]

N processes, one per GPU.  Each generates its share of the config's reads on the device (the config's pairs PER GPU,
as bench.py does on several GPUs), builds its share of the table with the sliced build and the super-k-mer exchange
inside the library (SkmExchange(native=True)) and finalizes.  Then every rank routes every window of its own reads
through sdtgpu_lookup_reads_exchange in batches of --batch-reads reads into one reused output, after one untimed
batch.  Every window was inserted on some rank, so the found fraction must be exactly 1.

Rank 0 prints one JSON line: windows per second per rank and in total (wall clock of the batches, each call returns
when its hits are in the output), the device ms of stage + answer + unstage (class 7 of sdtgpu_phase_times, summed
over ranks) and of the collectives (collective_ms: the counts all-gather and the two grouped send / recv), bytes moved
between ranks per window, and the card's name and power limit as NVML reports them (read only).  Compare with the
one-GPU rate of tools/lookup_bench.py."""
import argparse
import ctypes as C
import json
import os
import socket
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _worker(rank, world, port, args, out_dir):
    sys.path.insert(0, ROOT)
    import torch
    import torch.distributed as dist
    import sdt_pkg
    from tools.lookup_bench import card
    pkg = sdt_pkg.load()
    from soapdenovo_trans_b200.exchange import SkmExchange
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    synth = pkg.synth
    cfg = dict(synth.CONFIGS[args.config])
    K, kw, L = cfg["K"], cfg["key_words"], cfg["read_len"]
    n_pairs = args.pairs or cfg["n_pairs"]
    n = 2 * n_pairs
    stride = synth.stride_bytes(L)
    tr = synth.make_transcriptome(cfg["n_transcripts"], cfg["seed"], hot=cfg["hot"])
    tr_dev = dict(bases=torch.from_numpy(tr.bases).to(dev), starts=torch.from_numpy(tr.starts.astype(np.int64)).to(dev),
                  lengths=torch.from_numpy(tr.lengths.astype(np.int32)).to(dev),
                  cum=torch.from_numpy(tr.cum.astype(np.int64)).to(dev), n=len(tr.lengths))
    d_packed = torch.empty((n, stride), dtype=torch.uint8, device=dev)
    pkg.pregraph.synth_reads_device(tr_dev, cfg["seed"], rank * n_pairs, n_pairs, L, stride, d_packed, device=rank)
    torch.cuda.synchronize()
    maxwin = L - K + 1
    instances = n * maxwin
    hint = int(min(instances + 1024.0, instances * (1.0 - 0.99 ** K) * 1.05 + 65536.0))      # bench.py's rule on several GPUs
    g = pkg.PregraphGPU(K, kw, L, capacity_hint=hint, device=rank, sliced=True)
    ex = SkmExchange(pkg, g, world, rank, dev, native=True)
    for a in range(0, n, 1 << 22):
        b = min(a + (1 << 22), n)
        ex.round(g, d_packed[a:b], b - a, L, stride, 2 * rank * n_pairs + a)
    ex.flush(g)
    g.sync()
    freq, st = g.finalize(cfg["d"])
    batch = args.batch_reads
    out = torch.empty((min(batch, n), maxwin, 4), dtype=torch.int32, device=dev)
    g.lookup_reads_exchange(ex.comm, d_packed[: min(batch, n)], None, None, uniform_len=L, stride_bytes=stride, out=out)   # index, buffers, module load
    ms, nl = (C.c_double * 8)(), (C.c_uint64 * 8)()
    g._ck(g.L.sdtgpu_phase_times(g.h, 1, ms, nl))
    dist.barrier()
    t0 = time.perf_counter()
    coll_ms, found, windows, calls = 0.0, 0, 0, 0
    for a in range(0, n, batch):
        b = min(a + batch, n)
        h = g.lookup_reads_exchange(ex.comm, d_packed[a:b], None, None, uniform_len=L, stride_bytes=stride, out=out)
        coll_ms += g.last_collective_ms
        found += int(((h[..., 3] & pkg.HIT_FOUND) != 0).sum())
        windows += (b - a) * maxwin
        calls += 1
    wall = time.perf_counter() - t0
    g._ck(g.L.sdtgpu_phase_times(g.h, 1, ms, nl))
    mine = torch.tensor([windows, found, wall * 1e6, coll_ms * 1e3, ms[7] * 1e3, calls, st.n_nodes], dtype=torch.float64, device=dev)
    allv = torch.empty((world, mine.numel()), dtype=torch.float64, device=dev)
    dist.all_gather_into_tensor(allv.view(-1), mine)
    if rank == 0:
        v = allv.cpu().numpy()
        wall_max = v[:, 2].max() / 1e6
        tot_w, tot_f = int(v[:, 0].sum()), int(v[:, 1].sum())
        # a window's query travels when its owner is another rank: key words out, a 16-byte hit back
        moved_per_window = (8 * g.lookup_route()["key_words"] + 16) * (world - 1) / world
        res = dict(config=args.config, gpus=world, K=K, reads_per_rank=n, batch_reads=batch, calls_per_rank=int(v[0, 5]),
                   windows=tot_w, nodes=int(v[:, 6].sum()),
                   windows_per_s_total=tot_w / wall_max, windows_per_s_per_rank=[float(x) for x in v[:, 0] / (v[:, 2] / 1e6)],
                   wall_s=round(wall_max, 4), collective_ms_per_rank=[round(x / 1e3, 3) for x in v[:, 3]],
                   stage_answer_unstage_ms_per_rank=[round(x / 1e3, 3) for x in v[:, 4]],
                   bytes_moved_per_window=moved_per_window, found_fraction=tot_f / tot_w, **card(rank))
        with open(os.path.join(out_dir, "result.json"), "w") as f:
            json.dump(res, f)
    g.close()
    ex.comm.close()
    dist.barrier()
    dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=0, help="processes, one per GPU (default: every visible GPU)")
    ap.add_argument("--config", default="C2")
    ap.add_argument("--pairs", type=int, default=0, help="read pairs per GPU (default: the config's)")
    ap.add_argument("--batch-reads", type=int, default=1 << 20)
    args = ap.parse_args()
    import tempfile
    import torch
    import torch.multiprocessing as mp
    world = args.gpus or torch.cuda.device_count()
    if world < 1 or world > torch.cuda.device_count():
        sys.exit(f"lookup_exchange_bench: {world} GPUs asked, {torch.cuda.device_count()} visible")
    with tempfile.TemporaryDirectory() as tmp:
        mp.spawn(_worker, args=(world, _free_port(), args, tmp), nprocs=world, join=True)
        with open(os.path.join(tmp, "result.json")) as f:
            res = json.load(f)
    print(json.dumps(res))
    if res["found_fraction"] != 1.0:
        sys.exit("lookup_exchange_bench: not every window was found")


if __name__ == "__main__":
    main()
