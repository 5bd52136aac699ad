"""Routed lookups on two GPUs (skipped on a single-GPU box), one process per GPU as in test_gpu_multi.py: every rank
builds its share of the table with one of the multi-GPU drivers, then routes its own key set and its own read shard
through sdtgpu_lookup_kmers_exchange / sdtgpu_lookup_reads_exchange; one call has no queries on rank 1.  The main
process compares every rank's hits with the oracle's expectation."""
import os
import sys

import numpy as np
import pytest

from test_gpu_lookup import assert_hits_equal, expected_read_hits, key_queries, table_of
from test_gpu_multi import _free_port

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
pytestmark = pytest.mark.gpu
N_PAIRS = 3000


def _worker(rank, world, port, K, kw, L, d, out_dir, mode, queries):
    sys.path.insert(0, ROOT)
    import torch
    import torch.distributed as dist
    import sdt_pkg
    pkg = sdt_pkg.load()
    from soapdenovo_trans_b200.exchange import Exchange, ReplicatedReads, SkmExchange
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    synth = pkg.synth
    reads, lens = synth.make_reads(synth.make_transcriptome(40, 5), N_PAIRS, L, 77, ragged=30)
    n = len(reads)
    lo, hi = rank * n // world, (rank + 1) * n // world
    stride = synth.stride_bytes(L)
    d_packed = torch.from_numpy(synth.pack_reads(reads[lo:hi], lens[lo:hi], stride)).to(dev)
    d_lens = torch.from_numpy(lens[lo:hi].astype(np.int32)).to(dev)
    g = pkg.PregraphGPU(K, kw, L, capacity_hint=500_000, device=rank, sliced=mode.startswith("skm"))
    if mode.startswith("skm"):
        ex = SkmExchange(pkg, g, world, rank, dev, native=(mode == "skm_native"))
    elif mode == "records":
        ex = Exchange(pkg, g, world, rank, dev, max_round_instances=2048 * (L - K + 1))
        g.set_owner(rank, world)       # the record exchange's share, declared for the routed lookups
    else:
        ex = ReplicatedReads(pkg, g, world, rank, dev, max_round_reads=2048, stride=stride)
    for a in range(0, hi - lo, 2048):
        b = min(a + 2048, hi - lo)
        ex.round(g, d_packed[a:b], b - a, 0, stride, lo + a, d_lens=d_lens[a:b])
    ex.flush(g)
    g.sync()
    g.finalize(d)
    uid = torch.zeros(128, dtype=torch.uint8, device=dev)
    if rank == 0:
        uid.copy_(torch.frombuffer(bytearray(pkg.pregraph.SkmComm.unique_id()), dtype=torch.uint8))
    dist.broadcast(uid, src=0)
    comm = pkg.pregraph.SkmComm(rank, bytes(uid.cpu().numpy().tobytes()), rank, world)
    mine = np.load(queries)[rank::world]
    np.save(os.path.join(out_dir, f"keys{rank}.npy"), g.lookup_kmers_exchange(comm, mine))
    none = g.lookup_kmers_exchange(comm, mine if rank == 0 else mine[:0])
    assert len(none) == (len(mine) if rank == 0 else 0)
    out = g.lookup_reads_exchange(comm, d_packed, d_lens, None, stride_bytes=stride)
    np.save(os.path.join(out_dir, f"reads{rank}.npy"), pkg.hits_numpy(out))
    comm.close()
    g.close()
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.parametrize("mode", ["reads", "records", "skm", "skm_native"])
@pytest.mark.parametrize("K,kw,L,d", [(25, 1, 100, 0), (63, 2, 100, 2), (127, 4, 150, 0)])
def test_two_gpu_routed_lookups_match_oracle(pkg, oracle, tmp_path, K, kw, L, d, mode):
    import torch
    import torch.multiprocessing as mp
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    world = 2
    synth = pkg.synth
    reads, lens = synth.make_reads(synth.make_transcriptome(40, 5), N_PAIRS, L, 77, ragged=30)
    ref = oracle.run_hashing(reads, lens, K, kw, 8, d)
    queries, want = key_queries(pkg, oracle, ref, K, kw, np.random.default_rng(K))
    np.save(tmp_path / "queries.npy", queries)
    mp.spawn(_worker, args=(world, _free_port(), K, kw, L, d, str(tmp_path), mode, str(tmp_path / "queries.npy")), nprocs=world, join=True)
    table = table_of(ref)
    n = len(reads)
    for r in range(world):
        assert_hits_equal(np.load(tmp_path / f"keys{r}.npy"), want[r::world], f"{mode} keys of rank {r}")
        lo, hi = r * n // world, (r + 1) * n // world
        wr = expected_read_hits(pkg, oracle, table, reads[lo:hi], lens[lo:hi], K, kw, L)
        assert_hits_equal(np.load(tmp_path / f"reads{r}.npy"), wr, f"{mode} reads of rank {r}")
