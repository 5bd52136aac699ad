"""Multi-GPU sharding: one process per GPU, k-mers sharded by owner.

The reference's only parallelism is hash-partitioned shared-nothing tables (owner =
hash_kmer % thrd_num, prlHashReads.c:81) where every worker scans the whole batch and keeps what it
owns (:79-88).  Two ways to stretch that over GPUs live here:

* `ReplicatedReads` (default): the ranks all-gather their 2-bit packed reads (28 bytes per 100-bp
  read) over NVLink and every rank chops ALL reads but inserts only the k-mers it owns
  (sdtgpu_set_owner).  No per-k-mer records exist; the redundant chop is ~20x cheaper than an insert.
* `Exchange`: each rank chops only its own reads, buckets every instance as a 16-byte record by owner
  (sdtgpu_bucket_reads_device), the bins cross NVLink with one grouped NCCL send/recv per round and
  each rank upserts what it received (sdtgpu_insert_records_device).

* `SkmExchange` (sliced build, `PregraphGPU(..., sliced=True)`): each rank turns only its own reads
  into super-k-mer records (one record per ~8 consecutive windows, 4 bytes per instance), the table
  slices are dealt to the ranks in contiguous ranges, the records are grouped by slice — hence by
  owner — and cross NVLink in ONE variable-size all-to-all per epoch; every rank then builds its own
  slices in shared memory (sdtgpu_skm_stage / sdtgpu_skm_import).

Updates are commutative, so arrival order is free and the union of the ranks' tables is the
reference's multiset either way.

`exchange_records` is the backend-agnostic plumbing (counts all-to-all, offsets, payload
all-to-all); it is exercised on CPU with the gloo backend in tests/test_exchange_cpu.py.
"""
from __future__ import annotations

import torch
import torch.distributed as dist


def exchange_records(send: torch.Tensor, send_counts: torch.Tensor, recv: torch.Tensor, group=None):
    """send: [world, cap, words] int64 bins, bin d holds send_counts[d] valid records for rank d.
    recv: flat [recv_cap, words] int64.  Returns (n_received, recv_counts list).
    Two collectives: a tiny all-to-all of the counts, then the variable-size payload all-to-all
    (batched isend/irecv = one NCCL grouped send/recv; no packing copy — the bins are sent in place;
    the same code runs on gloo for the CPU tests)."""
    world = dist.get_world_size(group)
    counts_host = [int(x) for x in send_counts.tolist()]
    cap = send.shape[1]
    if max(counts_host) > cap:
        raise OverflowError(f"a send bin overflowed: {max(counts_host)} > {cap}")
    sc = torch.tensor(counts_host, dtype=torch.int64, device=send.device)
    rc = torch.empty(world, dtype=torch.int64, device=send.device)
    dist.all_to_all_single(rc, sc, group=group)
    recv_counts = [int(x) for x in rc.tolist()]
    total = sum(recv_counts)
    if total > recv.shape[0]:
        raise OverflowError(f"receive buffer too small: {total} > {recv.shape[0]}")
    rank = dist.get_rank(group)
    ops, off = [], 0
    for src, n in enumerate(recv_counts):
        seg = recv[off:off + n]
        off += n
        if n == 0:
            continue
        if src == rank:
            seg.copy_(send[rank, :n])      # own bin: device-local copy, never touches the fabric
        else:
            ops.append(dist.P2POp(dist.irecv, seg, src, group=group))
    for dst in range(world):
        if dst != rank and counts_host[dst]:
            ops.append(dist.P2POp(dist.isend, send[dst, :counts_host[dst]], dst, group=group))
    if ops:
        for req in dist.batch_isend_irecv(ops):      # NCCL: one grouped ncclSend/ncclRecv launch
            req.wait()
    return total, recv_counts


class Exchange:
    """Round driver for bench.py / multi-rank callers, software-pipelined over two buffer sets:
    bucket(r+1) and the NCCL exchange of round r+1 run on the table's auxiliary stream while
    insert(r) runs on its main stream; events order buffer reuse."""

    def __init__(self, pkg, g, world: int, rank: int, dev, max_round_instances: int, slack: float = 1.15):
        self.pkg, self.world, self.rank, self.dev = pkg, world, rank, dev
        self.words = g.record_bytes() // 8
        self.cap = int(max_round_instances / world * slack) + 65536
        self.send = [torch.empty((world, self.cap, self.words), dtype=torch.int64, device=dev) for _ in range(2)]
        self.counts = [torch.zeros(world, dtype=torch.int64, device=dev) for _ in range(2)]
        self.recv = [torch.empty((int(self.cap * world), self.words), dtype=torch.int64, device=dev) for _ in range(2)]
        self.inserted = [torch.cuda.Event() for _ in range(2)]     # insert(r) finished reading recv[r % 2]
        self.received = torch.cuda.Event()
        self.r = 0
        self.rebind(g)
        self.nvlink_bytes = 0

    def rebind(self, g):
        self.main = torch.cuda.ExternalStream(g.stream, device=self.dev)
        self.aux = torch.cuda.ExternalStream(g.aux_stream, device=self.dev)

    def round(self, g, d_packed, n_reads, uniform_len, stride, first_read_ordinal, d_lens=None, d_nmask=None):
        """d_nmask: the -n N mask of the round's reads (stride / 2 bytes per read), for handles created with n_kmer."""
        b = self.r & 1
        self.r += 1
        with torch.cuda.stream(self.aux):
            self.aux.wait_event(self.inserted[b])          # buffer set b is free again
            self.counts[b].zero_()
            g.bucket_reads_device(d_packed, d_lens, d_nmask, n_reads, uniform_len, stride, first_read_ordinal,
                                  self.world, self.send[b], self.cap, self.counts[b])
            total, rc = exchange_records(self.send[b], self.counts[b], self.recv[b])
            self.received.record(self.aux)
        self.nvlink_bytes += (total - rc[self.rank]) * self.words * 8
        with torch.cuda.stream(self.main):
            self.main.wait_event(self.received)
            g.insert_records_device(self.recv[b], total)
            self.inserted[b].record(self.main)

    def flush(self, g):
        pass


class ReplicatedReads:
    """Round driver of the replicated-reads sharding, pipelined over two gather buffers: the NCCL
    all-gather of round r+1 runs on the table's auxiliary stream while the inserts of round r run on
    its main stream."""

    def __init__(self, pkg, g, world: int, rank: int, dev, max_round_reads: int, stride: int, group=None):
        self.world, self.rank, self.dev, self.group = world, rank, dev, group
        g.set_owner(rank, world)
        self.buf = [torch.empty((world, max_round_reads, stride), dtype=torch.uint8, device=dev) for _ in range(2)]
        self.lens = [torch.empty((world, max_round_reads), dtype=torch.int32, device=dev) for _ in range(2)]
        self.mask = None        # [world, max_round_reads, stride / 2] x 2, made when a round first brings an N mask
        self.meta = [torch.empty((world, 2), dtype=torch.int64, device=dev) for _ in range(2)]
        self.inserted = [torch.cuda.Event() for _ in range(2)]
        self.received = torch.cuda.Event()
        self.max_round_reads, self.stride, self.r = max_round_reads, stride, 0
        self.nvlink_bytes = 0
        self.rebind(g)

    def rebind(self, g):
        g.set_owner(self.rank, self.world)
        self.main = torch.cuda.ExternalStream(g.stream, device=self.dev)
        self.aux = torch.cuda.ExternalStream(g.aux_stream, device=self.dev)

    def round(self, g, d_packed, n_reads, uniform_len, stride, first_read_ordinal, d_lens=None, d_nmask=None):
        """d_packed: this rank's reads of the round ([n_reads, stride] uint8 on the device).  Ranks may
        bring different numbers of reads (<= max_round_reads).  d_nmask: their -n N mask (all ranks or none)."""
        b = self.r & 1
        self.r += 1
        if d_nmask is not None and self.mask is None:
            self.mask = [torch.zeros((self.world, self.max_round_reads, stride // 2), dtype=torch.uint8, device=self.dev) for _ in range(2)]
        with torch.cuda.stream(self.aux):
            self.aux.wait_event(self.inserted[b])
            mine = torch.tensor([first_read_ordinal, n_reads], dtype=torch.int64, device=self.dev)
            dist.all_gather_into_tensor(self.meta[b].view(-1), mine, group=self.group)
            src = d_packed
            if n_reads != self.max_round_reads:          # NCCL all-gather wants equal contributions
                src = self.buf[b][self.rank]
                src[:n_reads].copy_(d_packed[:n_reads])
            dist.all_gather_into_tensor(self.buf[b].view(-1), src.reshape(-1)[: self.max_round_reads * self.stride], group=self.group)
            if d_lens is not None:
                ls = self.lens[b][self.rank]
                ls[:n_reads].copy_(d_lens[:n_reads])
                dist.all_gather_into_tensor(self.lens[b].view(-1), ls, group=self.group)
            if d_nmask is not None:
                mk = self.mask[b][self.rank]
                mk[:n_reads].copy_(d_nmask[:n_reads].reshape(n_reads, -1))
                dist.all_gather_into_tensor(self.mask[b].view(-1), mk.reshape(-1), group=self.group)
            meta = self.meta[b].tolist()
            self.received.record(self.aux)
        self.nvlink_bytes += sum(m[1] for i, m in enumerate(meta) if i != self.rank) * self.stride
        with torch.cuda.stream(self.main):
            self.main.wait_event(self.received)
            for s_rank, (first, n) in enumerate(meta):
                if n:
                    g.push_reads(self.buf[b][s_rank], self.lens[b][s_rank] if d_lens is not None else None,
                                 self.mask[b][s_rank] if d_nmask is not None else None, n_reads=int(n), uniform_len=uniform_len, stride_bytes=stride,
                                 first_read_ordinal=int(first), device=True)
            self.inserted[b].record(self.main)

    def flush(self, g):
        pass


def exchange_runs(send_list, words: int, make_recv, group=None):
    """The super-k-mer exchange's plumbing, backend-agnostic (NCCL on the GPUs, gloo in tests/test_exchange_cpu.py).
    send_list[r]: flat int64 tensor with the records for rank r (`words` int64 each; views into the buffer that
    sdtgpu_skm_stage hands out — nothing is packed).  make_recv(total_records) -> flat int64 tensor to receive into
    (sdtgpu_skm_import_buffer); the runs arrive in source-rank order.
    Two collectives: the counts, then the records (one grouped send/recv).  Returns (total_records, recv_counts)."""
    world = dist.get_world_size(group)
    rank = dist.get_rank(group)
    dev = send_list[0].device
    send_counts = [int(t.numel()) // words for t in send_list]
    sc = torch.tensor(send_counts, dtype=torch.int64, device=dev)
    rc = torch.empty(world, dtype=torch.int64, device=dev)
    dist.all_to_all_single(rc, sc, group=group)
    recv_counts = [int(x) for x in rc.tolist()]
    total = sum(recv_counts)
    recv = make_recv(total)
    ops, off = [], 0
    for src, n in enumerate(recv_counts):
        seg = recv[off * words:(off + n) * words]
        off += n
        if n == 0:
            continue
        if src == rank:
            seg.copy_(send_list[rank])      # own records: device-local copy, never touches the fabric
        else:
            ops.append(dist.P2POp(dist.irecv, seg, src, group=group))
    for dst in range(world):
        if dst != rank and send_counts[dst]:
            ops.append(dist.P2POp(dist.isend, send_list[dst], dst, group=group))
    if ops:
        for req in dist.batch_isend_irecv(ops):      # NCCL: one grouped ncclSend/ncclRecv launch
            req.wait()
    return total, recv_counts


class _DevMem:
    """A device allocation owned by the library, seen by torch through __cuda_array_interface__ (no copy)."""

    def __init__(self, ptr: int, nbytes: int):
        self.__cuda_array_interface__ = {"shape": (max(nbytes // 8, 1),), "typestr": "<i8", "data": (ptr, False), "version": 2}


def _wrap(ptr: int, nbytes: int, dev) -> torch.Tensor:
    if nbytes == 0 or ptr == 0:
        return torch.empty(0, dtype=torch.int64, device=dev)
    return torch.as_tensor(_DevMem(ptr, nbytes), device=dev)[: nbytes // 8]


class SkmExchange:
    """Round driver of the super-k-mer exchange (sliced build on several GPUs).  `round` only pushes this
    rank's reads (the emit kernel runs, nothing crosses the fabric yet); `flush` groups the records by
    slice, exchanges counts and records with two all-to-alls and builds this rank's slices."""

    def __init__(self, pkg, g, world: int, rank: int, dev, group=None, native: bool = False):
        """native: the exchange runs inside the library (sdtgpu_skm_exchange, NCCL bound by the library itself);
        torch.distributed then only carries the communicator's 128-byte id to the ranks, once."""
        self.world, self.rank, self.dev, self.group = world, rank, dev, group
        self.comm = None
        if native:
            uid, why = torch.zeros(128, dtype=torch.uint8, device=dev), ""
            if rank == 0:
                try:
                    uid.copy_(torch.frombuffer(bytearray(pkg.pregraph.SkmComm.unique_id()), dtype=torch.uint8))
                except Exception as e:      # noqa: BLE001  (the other ranks are waiting in the broadcast: tell them with an all-zero id)
                    why = str(e)
            dist.broadcast(uid, src=0 if group is None else dist.get_global_rank(group, 0), group=group)
            if not bool(uid.any()):
                raise RuntimeError(f"SkmExchange(native=True): no NCCL id from rank 0 {why}")
            self.comm = pkg.pregraph.SkmComm(torch.device(dev).index or 0, bytes(uid.cpu().numpy().tobytes()), rank, world)
        self.nvlink_bytes = 0
        self.collective_ms = 0.0        # device time of the counts + records exchange (CUDA events on the handle's stream)
        self.host_ms = {}               # wall clock of the phases of flush (host side, this rank)
        self.host_log = []
        self.rebind(g)

    def rebind(self, g):
        g.skm_set_world(self.rank, self.world)
        geo = g.slice_geometry()
        self.rec_bytes = int(geo["record_bytes"])
        self.main = torch.cuda.ExternalStream(g.stream, device=self.dev)
        self.aux = torch.cuda.ExternalStream(g.aux_stream, device=self.dev)     # the caller may stage a round's reads on it
        self.inserted = [torch.cuda.Event() for _ in range(2)]
        self.r = 0
        self.reads_end = 0
        # every rank must cut the minimizer space the same way: same capacity_hint, K and minimizer length
        mine = torch.tensor([geo["n_slices"], geo["m"], geo["slice_slots"]], dtype=torch.int64, device=self.dev)
        seen = torch.empty((self.world, 3), dtype=torch.int64, device=self.dev)
        dist.all_gather_into_tensor(seen.view(-1), mine, group=self.group)
        if not bool((seen == mine).all()):
            raise ValueError(f"SkmExchange: ranks disagree on the slice geometry (pass the same capacity_hint everywhere): {seen.tolist()}")

    def round(self, g, d_packed, n_reads, uniform_len, stride, first_read_ordinal, d_lens=None, d_nmask=None):
        b = self.r & 1
        self.r += 1
        self.reads_end = max(self.reads_end, int(first_read_ordinal) + int(n_reads))
        staged = torch.cuda.Event()
        staged.record(self.aux)                     # whatever the caller queued on the auxiliary stream (an H2D copy of the round)
        self.main.wait_event(staged)
        g.push_reads(d_packed, d_lens, d_nmask, n_reads=int(n_reads), uniform_len=uniform_len, stride_bytes=stride,
                     first_read_ordinal=int(first_read_ordinal), device=True)
        self.inserted[b].record(self.main)          # the round's buffer is free again (the library keeps its own copy of the reads)

    def flush(self, g):
        import time
        t0 = time.perf_counter()
        if self.comm is not None:
            total, ms = g.skm_exchange(self.comm, self.reads_end)
            t4 = time.perf_counter()
            self.collective_ms += ms
            self.host_ms["native"] = self.host_ms.get("native", 0.0) + 1e3 * (t4 - t0)
            self.host_ms["flushes"] = self.host_ms.get("flushes", 0) + 1
            self.host_log.append([round(1e3 * (t4 - t0), 2)])
            return total
        bound = torch.tensor([self.reads_end], dtype=torch.int64, device=self.dev)
        dist.all_reduce(bound, op=dist.ReduceOp.MAX, group=self.group)
        g.skm_set_ordinal_bound(int(bound.item()))  # reads of all ranks this epoch: 32-bit ordinals in the slice images when they fit
        t1 = time.perf_counter()
        ptr, starts, counts = g.skm_stage()         # merges this rank's copies, packs by owner; synchronises the handle's stream
        t2 = time.perf_counter()
        rb, w8 = self.rec_bytes, self.rec_bytes // 8
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        with torch.cuda.stream(self.main):
            send = [_wrap(ptr + starts[r] * rb, counts[r] * rb, self.dev) for r in range(self.world)]
            e0.record(self.main)
            total, _ = exchange_runs(send, w8, lambda n: _wrap(g.skm_import_buffer(n), n * rb, self.dev), group=self.group)
            e1.record(self.main)
            self.nvlink_bytes += (sum(counts) - counts[self.rank]) * rb
        t3 = time.perf_counter()
        g.skm_import(total)                         # on the handle's stream, after the exchange (drains the stream)
        t4 = time.perf_counter()
        self.collective_ms += e0.elapsed_time(e1)
        for k, v in zip(("bound", "stage", "exchange", "import"), (t1 - t0, t2 - t1, t3 - t2, t4 - t3)):
            self.host_ms[k] = self.host_ms.get(k, 0.0) + 1e3 * v
        self.host_ms["flushes"] = self.host_ms.get("flushes", 0) + 1
        self.host_log.append([round(1e3 * (b - a), 2) for a, b in ((t0, t1), (t1, t2), (t2, t3), (t3, t4))])   # per flush: bound, stage, exchange, import
        return total


def plan_reader(reader, dev, group=None) -> dict:
    """Plans a shard reader (pregraph.DeviceReadPacker(..., rank=, world=)) over torch.distributed: this rank's summary,
    an all-gather of every rank's 256 bytes, then the same host-side plan on every rank.  Collective over `group`,
    whose rank and size must be the reader's.  Returns the plan (records this rank returns, library_records, n1, n2)."""
    world = dist.get_world_size(group)
    if world != reader.world:
        raise ValueError(f"plan_reader: the group has {world} ranks, the reader {reader.world}")
    err = None
    try:
        mine = reader.summary()
    except Exception as e:      # noqa: BLE001  (the other ranks are in the all-gather: an all-zero block makes every plan refuse)
        mine, err = bytes(reader.SUMMARY_BYTES), e
    t = torch.frombuffer(bytearray(mine), dtype=torch.uint8).to(dev)
    allv = torch.empty((world, reader.SUMMARY_BYTES), dtype=torch.uint8, device=dev)
    dist.all_gather_into_tensor(allv.view(-1), t, group=group)
    host = allv.cpu().numpy()
    if err is not None:
        raise err
    return reader.plan([host[r].tobytes() for r in range(world)])
