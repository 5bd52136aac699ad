#!/usr/bin/env python
"""bench.py — k-mers inserted/s in pregraph hashing (BASELINE.json metric), 1..8 B200.

One "step" = one pass of the hot path over the whole synthetic workload: empty the handle, push every
read (sdtgpu_push_reads_device), sdtgpu_sync — reads -> super-k-mer records in per-slice chains ->
copies merged, chains cut into work items -> every item built in shared memory -> node store (at N > 1:
records merged per sender, exchanged by slice owner over NCCL, built by the owner).  Nothing about
the data is learned outside the timed region: the handle gets NO capacity hint on one GPU (the library
sizes itself from the number of windows pushed, inside the step) and the same closed-form estimate
on several GPUs (every rank must cut the minimizer space the same way).

`value`   the step with the packed reads already resident in HBM (CUDA events on the handle's stream);
`e2e`     the same job through the C ABI with HOST buffers (pinned): H2D copies and the D2H read of the
          result counters inside the timed region;
`e2e_from_files`  FASTA on disk -> sdtpack (parallel parse + 2-bit pack) -> sdtgpu_push_reads -> counters,
          on the SAME sample of reads the reference arm hashes (like for like with `cpu_baseline`), and with
          --files-full on the whole workload;
`roofline`  the insert pipeline's algorithmic bytes (SURVEY.md §8d: 64 B per instance for K <= 63, 96 B for
          K <= 127) over the summed CUDA-event times of its kernels, against the measured HBM copy bandwidth
          in MEASURED_PEAKS.json; `traffic` = the DRAM bytes ncu measured for the same kernels on this config;
`cpu_baseline`  the unmodified reference's prlRead2HashTable (oracle/_ref) on a bounded sample of the same reads;
`parity_checked`  the sliced build's table fingerprint equals the single-pass insert's on this workload (untimed).

--dump-outputs DIR  writes the table the last timed step built (dump_outputs) as .npy files, so that two builds of the
          project can be compared output for output on the same seeded inputs (one GPU).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--config C2] [--pairs P] [--impl reference] [--dump-outputs DIR]
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

BYTES_PER_INSTANCE = {1: 64, 2: 64, 4: 96}      # SURVEY.md §8d
# Measured on this pool's B200 with tools/randacc_bench.cu (profiles/r1_randacc_bench.txt): requests to
# cold lines of a table >> L2 complete at 36.65 G/s no matter their kind (load, CAS, RED) or width; an
# upsert needs at least one load and one atomic, so a single-pass insert cannot exceed half of that.
RANDOM_REQUESTS_PER_S = 36.65e9
MIN_REQUESTS_PER_INSTANCE = {1: 2, 2: 2, 4: 3}
METRIC = "k-mers inserted/s in pregraph hashing"
UNIT = "k-mer instances/s"


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def estimate_distinct(instances: int, K: int) -> int:
    """The library's own rule when it gets no hint (estimate_distinct, csrc/sdtgpu.cu)."""
    return int(min(instances + 1024.0, instances * (1.0 - 0.99 ** K) * 1.05 + 65536.0))


class ClockSampler(threading.Thread):
    """SM clocks and throttle reasons during the timed region (B200_PROFILING.md's clocks line), read through NVML
    (nvidia_ml_py) on this rank's GPU: an `nvidia-smi` process per sample takes a driver-wide lock for tens of
    milliseconds and stalls every CUDA call of every rank meanwhile.  Falls back to nvidia-smi without NVML."""

    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        super().__init__(daemon=True)
        self.index, self.samples, self.stop_flag = index, [], threading.Event()
        self.nvml, self.handle = None, None
        if index >= 0 and not os.environ.get("BENCH_NO_SAMPLER"):
            try:
                import pynvml
                pynvml.nvmlInit()
                # CUDA_VISIBLE_DEVICES may renumber the devices: go by the PCI bus id of the CUDA device
                import torch
                pr = torch.cuda.get_device_properties(index)
                try:
                    bus_id = f"{getattr(pr, 'pci_domain_id', 0):08X}:{pr.pci_bus_id:02X}:{pr.pci_device_id:02X}.0"
                    self.handle = pynvml.nvmlDeviceGetHandleByPciBusId(bus_id.encode())
                except Exception:
                    self.handle = pynvml.nvmlDeviceGetHandleByIndex(index)
                self.nvml = pynvml
                self._sample_nvml()      # the first queries initialise things inside NVML: not inside the timed region
                self.samples.clear()
            except Exception:
                self.nvml = None

    def _sample_nvml(self):
        n = self.nvml
        sm = n.nvmlDeviceGetClockInfo(self.handle, n.NVML_CLOCK_SM)
        mx = n.nvmlDeviceGetMaxClockInfo(self.handle, n.NVML_CLOCK_SM)
        try:
            r = n.nvmlDeviceGetCurrentClocksEventReasons(self.handle)
        except Exception:
            r = n.nvmlDeviceGetCurrentClocksThrottleReasons(self.handle)
        flags = [("hw_slowdown", getattr(n, "nvmlClocksThrottleReasonHwSlowdown", 0x8)), ("hw_thermal_slowdown", getattr(n, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40)),
                 ("sw_thermal_slowdown", getattr(n, "nvmlClocksThrottleReasonSwThermalSlowdown", 0x20)), ("sw_power_cap", getattr(n, "nvmlClocksThrottleReasonSwPowerCap", 0x4))]
        self.samples.append([str(sm), str(mx)] + ["Active" if r & bit else "Not Active" for _, bit in flags])

    def run(self):
        if self.index < 0 or os.environ.get("BENCH_NO_SAMPLER"):      # (several GPUs: rank 0 samples its GPU)
            return
        while not self.stop_flag.is_set():
            try:
                if self.nvml is not None:
                    self._sample_nvml()
                else:
                    out = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-i", str(self.index)],
                                         capture_output=True, text=True, timeout=5).stdout.strip()
                    if out:
                        self.samples.append([x.strip() for x in out.split(",")])
            except Exception:
                pass
            self.stop_flag.wait(0.1 if self.nvml is not None else 0.5)

    def summary(self):
        sm = [int(s[0]) for s in self.samples if s[0].isdigit()]
        mx = [int(s[1]) for s in self.samples if s[1].isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({n for s in self.samples for n, v in zip(names, s[2:6]) if v.lower().startswith("active")})
        return {"sm_mhz": int(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(self.samples), "source": "nvml" if self.nvml is not None else "nvidia-smi"}


def unpack_reads(packed: np.ndarray, read_len: int) -> np.ndarray:
    b = packed[:, : (read_len + 3) // 4]
    out = np.empty((b.shape[0], b.shape[1] * 4), dtype=np.uint8)
    out[:, 0::4], out[:, 1::4], out[:, 2::4], out[:, 3::4] = b >> 6, (b >> 4) & 3, (b >> 2) & 3, b & 3
    return out[:, :read_len]


def write_fasta_pair(dirpath: str, reads: np.ndarray, tag: str = "s"):
    """reads: base codes [n, L] in arrival order (read1, read2 alternately) -> f1/f2 FASTA, one sequence line per
    record, file sizes not a multiple of 32 768 (SURVEY.md appendix C).  Vectorised: C2 in full is 5.7 GB of text."""
    n, L = reads.shape
    lut = np.frombuffer(b"ACTG", dtype=np.uint8)
    paths = []
    for mate in (0, 1):
        r = reads[mate::2]
        m = len(r)
        hdr = np.frombuffer(b">" + tag.encode() + b"0000000000\n", dtype=np.uint8)
        rec = np.empty((m, len(hdr) + L + 1), dtype=np.uint8)
        rec[:, :len(hdr)] = hdr
        idx = np.arange(m, dtype=np.int64)
        for d in range(10):     # decimal read number into the header
            rec[:, len(hdr) - 2 - d] = 48 + (idx // 10 ** d) % 10
        rec[:, len(hdr):len(hdr) + L] = lut[r]
        rec[:, -1] = 10
        path = os.path.join(dirpath, f"{tag}_{mate + 1}.fa")
        with open(path, "wb") as f:
            f.write(rec.tobytes())
            if (rec.size % 32768) == 0:
                f.write(b"\n")
        paths.append(path)
    cfg = os.path.join(dirpath, f"{tag}.cfg")
    with open(cfg, "w") as f:
        f.write(f"max_rd_len={L}\n[LIB]\navg_ins=200\nreverse_seq=0\nasm_flags=3\nf1={paths[0]}\nf2={paths[1]}\n")
    return cfg, paths


def reference_run(cfg_d: dict, sample_reads: np.ndarray, threads: int):
    """Unmodified reference prlRead2HashTable (oracle/_ref/ref_hash_*) on `sample_reads` (base codes)."""
    from oracle import oracle as O
    with tempfile.TemporaryDirectory() as d:
        cfg, _ = write_fasta_pair(d, sample_reads)
        kw = 1 if cfg_d["key_words"] == 1 else 4
        info, _, _ = O.run_reference(cfg, os.path.join(d, "out"), cfg_d["K"], kw, threads, 0, dump=False)
    return info


def reference_built(cfg_d: dict) -> bool:
    """oracle/_ref is built only where the SOAPdenovo-Trans sources are at hand (oracle/Makefile)."""
    from oracle import oracle as O
    return O.ref_binary(1 if cfg_d["key_words"] == 1 else 4) is not None


DUMP_BYTES = 60_000_000     # all files of --dump-outputs together (under 64 MB)
DUMP_SEED = 0x5D7D06B5E1EC7ED


def _halves(a) -> np.ndarray:
    """uint64 -> float64 [..., 2] (high, low 32 bits): exact, unlike a plain cast."""
    a = np.asarray(a, dtype=np.uint64)
    return np.stack([(a >> np.uint64(32)).astype(np.float64), (a & np.uint64(0xFFFFFFFF)).astype(np.float64)], axis=-1)


def dump_outputs(pkg, g, out_dir: str) -> dict:
    """Writes what the handle holds after a step, i.e. what a caller of the timed path receives, as float64 .npy:
      stats           [n_instances, n_nodes, n_reads]
      table_checksum  [4, 2] sdtgpu_table_checksum (include/sdtgpu.h) as 32-bit halves: the fingerprint of the whole table
      nodes_key       [n, 2 x device key words] 32-bit halves, most significant first; nodes_count, nodes_l_links,
      nodes_rword, nodes_ordinal [n]: the n nodes with the smallest seeded hash of their key, sorted by key.
    The sample is chosen by content, so it does not depend on where a build keeps a node; n is as large as DUMP_BYTES allows.
    Returns {name: shape}."""
    st = g.stats()
    W = int(st.device_key_words)
    nodes = g.export_nodes(1)
    cap = min(len(nodes), (DUMP_BYTES - (1 << 16)) // (8 * (2 * W + 4)))
    hs, idx = [], []
    chunk = 1 << 24
    with np.errstate(over="ignore"):
        for a in range(0, len(nodes), chunk):
            key = nodes["key"][a:a + chunk]
            h = np.full(len(key), DUMP_SEED, dtype=np.uint64)
            for q in range(4 - W, 4):
                h = pkg.synth.mix64(h ^ key[:, q])
            keep = np.argpartition(h, cap - 1)[:cap] if len(h) > cap else np.arange(len(h))
            hs.append(h[keep])
            idx.append(keep + a)
    if cap:
        h, idx = np.concatenate(hs), np.concatenate(idx)
        sel = nodes[idx[np.argsort(h, kind="stable")[:cap]]]
        sel = sel[np.lexsort(tuple(sel["key"][:, q] for q in range(3, 3 - W, -1)))]
    else:
        sel = nodes[:0]
    del nodes
    out = {
        "stats": np.array([st.n_instances, st.n_nodes, st.n_reads], dtype=np.float64),
        "table_checksum": _halves(g.table_checksum()),
        "nodes_key": _halves(sel["key"][:, 4 - W:]).reshape(len(sel), 2 * W),
        "nodes_count": sel["count"].astype(np.float64),
        "nodes_l_links": sel["l_links"].astype(np.float64),
        "nodes_rword": sel["rword"].astype(np.float64),
        "nodes_ordinal": sel["ordinal"].astype(np.float64),
    }
    os.makedirs(out_dir, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)
    return {name: list(a.shape) for name, a in out.items()}


def host_sample(cfg_d: dict, n_pairs: int) -> np.ndarray:
    """The first n_pairs pairs of the workload, generated on the host (bit-identical to the device generator)."""
    import sdt_pkg
    synth = sdt_pkg.load().synth
    tr = synth.make_transcriptome(cfg_d["n_transcripts"], cfg_d["seed"], hot=cfg_d["hot"])
    out = []
    for a in range(0, n_pairs, 250_000):
        reads, _ = synth.make_reads(tr, min(250_000, n_pairs - a), cfg_d["read_len"], cfg_d["seed"], first_pair=a)
        out.append(reads)
    return np.concatenate(out)


def ref_threads() -> int:
    return max(1, min(os.cpu_count() or 8, 64))


def files_e2e(pkg, cfg_d, reads: np.ndarray, device: int, batch_reads: int, repeats: int = 2):
    """FASTA on disk -> sdtpack_next -> sdtgpu_push_reads (double-buffered pinned batches) -> counters.
    The handle gets no hint.  Returns (instances/s, seconds, instances, nodes) of the fastest repeat."""
    import ctypes as C
    L, K, kw = cfg_d["read_len"], cfg_d["K"], cfg_d["key_words"]
    lib = pkg.library()
    stride = pkg.synth.stride_bytes(L)
    best = None
    with tempfile.TemporaryDirectory() as d:
        _, paths = write_fasta_pair(d, reads, tag="f")
        bufs = []
        for _ in range(2):
            p, l = C.c_void_p(), C.c_void_p()
            assert lib.sdtgpu_host_alloc(C.byref(p), batch_reads * stride) == 0 and lib.sdtgpu_host_alloc(C.byref(l), batch_reads * 4) == 0
            bufs.append((p, l))
        try:
            with pkg.PregraphGPU(K, kw, L, capacity_hint=0, device=device, sliced=True) as g:
                for rep in range(repeats + 1):      # first pass: page cache + allocations
                    t0 = time.perf_counter()
                    g.reset()
                    rd = pkg.ReadPacker(paths[0], paths[1], fastq=False)
                    pushed, cur = 0, 0
                    while True:
                        p, l = bufs[cur]
                        n = lib.sdtpack_next(rd.h, L, 0, 0, p, l, None, batch_reads, stride)
                        if n <= 0:
                            break
                        g._ck(lib.sdtgpu_push_reads(g.h, p, l, None, n, 0, stride, pushed))
                        pushed += n
                        cur ^= 1
                    rd.close()
                    st = g.stats()
                    dt = time.perf_counter() - t0
                    if rep and (best is None or dt < best[1]):
                        best = (st.n_instances / dt, dt, int(st.n_instances), int(st.n_nodes))
        finally:
            for p, l in bufs:
                lib.sdtgpu_host_free(p)
                lib.sdtgpu_host_free(l)
    return best


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="C2")
    ap.add_argument("--pairs", type=int, default=0, help="override the config's read-pair count (testing)")
    ap.add_argument("--transcripts", type=int, default=0, help="override the config's transcript count (testing: keeps the coverage of the full workload at a smaller size)")
    ap.add_argument("--cpu-sample-pairs", type=int, default=1_000_000)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-parity", action="store_true", help="skip the untimed fingerprint check against the single-pass insert")
    ap.add_argument("--files-full", action="store_true", help="also measure e2e_from_files on the whole workload (writes it as FASTA first)")
    ap.add_argument("--batch-reads", type=int, default=1 << 22)
    ap.add_argument("--exchange", default="reads", choices=["reads", "records", "reads-replicated"],
                    help="multi-GPU sharding of --path direct: all-gather the packed reads and insert owned k-mers (default) or exchange k-mer records")
    ap.add_argument("--skm-exchange", default="native", choices=["native", "torch"],
                    help="several GPUs, sliced build: the exchange inside the library (sdtgpu_skm_exchange: NCCL bound by libsdtgpu.so) or driven from Python over torch.distributed")
    ap.add_argument("--path", default="sliced", choices=["auto", "direct", "sliced"],
                    help="insert path: the sliced build (super-k-mer records -> chains -> work items built in shared memory; every config) "
                         "or the single-pass upsert (direct)")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="several GPUs: weak = the config's reads PER GPU (the driver's contract); strong = the config's reads in total, split over the GPUs")
    ap.add_argument("--hint", type=int, default=-1, help="capacity_hint for the handle (-1: none on one GPU, the closed-form estimate on several)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the table the last one built to DIR/<name>.npy (float64, one GPU, see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and (args.impl != "ours" or int(os.environ.get("WORLD_SIZE", "1")) > 1):
        ap.error("--dump-outputs needs --impl ours on one GPU")
    if args.path == "auto":
        args.path = "sliced"
    import sdt_pkg
    pkg = sdt_pkg.load()
    synth = pkg.synth
    cfg_d = dict(synth.CONFIGS[args.config])
    sliced = args.path == "sliced"
    if args.pairs:
        cfg_d["n_pairs"] = args.pairs
    if args.transcripts:
        cfg_d["n_transcripts"] = args.transcripts
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.scaling == "strong" and world > 1:
        cfg_d["n_pairs"] = cfg_d["n_pairs"] // world      # the config's reads in total: rank r takes pairs [r, r + 1) x n_pairs / world
    if os.environ.get("BENCH_TRACE_RANK0") and rank == 0:
        os.environ["SDTGPU_TRACE"] = "1"
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    K, kw, L = cfg_d["K"], cfg_d["key_words"], cfg_d["read_len"]
    nwin = L - K + 1
    workload = (f"{args.config}: {'31mer' if kw == 1 else '127mer'} build K={K}, {2 * cfg_d['n_pairs']} synthetic "
                f"{L}bp PE reads from {cfg_d['n_transcripts']} transcripts (seed {cfg_d['seed']})")
    sample_pairs = min(args.cpu_sample_pairs, cfg_d["n_pairs"])
    sample_desc = f"first {2 * sample_pairs} reads of the workload ({2 * sample_pairs * nwin} instances), FASTA f1/f2"

    # ------------------------------------------------------------------ reference arm
    if args.impl == "reference":
        if rank != 0:
            return
        threads = ref_threads()
        reads = host_sample(cfg_d, sample_pairs)
        vals = []
        for i in range(args.warmup + args.steps):
            info = reference_run(cfg_d, reads, threads)
            if i >= args.warmup:
                vals.append(info["count_sum"] / info["seconds"])
        v = float(np.mean(vals))
        sample = f"{sample_desc} via the reference's own parser per step, -p {threads}"
        print(json.dumps({
            "impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * 2 * sample_pairs * nwin / v, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "u64", "data": "synthetic",
            "config": {"workload": workload},
            "cpu_baseline": {"value": v, "unit": UNIT, "cores": threads, "kind": "reference", "sample": sample},
            "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        }))
        return

    # ------------------------------------------------------------------ our arm
    import torch
    import torch.distributed as dist
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    real_stdout = None
    if world > 1:
        # stdout carries ONE JSON line; what libraries write to file descriptor 1 while the job runs (NCCL's
        # version banner at communicator creation) goes to stderr instead
        sys.stdout.flush()
        real_stdout = os.dup(1)
        os.dup2(2, 1)
        dist.init_process_group("nccl", device_id=dev)
    hbm_gbs, peak_src = load_peaks()

    # per-rank shard of the workload (weak scaling: the config's reads PER GPU)
    n_pairs = cfg_d["n_pairs"]
    first_pair = rank * n_pairs
    n_reads = 2 * n_pairs
    stride = synth.stride_bytes(L)
    tr = synth.make_transcriptome(cfg_d["n_transcripts"], cfg_d["seed"], hot=cfg_d["hot"])
    tr_dev = dict(bases=torch.from_numpy(tr.bases).to(dev), starts=torch.from_numpy(tr.starts.astype(np.int64)).to(dev),
                  lengths=torch.from_numpy(tr.lengths.astype(np.int32)).to(dev),
                  cum=torch.from_numpy(tr.cum.astype(np.int64)).to(dev), n=len(tr.lengths))
    d_packed = torch.empty((n_reads, stride), dtype=torch.uint8, device=dev)
    pkg.pregraph.synth_reads_device(tr_dev, cfg_d["seed"], first_pair, n_pairs, L, stride, d_packed, device=local_rank)
    torch.cuda.synchronize()
    instances_rank = n_reads * nwin
    batch = args.batch_reads

    def push_all(gg):
        for a in range(0, n_reads, batch):
            b = min(a + batch, n_reads)
            gg.push_reads(d_packed[a:b], None, None, n_reads=b - a, uniform_len=L, stride_bytes=stride,
                          first_read_ordinal=2 * first_pair + a, device=True)

    # ---- untimed: the fingerprint of the single-pass insert's table on this workload (one GPU)
    parity = None
    direct_fp = None
    if sliced and world == 1 and not args.no_parity:
        free_b, _ = torch.cuda.mem_get_info()
        est = estimate_distinct(instances_rank, K)
        slot_b = 64 if K > 63 else 32
        if free_b > max(est / 0.85, min(2 * est, (60 << 30) / slot_b)) * slot_b + (4 << 30):
            with pkg.PregraphGPU(K, kw, L, capacity_hint=est, device=local_rank) as gd:
                push_all(gd)
                gd.sync()
                direct_fp = gd.table_checksum().tolist()
        else:
            parity = "skipped: no room for the single-pass insert's table beside the reads"

    # the handle that is measured: no hint on one GPU; on several the closed-form estimate (identical on all ranks)
    if args.hint >= 0:
        hint = args.hint
    elif sliced and world == 1:
        hint = 0
    else:
        hint = estimate_distinct(instances_rank, K)
    g = pkg.PregraphGPU(K, kw, L, capacity_hint=hint, device=local_rank, sliced=sliced)
    ext = torch.cuda.ExternalStream(g.stream, device=dev)

    exch, exch_kind = None, None
    if world > 1:
        from soapdenovo_trans_b200.exchange import Exchange, ReplicatedReads, SkmExchange
        if sliced:
            native = args.skm_exchange == "native"
            if native:      # the library's own NCCL binding; if ANY rank cannot set it up, all ranks drive the same exchange over torch.distributed
                try:
                    exch = SkmExchange(pkg, g, world, rank, dev, native=True)
                    ok = torch.ones(1, dtype=torch.int32, device=dev)
                except Exception as e:      # noqa: BLE001
                    print(f"[bench] rank {rank}: native exchange unavailable ({e}); using torch.distributed", file=sys.stderr)
                    exch, ok = None, torch.zeros(1, dtype=torch.int32, device=dev)
                dist.all_reduce(ok, op=dist.ReduceOp.MIN)
                if int(ok.item()) == 0:
                    if exch is not None and exch.comm is not None:
                        exch.comm.close()
                    exch, native = None, False
                    args.skm_exchange = "torch"
            if exch is None:
                exch = SkmExchange(pkg, g, world, rank, dev, native=False)
            exch_kind = "skm"
        elif args.exchange == "records":
            exch = Exchange(pkg, g, world, rank, dev, max_round_instances=min(batch, n_reads) * nwin)
        else:
            exch = ReplicatedReads(pkg, g, world, rank, dev, max_round_reads=min(batch, n_reads), stride=stride)

    host_t = {"reset": 0.0, "push": 0.0, "flush": 0.0, "sync": 0.0, "n": 0}
    step_calls = []
    step_wall, step_events = [], []       # per step: wall clock; [epochs emitted again, device allocations (both cumulative), retried items, work items]

    def one_step(gg):
        t0 = time.perf_counter()
        gg.reset()
        t1 = time.perf_counter()
        if exch is None:
            push_all(gg)
            t2 = t3 = time.perf_counter()
        else:
            for a in range(0, n_reads, batch):
                b = min(a + batch, n_reads)
                exch.round(gg, d_packed[a:b], b - a, L, stride, 2 * first_pair + a)
            t2 = time.perf_counter()
            exch.flush(gg)
            t3 = time.perf_counter()
        gg.sync()      # end of the step: everything pushed is in the table
        t4 = time.perf_counter()
        for k, v in zip(("reset", "push", "flush", "sync"), (t1 - t0, t2 - t1, t3 - t2, t4 - t3)):
            host_t[k] += 1e3 * v
        host_t["n"] += 1
        step_wall.append(round(1e3 * (t4 - t0), 2))
        step_calls.append([round(1e3 * v, 2) for v in (t1 - t0, t2 - t1, t3 - t2, t4 - t3)])      # reset, push, flush, sync
        if sliced:
            geo_s = gg.slice_geometry()
            ph_s = gg.phase_times(reset=False)      # cumulative kernel times per phase: the difference between two steps tells which phase an outlier sat in
            step_events.append([geo_s["epochs_emitted_again"], geo_s["device_allocations"], geo_s["retried_items"], geo_s["work_items"],
                                {k: round(v[0], 1) for k, v in ph_s.items() if v[0]}])

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    barrier()        # (the first barrier of a process group sets up its communicator: before the warm-up, not next to the timed region)
    for _ in range(args.warmup):
        one_step(g)
    barrier()
    if direct_fp is not None:
        if args.warmup == 0:
            one_step(g)
        sliced_fp = g.table_checksum().tolist()
        parity = sliced_fp == direct_fp
        assert parity, ("the sliced build's table differs from the single-pass insert's", sliced_fp, direct_fp)
    g.kernel_time(reset=True)
    for k in host_t:
        host_t[k] = 0
    step_wall.clear()
    step_events.clear()
    step_calls.clear()
    if exch is not None and hasattr(exch, "collective_ms"):
        exch.collective_ms = 0.0
        exch.host_ms = {}
        exch.host_log = []
    sampler = ClockSampler(local_rank if rank == 0 else -1)
    sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record(ext)
    for _ in range(args.steps):
        one_step(g)
    e1.record(ext)
    barrier()
    sampler.stop_flag.set()
    sampler.join()
    ms = e0.elapsed_time(e1)
    step_wall_timed = list(step_wall)       # host wall clock of every timed step (this rank): an outlier shows here
    step_events_timed = list(step_events)
    exch_log_timed = list(getattr(exch, "host_log", []) or [])      # per timed step: [bound, stage, exchange, import] ms on the host
    if os.environ.get("BENCH_STEP_LOG"):     # diagnosis of outlier steps: every rank leaves its own per-step record
        with open(os.path.join(os.environ["BENCH_STEP_LOG"], f"steps_rank{rank}.json"), "w") as f:
            json.dump({"rank": rank, "step_wall_ms": step_wall_timed, "host_calls_ms": step_calls, "exchange_host_ms": exch_log_timed,
                       "events": [e[:4] for e in step_events_timed]}, f)
    host_ms = {k: v / max(host_t["n"], 1) for k, v in host_t.items() if k != "n"}      # wall clock of the host calls of a timed step (this rank)
    st = g.stats()
    distinct = int(st.n_nodes)
    assert exch is not None or st.n_instances == instances_rank, (st.n_instances, instances_rank)
    phases = g.phase_times(reset=False)
    insert_ms, insert_launches, all_launches = g.kernel_time(reset=True)
    t = torch.tensor([ms, float(st.n_instances), float(st.n_nodes), float(getattr(exch, "collective_ms", 0.0))], dtype=torch.float64, device=dev)
    if world > 1:
        tmax = t.clone()
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        tsum = t.clone()
        dist.all_reduce(tsum, op=dist.ReduceOp.SUM)
        ms, total_instances, total_nodes = float(tmax[0]), float(tsum[1]), float(tsum[2])
        collective_ms = float(tmax[3]) / args.steps
        assert total_instances == instances_rank * world, (total_instances, instances_rank * world)
    else:
        total_instances, total_nodes, collective_ms = float(st.n_instances), float(st.n_nodes), None
    ms_per_step = ms / args.steps
    value = total_instances / (ms_per_step * 1e-3)
    bpi = BYTES_PER_INSTANCE[st.device_key_words]
    slot_b = 64 if st.device_key_words == 4 else 32
    sliced_info = None
    if sliced:
        # The insert is a pipeline of streaming kernels (super-k-mer emit into chains, merge, build); the SURVEY figure
        # of 64 (96) algorithmic bytes per instance belongs to the whole insert, so `achieved` is taken over the SUM of
        # their CUDA-event times (all on the handle's stream).  Each phase's own DRAM stream (bytes it must read + write
        # per instance) is reported beside it.
        geo = g.slice_geometry()
        rec_b = geo["record_bytes"] * geo["n_records"] / max(st.n_instances, 1)      # record bytes per instance
        mrg_b = geo["record_bytes"] * geo["n_records_merged"] / max(st.n_instances, 1)
        read_b = stride / nwin
        node_b = st.n_nodes * slot_b / max(st.n_instances, 1)
        stream_b = {"emit": read_b + rec_b, "scatter": 2 * mrg_b if world > 1 else 0.0, "dedupe": rec_b + mrg_b, "build": mrg_b + node_b, "scan": 0.0, "retry": 0.0}
        insert_ms = sum(phases[k][0] for k in stream_b)
        insert_launches = max(phases["build"][1] + phases["retry"][1], 1)
        sliced_info = {"geometry": geo, "windows_per_record": st.n_instances / max(geo["n_records"], 1), "phases": {
            k: {"ms_per_step": phases[k][0] / args.steps, "launches_per_step": phases[k][1] / args.steps,
                "stream_bytes_per_instance": stream_b[k],
                "stream_gbs": (st.n_instances * args.steps * stream_b[k] / max(phases[k][0], 1e-9) / 1e6) if stream_b[k] else None}
            for k in stream_b},
            "phase_names": {"emit": "skm_emit_kernel (reads -> records appended to their slice's chain)", "scatter": "skm_append_kernel (multi-GPU: received records -> chains)",
                            "dedupe": "skm_merge_kernel (copies merged, chains -> work items)", "build": "skm_build_kernel",
                            "scan": "blocks per chain scanned and listed", "retry": "pieces of items that overflowed, skm_split_kernel + sub-slices"}}
        dominant = max(stream_b, key=lambda k: phases[k][0])
        sliced_info["dominant"] = "skm_" + {"dedupe": "merge", "scatter": "append"}.get(dominant, dominant) + "_kernel"
        ker_ms = insert_ms / args.steps                      # one pipeline pass = one "launch" of the insert
        inst_per_launch = float(st.n_instances)
    else:
        ker_ms = max(insert_ms, 1e-9) / max(insert_launches, 1)
        inst_per_launch = st.n_instances * args.steps / max(insert_launches, 1)
    achieved = inst_per_launch * bpi / (ker_ms * 1e-3) / 1e9
    traffic, traffic_src = None, None      # DRAM bytes per launch, from the committed ncu capture of this path on this config
    tp = os.path.join(ROOT, "profiles", "r2_traffic_sliced.json" if sliced else "r1_traffic.json")
    if os.path.exists(tp) and world == 1:
        with open(tp) as f:
            tj = json.load(f)
        if tj.get("key_words") == st.device_key_words:
            traffic = tj["dram_bytes_per_instance"] * inst_per_launch
            traffic_src = tj.get("source")
    if args.dump_outputs:      # before e2e, which empties the handle again
        shapes = dump_outputs(pkg, g, args.dump_outputs)
        print(f"[bench] outputs of the last timed step written to {args.dump_outputs}: {shapes}", file=sys.stderr)

    # ---- e2e: HOST (pinned) buffers, H2D inside the timed region, counters read back (D2H) every step.
    # N = 1: straight through the C ABI's host entry point (sdtgpu_push_reads).  N > 1: every rank
    # copies its round's reads from pinned host memory, then emit -> merge -> exchange -> build as above.
    e2e = None
    if not args.no_e2e:
        if sliced and world == 1 and hint == 0:
            # a caller that streams reads from the host knows how many it is going to push: with the closed-form hint for
            # that number (no pass over the data) the records are made while the next batch is copied
            g.close()
            g = pkg.PregraphGPU(K, kw, L, capacity_hint=estimate_distinct(instances_rank, K), device=local_rank, sliced=True)
        h_packed = torch.empty((n_reads, stride), dtype=torch.uint8).pin_memory()
        h_packed.copy_(d_packed)
        torch.cuda.synchronize()
        d_round = [torch.empty((min(batch, n_reads), stride), dtype=torch.uint8, device=dev) for _ in range(2)] if exch is not None else None

        def e2e_step():
            g.reset()
            for i, a in enumerate(range(0, n_reads, batch)):
                b = min(a + batch, n_reads)
                if exch is None:
                    g.push_reads(h_packed[a:b], None, None, n_reads=b - a, uniform_len=L, stride_bytes=stride,
                                 first_read_ordinal=a)
                else:
                    buf = d_round[i & 1]
                    with torch.cuda.stream(exch.aux):
                        exch.aux.wait_event(exch.inserted[exch.r & 1])      # same buffer parity as the exchange
                        buf[: b - a].copy_(h_packed[a:b], non_blocking=True)
                    exch.round(g, buf, b - a, L, stride, 2 * first_pair + a)
            if exch is not None:
                exch.flush(g)
            g.sync()
            return g.stats()
        e2e_step()
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            s2 = e2e_step()
        barrier()
        dt = (time.perf_counter() - t0) / args.steps
        assert exch is not None or (s2.n_instances == instances_rank and s2.n_nodes == distinct)
        tt = torch.tensor([dt, float(s2.n_instances)], dtype=torch.float64, device=dev)
        if world > 1:
            tm = tt.clone(); dist.all_reduce(tm, op=dist.ReduceOp.MAX)
            ts = tt.clone(); dist.all_reduce(ts, op=dist.ReduceOp.SUM)
            dt, e2e_inst = float(tm[0]), float(ts[1])
        else:
            e2e_inst = float(s2.n_instances)
        e2e = {"value": e2e_inst / dt, "unit": UNIT, "h2d_bytes_per_step": int(n_reads * stride) * world,
               "d2h_bytes_per_step": 2120 * world, "ms_per_step": dt * 1e3,
               "capacity_hint": "closed form from the number of reads to be pushed (instances x (1 - 0.99^K) x 1.05)"}
        del h_packed

    # ---- the reference on a bounded sample, and our whole path FROM FILES on the same sample (like for like)
    cpu, from_files = None, None
    cpu_leg = rank == 0 and world == 1 and not args.no_cpu_baseline
    if cpu_leg and not reference_built(cfg_d):
        print("[bench] cpu_baseline and e2e_from_files skipped: the reference binaries (oracle/_ref) are not built; "
              "oracle/Makefile builds them from the SOAPdenovo-Trans sources (REF=<src>)", file=sys.stderr)
        cpu_leg = False
    if cpu_leg:
        threads = ref_threads()
        sample = unpack_reads(d_packed[: 2 * sample_pairs].cpu().numpy(), L)
        info = reference_run(cfg_d, sample, threads)
        cpu = {"value": info["count_sum"] / info["seconds"], "unit": UNIT, "cores": threads, "kind": "reference",
               "sample": f"{sample_desc} ({info['count_sum']} instances, {info['nodes']} nodes) through the unmodified "
                         f"reference prlRead2HashTable (oracle/_ref), its own parser included, -p {threads}, {info['seconds']:.2f} s"}
        if sliced:
            v, dt, ninst, nnodes = files_e2e(pkg, cfg_d, sample, local_rank, min(batch, 1 << 20))
            assert ninst == info["count_sum"] and nnodes == info["nodes"], (ninst, nnodes, info["count_sum"], info["nodes"])
            from_files = {"same_sample_as_cpu_baseline": {"value": v, "unit": UNIT, "seconds": dt, "instances": ninst, "nodes": nnodes,
                                                          "vs_cpu_baseline": v / cpu["value"], "same_config": True,
                                                          "what": "FASTA f1/f2 on disk -> sdtpack (mmap, parallel parse + 2-bit pack) -> sdtgpu_push_reads -> sdtgpu_get_stats, "
                                                                  "no capacity hint; node and instance counts equal the reference's"}}
        del sample
        if sliced and args.files_full:
            full = unpack_reads(d_packed.cpu().numpy(), L)
            v, dt, ninst, nnodes = files_e2e(pkg, cfg_d, full, local_rank, batch, repeats=1)
            assert ninst == instances_rank and nnodes == distinct
            from_files["whole_workload"] = {"value": v, "unit": UNIT, "seconds": dt, "instances": ninst, "nodes": nnodes}
            del full

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None,
            "dtype": "u64", "data": "synthetic",
            "config": {"workload": workload + (f" per GPU x {world} GPUs, k-mers sharded by slice owner ({('super-k-mer records merged per sender and exchanged over NCCL inside the library (sdtgpu_skm_exchange), one grouped send/recv per step' if args.skm_exchange == 'native' else 'super-k-mer records merged per sender and exchanged over NCCL (torch.distributed), one grouped send/recv per step') if exch_kind == 'skm' else ('packed reads all-gathered over NCCL, every rank inserts the k-mers it owns' if args.exchange != 'records' else 'k-mer records exchanged over NCCL')})" if world > 1 else ""),
                       "instances_per_step": total_instances, "distinct_kmers": total_nodes,
                       "capacity_hint": hint, "hint_source": ("none: sized inside the timed region from the number of windows pushed" if hint == 0 else
                                                              ("closed form, instances x (1 - 0.99^K) x 1.05: no pass over the data" if args.hint < 0 else "--hint")),
                       "node_store_slots_per_gpu": int(st.capacity), "slot_bytes": slot_b,
                       "batch_reads": batch, "insert_path": args.path,
                       "l2": "reads, records and node store are far larger than the 126 MB L2; the table is rebuilt from empty every step"},
            "parity_checked": parity,
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": hbm_gbs, "unit": "GB/s", "frac": achieved / hbm_gbs,
                         "traffic": traffic, "traffic_source": traffic_src,
                         "kernel": ("skm_emit + skm_merge + skm_build kernels (the sliced insert pipeline; times summed)" if sliced else "insert_reads_kernel") if (world == 1 or sliced or args.exchange == "reads") else "insert_records_kernel",
                         "path": args.path, "sliced": sliced_info,
                         "bytes_per_instance": bpi, "kernel_ms_per_launch": ker_ms, "peak_source": peak_src,
                         "random_access": {"cold_line_requests_per_s_measured": RANDOM_REQUESTS_PER_S,
                                           "min_requests_per_instance": MIN_REQUESTS_PER_INSTANCE[st.device_key_words],
                                           "ceiling_instances_per_s_per_gpu": RANDOM_REQUESTS_PER_S / MIN_REQUESTS_PER_INSTANCE[st.device_key_words],
                                           "frac_of_ceiling": (inst_per_launch / (ker_ms * 1e-3)) / (RANDOM_REQUESTS_PER_S / MIN_REQUESTS_PER_INSTANCE[st.device_key_words]),
                                           "source": "tools/randacc_bench.cu, profiles/r1_randacc_bench.txt"}},
            "host_call_ms_per_step_rank0": host_ms, "step_wall_ms_rank0": step_wall_timed, "step_events_rank0": step_events_timed,
            "exchange_host_ms_steps_rank0": exch_log_timed or None,
            "collective_ms_per_step": collective_ms,
            "exchange_host_ms_per_step_rank0": ({k: v / max(exch.host_ms.get("flushes", 1), 1) for k, v in exch.host_ms.items() if k != "flushes"} if exch is not None and getattr(exch, "host_ms", None) else None),
            "cpu_baseline": cpu, "e2e": e2e, "e2e_from_files": from_files, "gpu_launches": int(all_launches),
            "clocks": sampler.summary(),
        }
        sys.stdout.flush()
        if real_stdout is not None:
            os.dup2(real_stdout, 1)
        print(json.dumps(line), flush=True)
    # orderly teardown: everything that was enqueued on the handle's streams is done, torch's views of the
    # streams and the library's buffers go first, then the handle (which owns the streams), then NCCL
    torch.cuda.synchronize()
    del ext
    exch = None
    g.close()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    sys.stdout.flush()


if __name__ == "__main__":
    main()
