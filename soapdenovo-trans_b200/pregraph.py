"""ctypes binding of libsdtgpu.so (include/sdtgpu.h) — the same entry points the reference's C
driver binds (INTEGRATION.md).  Method names follow the C ABI, which in turn names the reference
functions each call replaces (prlRead2HashTable's flush sites, deLowCov, Mark1in1outNode, ...).

No CPU fallback: a missing library or a failing CUDA call raises SdtGpuError.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

PKG_DIR = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(PKG_DIR, "libsdtgpu.so")

NODE_DTYPE = np.dtype([("key", "<u8", (4,)), ("l_links", "<u4"), ("rword", "<u4"), ("count", "<u4"),
                       ("set", "<u4"), ("ordinal", "<u8")])
assert NODE_DTYPE.itemsize == 56
# sdtgpu_hit: one lookup result (include/sdtgpu.h); status holds the HIT_* bits
HIT_DTYPE = np.dtype([("count", "<u4"), ("l_links", "<u4"), ("rword", "<u4"), ("status", "<u4")])
assert HIT_DTYPE.itemsize == 16
HIT_WINDOW, HIT_FOUND, HIT_RC = 1, 2, 4
# sdtgpu_edge: one edge or cycle of PregraphGPU.edges() (include/sdtgpu.h); seq counts bases into the sequence buffer
EDGE_DTYPE = np.dtype([("seq", "<u8"), ("length", "<u4"), ("flags", "<u4"), ("count_sum", "<u8"), ("link", "<u4"),
                       ("unused", "<u4")])
assert EDGE_DTYPE.itemsize == 32
EDGE_PALINDROME, EDGE_CYCLE = 1, 2
# sdtgpu_step: the step of one read window on the edges (include/sdtgpu.h); pos = index << 1 | strand, all ones = none
STEP_DTYPE = np.dtype([("record", "<u4"), ("pos", "<u4")])
assert STEP_DTYPE.itemsize == 8
STEP_NONE = 0xFFFFFFFF
# sdtgpu_arc: reads crossing a vertex from one record to the next; from / to = record << 1 | strand
ARC_DTYPE = np.dtype([("from", "<u4"), ("to", "<u4"), ("count", "<u4"), ("unused", "<u4")])
assert ARC_DTYPE.itemsize == 16
EDGE_COUNTS = ("edges", "palindromes", "cycles", "bases", "vertices", "linear_on_edges", "linear_on_cycles", "dangling")
# sdtgpu_prune's out[] and flags (include/sdtgpu.h)
PRUNE_COUNTS = ("minor_branches", "single_tips", "minor_tips", "tips", "rounds", "live", "linear", "vertices")
PRUNE_SINGLE_TIPS, PRUNE_MINOR_TIPS = 1, 2

F_NKMER = 1
F_SLICED = 4
PHASES = ("insert", "emit", "scatter", "dedupe", "build", "scan", "retry", "-")
_ERR = {1: "EINVAL", 2: "ECUDA", 3: "ENOMEM", 4: "ERANGE", 5: "ESTATE"}


class SdtGpuError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"sdtgpu error {code} ({_ERR.get(code, '?')}): {msg}")
        self.code = code


class Stats(C.Structure):
    _fields_ = [("n_instances", C.c_uint64), ("n_nodes", C.c_uint64), ("n_removed", C.c_uint64),
                ("n_linear", C.c_uint64), ("capacity", C.c_uint64), ("n_reads", C.c_uint64),
                ("n_grows", C.c_uint32), ("device_key_words", C.c_uint32)]


class KmerSet(C.Structure):
    """inc/newhash.h:79-88"""
    _fields_ = [("array", C.c_void_p), ("flags", C.POINTER(C.c_uint32)), ("size", C.c_uint64),
                ("count", C.c_uint64), ("max", C.c_uint64), ("load_factor", C.c_double), ("iter_ptr", C.c_uint64)]


def build_library(force: bool = False) -> str:
    """Compiles csrc/ + host/ for sm_100a into libsdtgpu.so (in-tree, so it travels to the GPU box)."""
    srcs = [os.path.join(PKG_DIR, p) for p in ("csrc/sdtgpu.cu", "csrc/sdt_synth.cu", "csrc/sdt_device.cuh",
                                               "csrc/sdt_kernels.cuh", "csrc/sdt_sliced.cuh", "csrc/sdt_skm.cuh", "csrc/sdt_build.cuh", "csrc/sdt_lookup.cuh", "csrc/sdt_route.cuh", "csrc/sdt_edges.cuh", "csrc/sdt_paths.cuh", "csrc/sdt_prune.cuh", "csrc/sdt_nccl.cu", "csrc/sdt_parse.cu", "host/kmerset_builder.cpp", "host/sdt_readpack.c", "../include/sdtpack.h",
                                               "../include/sdtgpu.h")]
    stale = (not os.path.exists(LIB_PATH)) or any(os.path.getmtime(s) > os.path.getmtime(LIB_PATH) for s in srcs)
    if force or stale:
        subprocess.check_call(["make", "-s", "-C", PKG_DIR, "libsdtgpu.so"])
    return LIB_PATH


_lib = None


def library() -> C.CDLL:
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise SdtGpuError(2, f"{LIB_PATH} is missing: run __graft_entry__.build() (there is no CPU fallback)")
    L = C.CDLL(LIB_PATH)
    vp, u64, u32, i32 = C.c_void_p, C.c_uint64, C.c_uint32, C.c_int
    L.sdtgpu_version.restype = i32
    L.sdtgpu_hash_kmer.restype = u64
    L.sdtgpu_hash_kmer.argtypes = [vp, i32]
    L.sdtgpu_last_error.restype = C.c_char_p
    L.sdtgpu_last_error.argtypes = [vp]
    L.sdtgpu_create.argtypes = [C.POINTER(vp), i32, i32, i32, i32, u64, C.c_uint]
    L.sdtgpu_destroy.argtypes = [vp]
    L.sdtgpu_destroy.restype = None
    L.sdtgpu_reset.argtypes = [vp]
    L.sdtgpu_sync.argtypes = [vp]
    L.sdtgpu_push_reads.argtypes = [vp, vp, vp, vp, u64, u32, u32, u64]
    L.sdtgpu_push_reads_device.argtypes = [vp, vp, vp, vp, u64, u32, u32, u64]
    L.sdtgpu_set_owner.argtypes = [vp, i32, i32]
    L.sdtgpu_skm_set_world.argtypes = [vp, i32, i32]
    L.sdtgpu_skm_stage.argtypes = [vp, C.POINTER(vp), C.POINTER(u64), C.POINTER(u64)]
    L.sdtgpu_skm_set_ordinal_bound.argtypes = [vp, u64]
    L.sdtgpu_skm_import_buffer.argtypes = [vp, u64, C.POINTER(vp)]
    L.sdtgpu_skm_import.argtypes = [vp, u64]
    L.sdtgpu_comm_unique_id.argtypes = [vp]
    L.sdtgpu_comm_create.argtypes = [C.POINTER(vp), i32, vp, i32, i32]
    L.sdtgpu_comm_destroy.argtypes = [vp]
    L.sdtgpu_comm_last_error.restype = C.c_char_p
    L.sdtgpu_comm_last_error.argtypes = [vp]
    L.sdtgpu_skm_exchange.argtypes = [vp, vp, u64, C.POINTER(u64), C.POINTER(C.c_double)]
    L.sdtgpu_record_bytes.restype = C.c_size_t
    L.sdtgpu_record_bytes.argtypes = [vp]
    L.sdtgpu_bucket_reads_device.argtypes = [vp, vp, vp, vp, u64, u32, u32, u64, i32, vp, u64, vp]
    L.sdtgpu_insert_records_device.argtypes = [vp, vp, u64]
    L.sdtgpu_finalize.argtypes = [vp, i32, vp, C.POINTER(Stats)]
    L.sdtgpu_get_stats.argtypes = [vp, C.POINTER(Stats)]
    L.sdtgpu_export_count.argtypes = [vp, C.POINTER(u64)]
    L.sdtgpu_export_nodes.argtypes = [vp, i32, i32, vp, u64, C.POINTER(u64)]
    L.sdtgpu_export_kmersets.argtypes = [vp, i32, C.POINTER(C.POINTER(KmerSet))]
    L.sdtgpu_build_kmersets.argtypes = [vp, u64, i32, i32, vp, C.POINTER(C.POINTER(KmerSet))]
    L.sdtgpu_free_kmersets.argtypes = [C.POINTER(C.POINTER(KmerSet)), i32]
    L.sdtgpu_free_kmersets.restype = None
    L.sdtgpu_stream.restype = vp
    L.sdtgpu_stream.argtypes = [vp]
    L.sdtgpu_aux_stream.restype = vp
    L.sdtgpu_aux_stream.argtypes = [vp]
    L.sdtgpu_kernel_time.argtypes = [vp, i32, C.POINTER(C.c_double), C.POINTER(u64), C.POINTER(u64)]
    L.sdtgpu_table_checksum.argtypes = [vp, vp]
    L.sdtgpu_lookup_kmers_device.argtypes = [vp, vp, u64, vp]
    L.sdtgpu_lookup_reads_device.argtypes = [vp, vp, vp, vp, u64, u32, u32, vp]
    L.sdtgpu_lookup_route.argtypes = [vp, vp]
    L.sdtgpu_lookup_stage_kmers.argtypes = [vp, vp, u64, C.POINTER(vp), vp, vp]
    L.sdtgpu_lookup_stage_reads.argtypes = [vp, vp, vp, vp, u64, u32, u32, C.POINTER(vp), vp, vp]
    L.sdtgpu_lookup_answer_buffer.argtypes = [vp, u64, C.POINTER(vp), C.POINTER(vp)]
    L.sdtgpu_lookup_answer.argtypes = [vp, u64]
    L.sdtgpu_lookup_unstage_buffer.argtypes = [vp, C.POINTER(vp)]
    L.sdtgpu_lookup_unstage.argtypes = [vp, vp]
    L.sdtgpu_lookup_kmers_exchange.argtypes = [vp, vp, vp, u64, vp, C.POINTER(C.c_double)]
    L.sdtgpu_lookup_reads_exchange.argtypes = [vp, vp, vp, vp, vp, u64, u32, u32, vp, C.POINTER(C.c_double)]
    L.sdtgpu_edges_build.argtypes = [vp, vp, C.POINTER(C.c_double)]
    L.sdtgpu_edges_buffers.argtypes = [vp, C.POINTER(vp), C.POINTER(vp)]
    L.sdtgpu_edges_map_reads.argtypes = [vp, vp, vp, vp, u64, u32, u32, vp, i32]
    L.sdtgpu_arcs_build.argtypes = [vp, C.POINTER(u64), C.POINTER(C.c_double)]
    L.sdtgpu_arcs_buffers.argtypes = [vp, C.POINTER(vp)]
    L.sdtgpu_arcs_clear.argtypes = [vp]
    L.sdtgpu_prune.argtypes = [vp, i32, C.c_uint, C.POINTER(u64), C.POINTER(C.c_double)]
    L.sdtgpu_last_ordinals.argtypes = [vp, i32, vp]
    L.sdtgpu_kernel_times.argtypes = [vp, i32, C.POINTER(C.c_double), C.POINTER(u64)]
    L.sdtgpu_phase_times.argtypes = [vp, i32, C.POINTER(C.c_double), C.POINTER(u64)]
    L.sdtgpu_slice_geometry.argtypes = [vp, C.POINTER(u64)]
    L.sdtgpu_debug_prof.argtypes = [C.POINTER(u64), i32]
    L.sdtpack_open.argtypes = [C.POINTER(vp), C.c_char_p, C.c_char_p, i32, i32]
    L.sdtpack_next.restype = C.c_int64
    L.sdtpack_next.argtypes = [vp, i32, i32, i32, vp, vp, vp, u64, u32]
    L.sdtpack_close.argtypes = [vp]
    L.sdtpack_close.restype = None
    L.sdtgpu_synth_reads_device.argtypes = [i32, vp, vp, vp, vp, vp, u32, u64, u64, u64, u32, u32, vp]
    L.sdtgpu_reader_open.argtypes = [C.POINTER(vp), i32, C.c_char_p, C.c_char_p, i32, u64]
    L.sdtgpu_reader_next.argtypes = [vp, vp, i32, i32, i32, vp, vp, vp, u64, u32, C.POINTER(u64)]
    L.sdtgpu_reader_stats.argtypes = [vp, C.POINTER(u64)]
    L.sdtgpu_reader_last_error.restype = C.c_char_p
    L.sdtgpu_reader_last_error.argtypes = [vp]
    L.sdtgpu_reader_close.argtypes = [vp]
    L.sdtgpu_reader_close.restype = None
    L.sdtgpu_reader_open_shard.argtypes = [C.POINTER(vp), i32, C.c_char_p, C.c_char_p, i32, u64, i32, i32]
    L.sdtgpu_reader_summary.argtypes = [vp, vp]
    L.sdtgpu_reader_plan.argtypes = [vp, vp, vp]
    L.sdtgpu_reader_tell.argtypes = [vp, C.POINTER(u64)]
    L.sdtgpu_reader_plan_exchange.argtypes = [vp, vp, vp]
    _lib = L
    return L


def debug_prof(reset: bool = True):
    """Phase clocks of the slice build kernel (SM cycles summed over the groups' first threads)."""
    out = (C.c_uint64 * 8)()
    library().sdtgpu_debug_prof(out, int(reset))
    names = ("prepare", "wait_image", "insert", "compact", "items", "chunks")
    return {n: int(out[i]) for i, n in enumerate(names)}


def hash_kmer(key_words4, key_words: int) -> int:
    """hashFunction.c:108 through the product library's own restatement."""
    k = (C.c_uint64 * 4)(*[int(x) for x in key_words4])
    return int(library().sdtgpu_hash_kmer(k, key_words))


def _ptr(x) -> int | None:
    """Host numpy array -> address; torch tensor -> data_ptr; int passthrough; None -> NULL."""
    if x is None:
        return None
    if isinstance(x, int):
        return x
    if isinstance(x, np.ndarray):
        assert x.flags["C_CONTIGUOUS"]
        return x.ctypes.data
    return x.data_ptr()


def hits_numpy(hits) -> np.ndarray:
    """Hits as returned by PregraphGPU.lookup_* on the device (int32 [..., 4]) -> a HIT_DTYPE array of shape [...]."""
    a = np.ascontiguousarray(hits.cpu().numpy() if hasattr(hits, "cpu") else hits).view(np.uint32)
    return a.view(HIT_DTYPE)[..., 0]


def steps_numpy(steps) -> np.ndarray:
    """Steps as returned by PregraphGPU.map_reads (int32 [..., 2]) -> int64 [..., 3] of (record, index, strand),
    all three -1 where the window's (K+1)-mer is not a step of the graph."""
    a = np.ascontiguousarray(steps.cpu().numpy() if hasattr(steps, "cpu") else steps).view(np.uint32)
    rec, pos = a[..., 0].astype(np.int64), a[..., 1].astype(np.int64)
    none = rec == STEP_NONE
    out = np.stack([rec, pos >> 1, pos & 1], axis=-1)
    out[none] = -1
    return out


def edge_codes(edges: np.ndarray, seq: np.ndarray, i: int, K: int) -> np.ndarray:
    """Base codes (uint8, A=0 C=1 T=2 G=3) of edge i of PregraphGPU.edges(): m + K bases, m + K - 1 for a cycle."""
    e = edges[i]
    n = int(e["length"]) + K - (1 if int(e["flags"]) & EDGE_CYCLE else 0)
    a = int(e["seq"]) // 4
    raw = seq[a: a + (n + 3) // 4]
    return (raw[:, None] >> np.array([6, 4, 2, 0], dtype=np.uint8) & 3).reshape(-1)[:n]


class _DeviceBytes:
    """A device buffer owned by the library, seen by torch through __cuda_array_interface__ (no copy)."""

    def __init__(self, ptr: int, nbytes: int):
        self.__cuda_array_interface__ = {"shape": (nbytes,), "typestr": "|u1", "data": (ptr, False), "version": 2}


def _device_bytes(ptr: int, nbytes: int, dev):
    import torch
    return torch.as_tensor(_DeviceBytes(ptr, nbytes), device=dev)


def node_bytes(key_words: int) -> int:
    return {1: 24, 2: 32, 4: 48}[key_words]


def read_kmersets(sets, thrd_num: int, key_words: int):
    """Decodes reference-layout KmerSets (as handed back by export_kmersets) into the oracle's
    64-byte dump records in (set, slot) order plus (size, count, max) per set."""
    from_dtype = np.dtype([("key", "<u8", (key_words,)), ("l_links", "<u4"), ("rword", "<u4"), ("count", "<u4")]
                          + ([("pad", "<u4")] if node_bytes(key_words) > 8 * key_words + 12 else []))
    assert from_dtype.itemsize == node_bytes(key_words)
    rec_dtype = np.dtype([("set", "<u4"), ("pad0", "<u4"), ("slot", "<u8"), ("key", "<u8", (4,)),
                          ("l_links", "<u4"), ("rword", "<u4"), ("count", "<u4"), ("pad1", "<u4")])
    out, info = [], np.zeros((thrd_num, 3), dtype=np.uint64)
    for t in range(thrd_num):
        s = sets[t].contents
        info[t] = (s.size, s.count, s.max)
        nwords = (s.size + 15) // 16
        flags = np.ctypeslib.as_array(s.flags, shape=(nwords,))
        slots = np.arange(s.size, dtype=np.int64)
        null = (flags[slots >> 4] >> ((slots & 15) << 1).astype(np.uint32)) & 1	# is_kmer_entity_null, newhash.h:47
        occ = np.nonzero(null == 0)[0]
        arr = np.ctypeslib.as_array(C.cast(s.array, C.POINTER(C.c_uint8)), shape=(s.size * from_dtype.itemsize,)).view(from_dtype)
        rec = np.zeros(len(occ), dtype=rec_dtype)
        rec["set"] = t
        rec["slot"] = occ
        rec["key"][:, 4 - key_words:] = arr["key"][occ]
        rec["l_links"], rec["rword"], rec["count"] = arr["l_links"][occ], arr["rword"][occ], arr["count"][occ]
        out.append(rec)
    return np.concatenate(out) if out else np.zeros(0, dtype=rec_dtype), info


def nodes_to_records(nodes: np.ndarray) -> np.ndarray:
    """Order-free multiset view (key, count, l_links, rword) sorted by key — comparable with
    oracle.sorted_multiset()."""
    m = np.zeros(len(nodes), dtype=[("key", "<u8", (4,)), ("count", "<u4"), ("l_links", "<u4"), ("rword", "<u4")])
    m["key"], m["count"], m["l_links"], m["rword"] = nodes["key"], nodes["count"], nodes["l_links"], nodes["rword"]
    order = np.lexsort((nodes["key"][:, 3], nodes["key"][:, 2], nodes["key"][:, 1], nodes["key"][:, 0]))
    return m[order]


class PregraphGPU:
    """One GPU's k-mer table: the device replacement of the reference's KmerSets for the hashing
    stage of `pregraph` (prlRead2HashTable, prlHashReads.c:338)."""

    def __init__(self, K: int, key_words: int, max_read_len: int, capacity_hint: int = 0, device: int = 0,
                 n_kmer: bool = False, sliced: bool = False):
        self.L = library()
        self.h = C.c_void_p()
        self.K, self.key_words, self.max_read_len, self.device = K, key_words, max_read_len, device
        rc = self.L.sdtgpu_create(C.byref(self.h), device, K, key_words, max_read_len, capacity_hint,
                                  (F_NKMER if n_kmer else 0) | (F_SLICED if sliced else 0))
        if rc:
            raise SdtGpuError(rc, self.L.sdtgpu_last_error(None).decode())

    def _ck(self, rc: int):
        if rc:
            raise SdtGpuError(rc, self.L.sdtgpu_last_error(self.h).decode())

    def close(self):
        if getattr(self, "h", None):
            self.L.sdtgpu_destroy(self.h)
            self.h = None

    __del__ = close

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def reset(self):
        self._ck(self.L.sdtgpu_reset(self.h))

    def sync(self):
        self._ck(self.L.sdtgpu_sync(self.h))

    @property
    def stream(self) -> int:
        return int(self.L.sdtgpu_stream(self.h) or 0)

    @property
    def aux_stream(self) -> int:
        return int(self.L.sdtgpu_aux_stream(self.h) or 0)

    def push_reads(self, packed, lens=None, nmask=None, n_reads=None, uniform_len=0, stride_bytes=None,
                   first_read_ordinal=0, device=False):
        """HOST buffers (numpy / pinned torch CPU tensors) unless device=True (CUDA pointers)."""
        if n_reads is None:
            n_reads = packed.shape[0]
        if stride_bytes is None:
            stride_bytes = packed.shape[1]
        fn = self.L.sdtgpu_push_reads_device if device else self.L.sdtgpu_push_reads
        self._ck(fn(self.h, _ptr(packed), _ptr(lens), _ptr(nmask), n_reads, uniform_len, stride_bytes, first_read_ordinal))

    def set_owner(self, rank: int, n_ranks: int):
        self._ck(self.L.sdtgpu_set_owner(self.h, rank, n_ranks))

    # ---- super-k-mer exchange (multi-GPU sliced build; include/sdtgpu.h)
    def skm_set_world(self, rank: int, world: int):
        self._ck(self.L.sdtgpu_skm_set_world(self.h, rank, world))
        self._skm_world = world

    def skm_stage(self):
        """-> (device address of the records, starts[world], counts[world] in records): rank r's share."""
        world = getattr(self, "_skm_world", 1)
        ptr, starts, counts = C.c_void_p(), (C.c_uint64 * world)(), (C.c_uint64 * world)()
        self._ck(self.L.sdtgpu_skm_stage(self.h, C.byref(ptr), starts, counts))
        return int(ptr.value or 0), [int(x) for x in starts], [int(x) for x in counts]

    def skm_set_ordinal_bound(self, n_reads_all_ranks: int):
        self._ck(self.L.sdtgpu_skm_set_ordinal_bound(self.h, n_reads_all_ranks))

    def skm_import_buffer(self, n_records: int) -> int:
        ptr = C.c_void_p()
        self._ck(self.L.sdtgpu_skm_import_buffer(self.h, n_records, C.byref(ptr)))
        return int(ptr.value or 0)

    def skm_import(self, n_records: int):
        self._ck(self.L.sdtgpu_skm_import(self.h, n_records))

    def skm_exchange(self, comm: "SkmComm", reads_end: int):
        """include/sdtgpu.h sdtgpu_skm_exchange: the whole exchange of an epoch in one call (NCCL inside the library).
        -> (records received, device ms of the counts + records collectives)."""
        n, ms = C.c_uint64(), C.c_double()
        rc = self.L.sdtgpu_skm_exchange(self.h, comm.c, reads_end, C.byref(n), C.byref(ms))
        if rc:
            raise SdtGpuError(rc, (self.L.sdtgpu_comm_last_error(comm.c) or b"").decode())
        return int(n.value), float(ms.value)

    def record_bytes(self) -> int:
        return int(self.L.sdtgpu_record_bytes(self.h))

    def bucket_reads_device(self, packed, lens, nmask, n_reads, uniform_len, stride_bytes, first_read_ordinal,
                            n_ranks, bins, bin_capacity, counts):
        self._ck(self.L.sdtgpu_bucket_reads_device(self.h, _ptr(packed), _ptr(lens), _ptr(nmask), n_reads, uniform_len,
                                                   stride_bytes, first_read_ordinal, n_ranks, _ptr(bins), bin_capacity,
                                                   _ptr(counts)))

    def insert_records_device(self, records, n_records):
        self._ck(self.L.sdtgpu_insert_records_device(self.h, _ptr(records), n_records))

    def finalize(self, deLowKmer: int = 0):
        freq = np.zeros(257, dtype=np.int64)
        st = Stats()
        self._ck(self.L.sdtgpu_finalize(self.h, deLowKmer, freq.ctypes.data, C.byref(st)))
        return freq, st

    def stats(self) -> Stats:
        st = Stats()
        self._ck(self.L.sdtgpu_get_stats(self.h, C.byref(st)))
        return st

    def table_checksum(self) -> np.ndarray:
        out = np.zeros(4, dtype=np.uint64)
        self._ck(self.L.sdtgpu_table_checksum(self.h, out.ctypes.data))
        return out

    def export_nodes(self, thrd_num: int = 8, sort_by_ordinal: bool = False) -> np.ndarray:
        n = C.c_uint64()
        self._ck(self.L.sdtgpu_export_count(self.h, C.byref(n)))
        out = np.zeros(max(n.value, 1), dtype=NODE_DTYPE)
        self._ck(self.L.sdtgpu_export_nodes(self.h, thrd_num, int(sort_by_ordinal), out.ctypes.data, len(out), C.byref(n)))
        return out[: n.value]

    def export_kmersets(self, thrd_num: int = 8):
        """Returns (records in (set, slot) order, set_info) decoded from reference-layout KmerSets."""
        sets = (C.POINTER(KmerSet) * thrd_num)()
        self._ck(self.L.sdtgpu_export_kmersets(self.h, thrd_num, sets))
        try:
            return read_kmersets(sets, thrd_num, self.key_words)
        finally:
            self.L.sdtgpu_free_kmersets(sets, thrd_num)

    # ---- lookups in the finalized table (include/sdtgpu.h sdtgpu_lookup_*)
    def _torch_device(self):
        import torch
        return torch.device("cuda", self.device)

    def lookup_kmers(self, keys):
        """keys: uint64 [n, 4] in the sdtgpu_node layout, a numpy array or a CUDA tensor (int64 or uint64).
        numpy in -> HIT_DTYPE numpy array [n] out; CUDA tensor in -> CUDA int32 tensor [n, 4] (count, l_links, rword,
        status; hits_numpy() decodes it).  Synchronises the handle's stream."""
        import torch
        dev = self._torch_device()
        host = isinstance(keys, np.ndarray)
        if host:
            keys = torch.from_numpy(np.ascontiguousarray(keys, dtype=np.uint64).view(np.int64)).to(dev)
        keys = keys.contiguous()
        assert keys.ndim == 2 and keys.shape[1] == 4 and keys.element_size() == 8, "keys must be [n, 4] 64-bit words"
        n = keys.shape[0]
        out = torch.empty((n, 4), dtype=torch.int32, device=dev)
        torch.cuda.current_stream(dev).synchronize()          # the keys are written on torch's stream, read on the handle's
        self._ck(self.L.sdtgpu_lookup_kmers_device(self.h, _ptr(keys), n, _ptr(out)))
        self.sync()
        return hits_numpy(out) if host else out

    def lookup_reads(self, packed, lens=None, nmask=None, n_reads=None, uniform_len=0, stride_bytes=None):
        """Every window of a batch of reads in CUDA tensors (the conventions of push_reads(..., device=True)) ->
        CUDA int32 tensor [n_reads, max_read_len - K + 1, 4] of hits: window j of read r at [r, j]; windows a read
        does not have are all zero.  Synchronises the handle's stream."""
        import torch
        if n_reads is None:
            n_reads = packed.shape[0]
        if stride_bytes is None:
            stride_bytes = packed.shape[1]
        out = torch.empty((n_reads, self.max_read_len - self.K + 1, 4), dtype=torch.int32, device=self._torch_device())
        torch.cuda.current_stream(self._torch_device()).synchronize()
        self._ck(self.L.sdtgpu_lookup_reads_device(self.h, _ptr(packed), _ptr(lens), _ptr(nmask), n_reads, uniform_len,
                                                   stride_bytes, _ptr(out)))
        self.sync()
        return out

    # ---- edges between junction k-mers (include/sdtgpu.h sdtgpu_edges_*)
    def edges_build(self) -> dict:
        """Compacts the finalized table into edges and cycles on the device -> the eight counts of sdtgpu_edges_build
        (EDGE_COUNTS) and ms, the device time of the build."""
        out, ms = (C.c_uint64 * 8)(), C.c_double()
        self._ck(self.L.sdtgpu_edges_build(self.h, out, C.byref(ms)))
        self._n_edges = int(out[0])
        res = {k: int(v) for k, v in zip(EDGE_COUNTS, out)}
        res["ms"] = float(ms.value)
        return res

    def edges(self):
        """The last edges_build's records and sequences, copied to the host -> (EDGE_DTYPE array, uint8 sequence
        buffer in the tight-string convention; edge_codes() decodes one edge)."""
        import torch
        e, q = C.c_void_p(), C.c_void_p()
        self._ck(self.L.sdtgpu_edges_buffers(self.h, C.byref(e), C.byref(q)))
        n = self._n_edges
        if n == 0:
            return np.zeros(0, dtype=EDGE_DTYPE), np.zeros(0, dtype=np.uint8)
        dev = self._torch_device()
        edges = _device_bytes(int(e.value), n * EDGE_DTYPE.itemsize, dev).cpu().numpy().view(EDGE_DTYPE)
        last = edges[-1]      # the records are in sequence order
        bases = int(last["length"]) + self.K - (1 if int(last["flags"]) & EDGE_CYCLE else 0)
        words = (int(last["seq"]) + bases + 31) // 32
        return edges, _device_bytes(int(q.value), words * 8, dev).cpu().numpy()

    # ---- reads mapped onto the edges (include/sdtgpu.h sdtgpu_edges_map_reads, sdtgpu_arcs_*)
    def map_reads(self, packed, lens=None, nmask=None, n_reads=None, uniform_len=0, stride_bytes=None, count_arcs=True,
                  out=None):
        """Every read (K+1)-mer of a batch in CUDA tensors (the conventions of lookup_reads) onto the last edges_build ->
        CUDA int32 tensor [n_reads, max_read_len - K + 1, 2] of sdtgpu_step (record, index << 1 | strand; all ones =
        none; steps_numpy() decodes it), window j of read r at [r, j].  count_arcs adds the batch's vertex crossings
        to the handle's arc counters.  out: a tensor of that shape to write into.  Synchronises the handle's stream."""
        import torch
        if n_reads is None:
            n_reads = packed.shape[0]
        if stride_bytes is None:
            stride_bytes = packed.shape[1]
        if out is None:
            out = torch.empty((n_reads, self.max_read_len - self.K + 1, 2), dtype=torch.int32, device=self._torch_device())
        assert out.is_contiguous() and out.numel() >= n_reads * (self.max_read_len - self.K + 1) * 2
        torch.cuda.current_stream(self._torch_device()).synchronize()
        self._ck(self.L.sdtgpu_edges_map_reads(self.h, _ptr(packed), _ptr(lens), _ptr(nmask), n_reads, uniform_len,
                                               stride_bytes, _ptr(out), int(bool(count_arcs))))
        self.sync()
        return out

    def arcs_build(self) -> dict:
        """The non-zero arc counters as records on the device -> arcs, crossings (the sum of their counts) and ms, the
        device time of the build."""
        out, ms = (C.c_uint64 * 2)(), C.c_double()
        self._ck(self.L.sdtgpu_arcs_build(self.h, out, C.byref(ms)))
        self._n_arcs = int(out[0])
        return dict(arcs=int(out[0]), crossings=int(out[1]), ms=float(ms.value))

    def arcs(self) -> np.ndarray:
        """The last arcs_build's records, copied to the host -> ARC_DTYPE array in (vertex position, left base, right
        base) order."""
        a = C.c_void_p()
        self._ck(self.L.sdtgpu_arcs_buffers(self.h, C.byref(a)))
        if self._n_arcs == 0:
            return np.zeros(0, dtype=ARC_DTYPE)
        return _device_bytes(int(a.value), self._n_arcs * ARC_DTYPE.itemsize, self._torch_device()).cpu().numpy().view(ARC_DTYPE)

    def arcs_clear(self):
        self._ck(self.L.sdtgpu_arcs_clear(self.h))

    # ---- the table pruned of minor branches and tips (include/sdtgpu.h sdtgpu_prune)
    def prune(self, minor_pct: int = 5, single_tips=None, minor_tips: bool = True) -> dict:
        """Prunes the finalized table once, with the reference's defaults -> the eight counts of sdtgpu_prune
        (PRUNE_COUNTS) and ms, its device time.  single_tips=None: on when finalize had -d 0, as call_pregraph does."""
        if single_tips is None:
            single_tips = self.lookup_route()["deLowKmer"] == 0
        flags = (PRUNE_SINGLE_TIPS if single_tips else 0) | (PRUNE_MINOR_TIPS if minor_tips else 0)
        out, ms = (C.c_uint64 * 8)(), C.c_double()
        self._ck(self.L.sdtgpu_prune(self.h, minor_pct, flags, out, C.byref(ms)))
        res = {k: int(v) for k, v in zip(PRUNE_COUNTS, out)}
        res["ms"] = float(ms.value)
        return res

    # ---- lookups routed to the rank that owns each k-mer (include/sdtgpu.h sdtgpu_lookup_stage_* ... _exchange)
    def lookup_route(self) -> dict:
        """How this handle's keys are sharded (sdtgpu_lookup_route)."""
        out = (C.c_uint64 * 12)()
        self._ck(self.L.sdtgpu_lookup_route(self.h, out))
        names = ("kind", "rank", "world", "K", "key_words", "n_slices", "n_local", "m", "lo", "w", "deLowKmer", "finalized")
        return {k: int(v) for k, v in zip(names, out)}

    def _stage(self, fn, *args):
        world = self.lookup_route()["world"]
        ptr, starts, counts = C.c_void_p(), (C.c_uint64 * world)(), (C.c_uint64 * world)()
        self._ck(fn(self.h, *args, C.byref(ptr), starts, counts))
        self.sync()
        return int(ptr.value or 0), [int(x) for x in starts], [int(x) for x in counts]

    def lookup_stage_kmers(self, keys):
        """keys: CUDA tensor [n, 4] of 64-bit words (the layout of lookup_kmers) -> (device address of the staged
        queries, starts[world], counts[world] in queries of key_words u64 each).  Synchronises the handle's stream."""
        import torch
        torch.cuda.current_stream(self._torch_device()).synchronize()
        return self._stage(self.L.sdtgpu_lookup_stage_kmers, _ptr(keys), keys.shape[0])

    def lookup_stage_reads(self, packed, lens=None, nmask=None, n_reads=None, uniform_len=0, stride_bytes=None):
        """Every window of a batch of reads (the conventions of lookup_reads) staged by owner; as lookup_stage_kmers."""
        import torch
        n_reads = packed.shape[0] if n_reads is None else n_reads
        stride_bytes = packed.shape[1] if stride_bytes is None else stride_bytes
        torch.cuda.current_stream(self._torch_device()).synchronize()
        return self._stage(self.L.sdtgpu_lookup_stage_reads, _ptr(packed), _ptr(lens), _ptr(nmask), n_reads, uniform_len, stride_bytes)

    def lookup_answer_buffer(self, n: int):
        """-> (device address for n received queries, device address of their n hits)."""
        q, r = C.c_void_p(), C.c_void_p()
        self._ck(self.L.sdtgpu_lookup_answer_buffer(self.h, n, C.byref(q), C.byref(r)))
        return int(q.value or 0), int(r.value or 0)

    def lookup_answer(self, n: int):
        """Answers the n queries in the answer buffer.  Synchronises the handle's stream."""
        self._ck(self.L.sdtgpu_lookup_answer(self.h, n))
        self.sync()

    def lookup_unstage_buffer(self) -> int:
        """-> device address for the hits of this rank's staged queries, in staged order."""
        p = C.c_void_p()
        self._ck(self.L.sdtgpu_lookup_unstage_buffer(self.h, C.byref(p)))
        return int(p.value or 0)

    def lookup_unstage(self, out):
        """Writes the hits to out (a CUDA int32 tensor shaped as lookup_kmers' or lookup_reads' output).  Synchronises
        the handle's stream."""
        import torch
        torch.cuda.current_stream(self._torch_device()).synchronize()
        self._ck(self.L.sdtgpu_lookup_unstage(self.h, _ptr(out)))
        self.sync()
        return out

    def _exchange(self, fn, comm: "SkmComm", *args):
        ms = C.c_double()
        rc = fn(self.h, comm.c, *args, C.byref(ms))
        if rc:     # (argument errors are reported without the communicator)
            raise SdtGpuError(rc, (self.L.sdtgpu_comm_last_error(comm.c) or self.L.sdtgpu_comm_last_error(None) or b"").decode())
        self.last_collective_ms = float(ms.value)

    def lookup_kmers_exchange(self, comm: "SkmComm", keys):
        """lookup_kmers over all ranks of comm (every rank calls it with its own keys, possibly none): each key is
        answered by the rank that owns it.  Same inputs and outputs as lookup_kmers; the device time of the collectives
        is left in self.last_collective_ms."""
        import torch
        dev = self._torch_device()
        host = isinstance(keys, np.ndarray)
        if host:
            keys = torch.from_numpy(np.ascontiguousarray(keys, dtype=np.uint64).view(np.int64)).to(dev)
        keys = keys.contiguous()
        assert keys.ndim == 2 and keys.shape[1] == 4 and keys.element_size() == 8, "keys must be [n, 4] 64-bit words"
        out = torch.empty((keys.shape[0], 4), dtype=torch.int32, device=dev)
        torch.cuda.current_stream(dev).synchronize()
        self._exchange(self.L.sdtgpu_lookup_kmers_exchange, comm, _ptr(keys), keys.shape[0], _ptr(out))
        return hits_numpy(out) if host else out

    def lookup_reads_exchange(self, comm: "SkmComm", packed, lens=None, nmask=None, n_reads=None, uniform_len=0,
                              stride_bytes=None, out=None):
        """lookup_reads over all ranks of comm, every window answered by the rank that owns it.  Same inputs and outputs
        as lookup_reads; out (optional): a CUDA int32 tensor [>= n_reads, max_read_len - K + 1, 4] to reuse."""
        import torch
        dev = self._torch_device()
        n_reads = packed.shape[0] if n_reads is None else n_reads
        stride_bytes = packed.shape[1] if stride_bytes is None else stride_bytes
        if out is None:
            out = torch.empty((n_reads, self.max_read_len - self.K + 1, 4), dtype=torch.int32, device=dev)
        else:
            out = out[:n_reads]
        torch.cuda.current_stream(dev).synchronize()
        self._exchange(self.L.sdtgpu_lookup_reads_exchange, comm, _ptr(packed), _ptr(lens), _ptr(nmask), n_reads,
                       uniform_len, stride_bytes, _ptr(out))
        return out

    def kernel_time(self, reset: bool = True):
        ms, nl, al = C.c_double(), C.c_uint64(), C.c_uint64()
        self._ck(self.L.sdtgpu_kernel_time(self.h, int(reset), C.byref(ms), C.byref(nl), C.byref(al)))
        return ms.value, nl.value, al.value

    def phase_times(self, reset: bool = True):
        """{phase: (ms, launches)} per kernel class (PHASES) since the last reset."""
        ms, nl = (C.c_double * 8)(), (C.c_uint64 * 8)()
        self._ck(self.L.sdtgpu_phase_times(self.h, int(reset), ms, nl))
        return {PHASES[i]: (ms[i], nl[i]) for i in range(7)}

    def slice_geometry(self):
        out = (C.c_uint64 * 12)()
        self._ck(self.L.sdtgpu_slice_geometry(self.h, out))
        return dict(n_slices=out[0], slice_slots=out[1], m=out[2], mmers_per_window=out[3], record_bytes=out[4],
                    n_records=out[5], n_nodes=out[6], retried_items=out[7], n_records_merged=out[8], work_items=out[9],
                    epochs_emitted_again=out[10], device_allocations=out[11])

    def kernel_times(self, reset: bool = True):
        """(ms[3], launches[3]) for insert / partition-count / partition-scatter kernels."""
        ms, nl = (C.c_double * 3)(), (C.c_uint64 * 3)()
        self._ck(self.L.sdtgpu_kernel_times(self.h, int(reset), ms, nl))
        return list(ms), list(nl)


class SkmComm:
    """include/sdtgpu.h sdtgpu_comm_*: the NCCL communicator of the super-k-mer exchange, owned by the library.
    `unique_id()` on rank 0, the 128 bytes to every rank by whatever means the host has, then SkmComm(...)."""

    @staticmethod
    def unique_id() -> bytes:
        import torch      # noqa: F401  (its NCCL must be in the process FIRST: the library binds whatever libnccl.so.2 is loaded, else the system's — and torch cannot live with an older one)
        L = library()
        buf = (C.c_uint8 * 128)()
        rc = L.sdtgpu_comm_unique_id(buf)
        if rc:
            raise SdtGpuError(rc, (L.sdtgpu_comm_last_error(None) or b"").decode())
        return bytes(buf)

    def __init__(self, device: int, unique_id: bytes, rank: int, world: int):
        import torch      # noqa: F401  (see unique_id)
        self.L = library()
        self.c = C.c_void_p()
        buf = (C.c_uint8 * 128).from_buffer_copy(unique_id)
        rc = self.L.sdtgpu_comm_create(C.byref(self.c), device, buf, rank, world)
        if rc:
            raise SdtGpuError(rc, (self.L.sdtgpu_comm_last_error(None) or b"").decode())

    def close(self):
        if self.c:
            self.L.sdtgpu_comm_destroy(self.c)
            self.c = C.c_void_p()


def synth_reads_device(tr_dev: dict, seed: int, first_pair: int, n_pairs: int, read_len: int, stride_bytes: int,
                       out, device: int = 0, stream: int = 0):
    """tr_dev: dict of CUDA tensors bases(u8) starts(i64 viewed as u64) lengths(i32 as u32) cum(i64 as u64)."""
    rc = library().sdtgpu_synth_reads_device(device, stream, _ptr(tr_dev["bases"]), _ptr(tr_dev["starts"]),
                                             _ptr(tr_dev["lengths"]), _ptr(tr_dev["cum"]), tr_dev["n"], seed,
                                             first_pair, n_pairs, read_len, stride_bytes, _ptr(out))
    if rc:
        raise SdtGpuError(rc, "sdtgpu_synth_reads_device")


class ReadPacker:
    """include/sdtpack.h: multi-threaded FASTA/FASTQ parser + 2-bit packer (host only)."""

    def __init__(self, path1: str, path2: str | None = None, fastq: bool = False, n_threads: int = 0):
        self.L = library()
        self.h = C.c_void_p()
        if self.L.sdtpack_open(C.byref(self.h), path1.encode(), path2.encode() if path2 else None, int(fastq), n_threads):
            raise OSError(C.get_errno(), f"sdtpack_open({path1}, {path2})")

    def next(self, max_read_len: int, max_reads: int, n_kmer: bool = False, reverse: bool = False, stride_bytes: int | None = None):
        """Returns (packed[n, stride], lens[n], nmask[n, stride/2] or None); n == 0 at end of input."""
        from .synth import stride_bytes as _sb
        stride = stride_bytes or _sb(max_read_len)
        packed = np.empty((max_reads, stride), dtype=np.uint8)
        lens = np.empty(max_reads, dtype=np.uint32)
        nmask = np.empty((max_reads, stride // 2), dtype=np.uint8) if n_kmer else None
        n = self.L.sdtpack_next(self.h, max_read_len, int(n_kmer), int(reverse), packed.ctypes.data, lens.ctypes.data,
                                nmask.ctypes.data if n_kmer else None, max_reads, stride)
        if n < 0:
            raise OSError("sdtpack_next failed")
        return packed[:n], lens[:n], (nmask[:n] if n_kmer else None)

    def close(self):
        if getattr(self, "h", None):
            self.L.sdtpack_close(self.h)
            self.h = None

    __del__ = close


class DeviceReadPacker:
    """include/sdtgpu.h sdtgpu_reader_*: FASTA/FASTQ parsed and packed on the GPU.  Same records, order and bytes as
    ReadPacker, delivered as CUDA tensors in the layout of PregraphGPU.push_reads(..., device=True).

    world > 0 makes a shard reader (sdtgpu_reader_open_shard): rank `rank` of `world` readers of the same library, each
    parsing only its own byte range.  Every rank calls summary(), the ranks share the bytes, every rank calls
    plan(all summaries in rank order) (or plan_exchange(comm) / exchange.plan_reader for both steps), then next();
    tell() gives the global ordinal of the next record."""

    SUMMARY_BYTES = 256

    def __init__(self, path1: str, path2: str | None = None, fastq: bool = False, device: int = 0, chunk_bytes: int = 0,
                 rank: int = 0, world: int = 0):
        self.L = library()
        self.h = C.c_void_p()
        self.device = device
        self.world = world
        p1, p2 = path1.encode(), path2.encode() if path2 else None
        if world:
            rc = self.L.sdtgpu_reader_open_shard(C.byref(self.h), device, p1, p2, int(fastq), chunk_bytes, rank, world)
        else:
            rc = self.L.sdtgpu_reader_open(C.byref(self.h), device, p1, p2, int(fastq), chunk_bytes)
        if rc:
            raise SdtGpuError(rc, self.L.sdtgpu_reader_last_error(None).decode())

    def _rck(self, rc: int, what: str):
        if rc:
            raise SdtGpuError(rc, f"{what}: " + self.L.sdtgpu_reader_last_error(self.h).decode())

    def summary(self) -> bytes:
        """This rank's 256-byte summary (a device pass over its byte range the first time)."""
        buf = (C.c_uint8 * self.SUMMARY_BYTES)()
        self._rck(self.L.sdtgpu_reader_summary(self.h, buf), "sdtgpu_reader_summary")
        return bytes(buf)

    @staticmethod
    def _plan_dict(out) -> dict:
        return dict(records=int(out[0]), library_records=int(out[1]), n1=int(out[2]), n2=int(out[3]))

    def plan(self, summaries) -> dict:
        """Plans from every rank's summary, in rank order: {records (this rank returns), library_records, n1, n2}."""
        summaries = list(summaries)
        if len(summaries) != self.world or any(len(s) != self.SUMMARY_BYTES for s in summaries):
            raise SdtGpuError(1, f"plan: need {self.world} summaries of {self.SUMMARY_BYTES} bytes, got {len(summaries)}")
        blob = b"".join(bytes(s) for s in summaries)
        buf = (C.c_uint8 * len(blob)).from_buffer_copy(blob)
        out = (C.c_uint64 * 4)()
        self._rck(self.L.sdtgpu_reader_plan(self.h, buf, out), "sdtgpu_reader_plan")
        return self._plan_dict(out)

    def plan_exchange(self, comm: "SkmComm") -> dict:
        """summary + all-gather over the library's communicator + plan, in one collective call."""
        out = (C.c_uint64 * 4)()
        rc = self.L.sdtgpu_reader_plan_exchange(self.h, comm.c, out)
        if rc:
            raise SdtGpuError(rc, (self.L.sdtgpu_comm_last_error(comm.c) or self.L.sdtgpu_comm_last_error(None) or b"").decode())
        return self._plan_dict(out)

    def tell(self) -> int:
        """The global ordinal of the next record (a plain reader: records returned so far)."""
        o = C.c_uint64()
        self._rck(self.L.sdtgpu_reader_tell(self.h, C.byref(o)), "sdtgpu_reader_tell")
        return int(o.value)

    def next(self, max_read_len: int, max_reads: int, n_kmer: bool = False, reverse: bool = False,
             stride_bytes: int | None = None):
        """Returns (packed[n, stride], lens[n], nmask[n, stride/2] or None) as CUDA uint8 / int32 (lens: uint32 bits)
        tensors; n == 0 at end of input.  Written on torch's current stream of the device."""
        import torch
        from .synth import stride_bytes as _sb
        stride = stride_bytes or _sb(max_read_len)
        dev = torch.device("cuda", self.device)
        packed = torch.empty((max_reads, stride), dtype=torch.uint8, device=dev)
        lens = torch.empty(max_reads, dtype=torch.int32, device=dev)
        nmask = torch.empty((max_reads, stride // 2), dtype=torch.uint8, device=dev) if n_kmer else None
        n = C.c_uint64()
        rc = self.L.sdtgpu_reader_next(self.h, torch.cuda.current_stream(dev).cuda_stream, max_read_len, int(n_kmer),
                                       int(reverse), _ptr(packed), _ptr(lens), _ptr(nmask), max_reads, stride, C.byref(n))
        if rc:
            raise SdtGpuError(rc, self.L.sdtgpu_reader_last_error(self.h).decode())
        n = int(n.value)
        return packed[:n], lens[:n], (nmask[:n] if n_kmer else None)

    def stats(self) -> dict:
        out = (C.c_uint64 * 4)()
        rc = self.L.sdtgpu_reader_stats(self.h, out)
        if rc:
            raise SdtGpuError(rc, "sdtgpu_reader_stats")
        return dict(text_bytes=int(out[0]), records=int(out[1]), chunks=int(out[2]), allocations=int(out[3]))

    def close(self):
        if getattr(self, "h", None):
            self.L.sdtgpu_reader_close(self.h)
            self.h = None

    __del__ = close

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()
