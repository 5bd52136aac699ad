"""CPU-side checks of the routed lookups (sdtgpu_lookup_stage_* / _answer / _unstage / _route and the NCCL-driven
sdtgpu_lookup_*_exchange): every entry point is exported and rejects a NULL handle, buffer or communicator with
SDTGPU_EINVAL before any CUDA call."""
import ctypes as C

EINVAL = 1
ENTRY_POINTS = ("sdtgpu_lookup_route", "sdtgpu_lookup_stage_kmers", "sdtgpu_lookup_stage_reads", "sdtgpu_lookup_answer_buffer",
                "sdtgpu_lookup_answer", "sdtgpu_lookup_unstage_buffer", "sdtgpu_lookup_unstage",
                "sdtgpu_lookup_kmers_exchange", "sdtgpu_lookup_reads_exchange")


def test_routed_lookup_symbols_are_exported(pkg):
    L = pkg.library()
    for name in ENTRY_POINTS:
        assert hasattr(L, name), name


def test_routed_lookups_reject_null_arguments_without_a_gpu(pkg):
    L = pkg.library()
    buf = (C.c_uint64 * 64)()
    p = C.c_void_p()
    fake = C.cast(buf, C.c_void_p)       # never dereferenced: the NULL argument beside it is rejected first
    assert L.sdtgpu_lookup_route(None, buf) == EINVAL
    assert L.sdtgpu_lookup_stage_kmers(None, buf, 1, C.byref(p), buf, buf) == EINVAL
    assert L.sdtgpu_lookup_stage_kmers(None, None, 0, None, None, None) == EINVAL
    assert L.sdtgpu_lookup_stage_reads(None, buf, None, None, 1, 100, 28, C.byref(p), buf, buf) == EINVAL
    assert L.sdtgpu_lookup_answer_buffer(None, 1, C.byref(p), C.byref(p)) == EINVAL
    assert L.sdtgpu_lookup_answer(None, 0) == EINVAL
    assert L.sdtgpu_lookup_unstage_buffer(None, C.byref(p)) == EINVAL
    assert L.sdtgpu_lookup_unstage(None, buf) == EINVAL
    # a NULL communicator, and a NULL buffer with queries to route
    assert L.sdtgpu_lookup_kmers_exchange(None, None, buf, 1, buf, None) == EINVAL
    assert L.sdtgpu_lookup_kmers_exchange(fake, None, buf, 1, buf, None) == EINVAL
    assert L.sdtgpu_lookup_kmers_exchange(fake, fake, None, 1, buf, None) == EINVAL
    assert L.sdtgpu_lookup_kmers_exchange(fake, fake, buf, 1, None, None) == EINVAL
    assert L.sdtgpu_lookup_reads_exchange(None, None, buf, None, None, 1, 100, 28, buf, None) == EINVAL
    assert L.sdtgpu_lookup_reads_exchange(fake, None, buf, None, None, 1, 100, 28, buf, None) == EINVAL
    assert L.sdtgpu_lookup_reads_exchange(fake, fake, None, None, None, 1, 100, 28, buf, None) == EINVAL
    assert L.sdtgpu_lookup_reads_exchange(fake, fake, buf, None, None, 1, 100, 28, None, None) == EINVAL
