"""Shard readers' C ABI (include/sdtgpu.h sdtgpu_reader_open_shard / _summary / _plan / _tell / _plan_exchange)
without a GPU: the symbols exist, open_shard touches no CUDA state and rejects bad ranks, worlds and paths, and every
NULL argument is SDTGPU_EINVAL before any CUDA call."""
import ctypes as C

import pytest

EINVAL = 1


@pytest.fixture()
def files(tmp_path):
    a, b = tmp_path / "1.fa", tmp_path / "2.fa"
    a.write_bytes(b">a\nACGT\n>b\nGG\n")
    b.write_bytes(b">a\nTTTT\n>b\nCC\n")
    return str(a).encode(), str(b).encode()


def test_symbols_exported(pkg):
    L = pkg.library()
    for name in ("sdtgpu_reader_open_shard", "sdtgpu_reader_summary", "sdtgpu_reader_plan", "sdtgpu_reader_tell",
                 "sdtgpu_reader_plan_exchange"):
        assert hasattr(L, name), name


@pytest.mark.parametrize("rank,world", [(-1, 2), (2, 2), (5, 2), (0, 0), (0, -1), (0, 1025), (1024, 1024)])
def test_open_shard_rejects_rank_and_world(pkg, files, rank, world):
    L = pkg.library()
    h = C.c_void_p()
    assert L.sdtgpu_reader_open_shard(C.byref(h), 0, files[0], files[1], 0, 0, rank, world) == EINVAL
    assert not h.value
    assert L.sdtgpu_reader_last_error(None)


def test_open_shard_accepts_every_rank(pkg, files):
    L = pkg.library()
    for rank, world in ((0, 1), (1023, 1024), (3, 7)):
        h = C.c_void_p()
        assert L.sdtgpu_reader_open_shard(C.byref(h), 0, files[0], None, 1, 64, rank, world) == 0
        assert h.value
        L.sdtgpu_reader_close(h)


def test_open_shard_null_and_missing_paths(pkg, files, tmp_path):
    L = pkg.library()
    h = C.c_void_p()
    assert L.sdtgpu_reader_open_shard(None, 0, files[0], None, 0, 0, 0, 1) == EINVAL
    assert L.sdtgpu_reader_open_shard(C.byref(h), 0, None, None, 0, 0, 0, 1) == EINVAL
    assert L.sdtgpu_reader_open_shard(C.byref(h), 0, None, files[1], 0, 0, 0, 1) == EINVAL
    missing = str(tmp_path / "no_such.fa")
    assert L.sdtgpu_reader_open_shard(C.byref(h), 0, files[0], missing.encode(), 0, 0, 0, 2) == EINVAL
    assert not h.value
    assert missing in L.sdtgpu_reader_last_error(None).decode()


def test_null_arguments(pkg, files):
    L = pkg.library()
    h = C.c_void_p()
    assert L.sdtgpu_reader_open_shard(C.byref(h), 0, files[0], files[1], 0, 0, 0, 2) == 0
    buf = (C.c_uint8 * 512)()
    out = (C.c_uint64 * 4)()
    o = C.c_uint64()
    assert L.sdtgpu_reader_summary(None, buf) == EINVAL
    assert L.sdtgpu_reader_summary(h, None) == EINVAL
    assert L.sdtgpu_reader_plan(None, buf, out) == EINVAL
    assert L.sdtgpu_reader_plan(h, None, out) == EINVAL
    assert L.sdtgpu_reader_plan(h, buf, None) == EINVAL
    assert L.sdtgpu_reader_tell(None, C.byref(o)) == EINVAL
    assert L.sdtgpu_reader_tell(h, None) == EINVAL
    comm = 1 << 20      # never dereferenced: the checks come first
    assert L.sdtgpu_reader_plan_exchange(None, comm, out) == EINVAL
    assert L.sdtgpu_reader_plan_exchange(h, None, out) == EINVAL
    assert L.sdtgpu_reader_plan_exchange(h, comm, None) == EINVAL
    st = (C.c_uint64 * 4)()
    assert L.sdtgpu_reader_stats(h, st) == 0 and list(st) == [0, 0, 0, 0]
    L.sdtgpu_reader_close(h)


def test_plan_refuses_bad_summaries_without_cuda(pkg, files):
    """plan is host arithmetic: summaries that are not this library's are refused with no device present."""
    L = pkg.library()
    h = C.c_void_p()
    assert L.sdtgpu_reader_open_shard(C.byref(h), 0, files[0], files[1], 0, 0, 1, 2) == 0
    out = (C.c_uint64 * 4)()
    assert L.sdtgpu_reader_plan(h, (C.c_uint8 * 512)(), out) == EINVAL
    assert L.sdtgpu_reader_last_error(h)
    L.sdtgpu_reader_close(h)


def test_python_wrapper_checks_the_count(pkg, files):
    rd = pkg.DeviceReadPacker(files[0].decode(), files[1].decode(), rank=0, world=2)
    with pytest.raises(pkg.pregraph.SdtGpuError) as e:
        rd.plan([bytes(256)])
    assert e.value.code == EINVAL
    with pytest.raises(pkg.pregraph.SdtGpuError) as e:
        rd.plan([bytes(256), bytes(256)])
    assert e.value.code == EINVAL
    rd.close()
