"""The device FASTA/FASTQ reader's C ABI (include/sdtgpu.h sdtgpu_reader_*) without a GPU: the symbols exist, open
touches no CUDA state, and every argument error is SDTGPU_EINVAL before any CUDA call."""
import ctypes as C

import pytest

EINVAL = 1


@pytest.fixture()
def reader(pkg, tmp_path):
    p = tmp_path / "r.fa"
    p.write_bytes(b">a\nACGT\n")
    L = pkg.library()
    h = C.c_void_p()
    assert L.sdtgpu_reader_open(C.byref(h), 0, str(p).encode(), None, 0, 0) == 0
    yield L, h
    L.sdtgpu_reader_close(h)


def test_symbols_exported(pkg):
    L = pkg.library()
    for name in ("sdtgpu_reader_open", "sdtgpu_reader_next", "sdtgpu_reader_stats", "sdtgpu_reader_last_error",
                 "sdtgpu_reader_close"):
        assert hasattr(L, name), name


def test_missing_file_names_the_path(pkg, tmp_path):
    L = pkg.library()
    h = C.c_void_p()
    missing = str(tmp_path / "no_such_file.fq")
    assert L.sdtgpu_reader_open(C.byref(h), 0, missing.encode(), None, 1, 0) == EINVAL
    assert not h.value
    assert missing in L.sdtgpu_reader_last_error(None).decode()
    good = tmp_path / "r1.fa"
    good.write_bytes(b">a\nACGT\n")
    assert L.sdtgpu_reader_open(C.byref(h), 0, str(good).encode(), missing.encode(), 0, 0) == EINVAL
    assert missing in L.sdtgpu_reader_last_error(None).decode()


def test_null_arguments(pkg, reader):
    L, h = reader
    n = C.c_uint64()
    assert L.sdtgpu_reader_open(None, 0, b"x", None, 0, 0) == EINVAL
    hh = C.c_void_p()
    assert L.sdtgpu_reader_open(C.byref(hh), 0, None, None, 0, 0) == EINVAL
    buf = 1 << 20      # never dereferenced: the checks come first
    assert L.sdtgpu_reader_next(None, None, 100, 0, 0, buf, buf, None, 10, 28, C.byref(n)) == EINVAL
    assert L.sdtgpu_reader_next(h, None, 100, 0, 0, None, buf, None, 10, 28, C.byref(n)) == EINVAL
    assert L.sdtgpu_reader_next(h, None, 100, 0, 0, buf, None, None, 10, 28, C.byref(n)) == EINVAL
    assert L.sdtgpu_reader_next(h, None, 100, 0, 0, buf, buf, None, 10, 28, None) == EINVAL
    out = (C.c_uint64 * 4)()
    assert L.sdtgpu_reader_stats(None, out) == EINVAL
    assert L.sdtgpu_reader_stats(h, out) == 0 and list(out) == [0, 0, 0, 0]
    L.sdtgpu_reader_close(None)


@pytest.mark.parametrize("max_read_len,n_kmer,nmask,max_reads,stride", [
    (100, 0, False, 10, 30),      # stride not a multiple of 4
    (100, 0, False, 10, 24),      # stride * 4 < max_read_len
    (100, 1, False, 10, 28),      # n_kmer without an nmask
    (100, 0, False, 0, 28),       # max_reads < number of files
    (0, 0, False, 10, 28),        # max_read_len < 1
])
def test_inconsistent_arguments(pkg, reader, max_read_len, n_kmer, nmask, max_reads, stride):
    L, h = reader
    n = C.c_uint64()
    buf = 1 << 20
    assert L.sdtgpu_reader_next(h, None, max_read_len, n_kmer, 0, buf, buf, buf if nmask else None, max_reads, stride,
                                C.byref(n)) == EINVAL
    assert L.sdtgpu_reader_last_error(h)


def test_pairs_need_two_reads(pkg, tmp_path):
    a, b = tmp_path / "1.fa", tmp_path / "2.fa"
    a.write_bytes(b">a\nACGT\n")
    b.write_bytes(b">b\nACGT\n")
    L = pkg.library()
    h = C.c_void_p()
    assert L.sdtgpu_reader_open(C.byref(h), 0, str(a).encode(), str(b).encode(), 0, 0) == 0
    n = C.c_uint64()
    buf = 1 << 20
    assert L.sdtgpu_reader_next(h, None, 100, 0, 0, buf, buf, None, 1, 28, C.byref(n)) == EINVAL
    L.sdtgpu_reader_close(h)
