"""CPU-side checks of the read paths (sdtgpu_edges_map_reads, sdtgpu_arcs_*): the symbols are exported, argument errors
are reported before any CUDA call, and the Python layouts and decoding match the C structs."""
import ctypes as C

import numpy as np

EINVAL = 1


def test_path_symbols_exported(pkg):
    L = pkg.library()
    for name in ("sdtgpu_edges_map_reads", "sdtgpu_arcs_build", "sdtgpu_arcs_buffers", "sdtgpu_arcs_clear"):
        assert hasattr(L, name), name


def test_path_calls_reject_null_arguments_without_a_gpu(pkg):
    L = pkg.library()
    out, ms, a = (C.c_uint64 * 2)(), C.c_double(), C.c_void_p()
    assert L.sdtgpu_edges_map_reads(None, None, None, None, 0, 100, 28, None, 1) == EINVAL
    assert L.sdtgpu_edges_map_reads(None, None, None, None, 0, 100, 28, None, 0) == EINVAL
    assert L.sdtgpu_arcs_build(None, out, C.byref(ms)) == EINVAL
    assert L.sdtgpu_arcs_build(None, None, None) == EINVAL
    assert L.sdtgpu_arcs_buffers(None, C.byref(a)) == EINVAL
    assert L.sdtgpu_arcs_buffers(None, None) == EINVAL
    assert L.sdtgpu_arcs_clear(None) == EINVAL


def test_path_layouts_and_decoding(pkg):
    assert pkg.STEP_DTYPE.itemsize == 8 and pkg.STEP_DTYPE.names == ("record", "pos")
    assert pkg.ARC_DTYPE.itemsize == 16 and pkg.ARC_DTYPE.names == ("from", "to", "count", "unused")
    assert pkg.STEP_NONE == 0xFFFFFFFF
    raw = np.zeros((2, 3), dtype=pkg.STEP_DTYPE)
    raw[0, 0] = (7, 5 << 1)                      # record 7, step 5, strand 0
    raw[0, 1] = (3, 2 << 1 | 1)                  # record 3, step 2, strand 1
    raw[0, 2] = (pkg.STEP_NONE, pkg.STEP_NONE)
    raw[1, :] = (pkg.STEP_NONE, pkg.STEP_NONE)
    raw[1, 1] = (0, 1)                           # record 0, step 0, strand 1
    as_tensor = raw.view(np.int32).reshape(2, 3, 2)   # what map_reads returns, as int32 pairs
    got = pkg.steps_numpy(as_tensor)
    assert got.shape == (2, 3, 3) and got.dtype == np.int64
    assert got[0].tolist() == [[7, 5, 0], [3, 2, 1], [-1, -1, -1]]
    assert got[1].tolist() == [[-1, -1, -1], [0, 0, 1], [-1, -1, -1]]
