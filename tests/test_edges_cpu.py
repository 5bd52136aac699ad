"""CPU-side checks of the edge build (sdtgpu_edges_build, sdtgpu_edges_buffers): the symbols are exported, argument
errors are reported before any CUDA call, and the Python record layout matches the C struct."""
import ctypes as C

import numpy as np

EINVAL = 1


def test_edge_symbols_exported(pkg):
    L = pkg.library()
    for name in ("sdtgpu_edges_build", "sdtgpu_edges_buffers"):
        assert hasattr(L, name), name


def test_edge_calls_reject_null_arguments_without_a_gpu(pkg):
    L = pkg.library()
    out, ms = (C.c_uint64 * 8)(), C.c_double()
    e, q = C.c_void_p(), C.c_void_p()
    assert L.sdtgpu_edges_build(None, out, C.byref(ms)) == EINVAL
    assert L.sdtgpu_edges_build(None, None, None) == EINVAL
    assert L.sdtgpu_edges_buffers(None, C.byref(e), C.byref(q)) == EINVAL
    assert L.sdtgpu_edges_buffers(None, None, None) == EINVAL


def test_edge_layout_and_decoding(pkg):
    assert pkg.EDGE_DTYPE.itemsize == 32
    assert pkg.EDGE_DTYPE.names == ("seq", "length", "flags", "count_sum", "link", "unused")
    assert (pkg.EDGE_PALINDROME, pkg.EDGE_CYCLE) == (1, 2)
    K = 5
    codes = [np.array([0, 1, 2, 3, 3, 2, 1, 0]), np.array([2, 2, 1, 0, 3])]       # an edge of m = 3, a cycle of m = 1
    seq = np.zeros(16, dtype=np.uint8)
    edges = np.zeros(2, dtype=pkg.EDGE_DTYPE)
    edges[0] = (0, 3, 0, 0, 0, 0)
    edges[1] = (32, 1, pkg.EDGE_CYCLE, 0, 0, 0)
    for e, c in zip(edges, codes):
        for j, b in enumerate(c):
            seq[int(e["seq"]) // 4 + j // 4] |= int(b) << (6 - 2 * (j % 4))
    for i, c in enumerate(codes):
        assert np.array_equal(pkg.edge_codes(edges, seq, i, K), c)
