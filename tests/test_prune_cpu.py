"""CPU-side checks of pruning (sdtgpu_prune): the symbol is exported, argument errors are reported before any CUDA
call, and the Python names match the C ABI."""
import ctypes as C

EINVAL = 1


def test_prune_symbol_exported(pkg):
    assert hasattr(pkg.library(), "sdtgpu_prune")


def test_prune_rejects_bad_arguments_without_a_gpu(pkg):
    L = pkg.library()
    out, ms = (C.c_uint64 * 8)(), C.c_double()
    assert L.sdtgpu_prune(None, 5, 3, out, C.byref(ms)) == EINVAL
    assert L.sdtgpu_prune(None, 5, 3, None, C.byref(ms)) == EINVAL
    assert L.sdtgpu_prune(None, 5, 3, out, None) == EINVAL
    assert L.sdtgpu_prune(None, -1, 3, out, C.byref(ms)) == EINVAL
    assert L.sdtgpu_prune(None, 101, 3, out, C.byref(ms)) == EINVAL
    assert L.sdtgpu_prune(None, 5, 4, out, C.byref(ms)) == EINVAL


def test_prune_names(pkg):
    assert len(pkg.PRUNE_COUNTS) == 8 and len(set(pkg.PRUNE_COUNTS)) == 8
    assert pkg.PRUNE_COUNTS[-1] == "vertices"
    assert (pkg.PRUNE_SINGLE_TIPS, pkg.PRUNE_MINOR_TIPS) == (1, 2)
