"""CPU-side checks of the lookup entry points (sdtgpu_lookup_kmers_device, sdtgpu_lookup_reads_device): argument
errors are reported before any CUDA call, and the Python hit layout matches the C struct."""
import ctypes as C

import numpy as np


def test_lookup_calls_reject_null_arguments_without_a_gpu(pkg):
    L = pkg.library()
    buf = (C.c_uint64 * 8)()
    assert L.sdtgpu_lookup_kmers_device(None, None, 0, None) == 1                   # SDTGPU_EINVAL
    assert L.sdtgpu_lookup_kmers_device(None, buf, 1, buf) == 1
    assert L.sdtgpu_lookup_reads_device(None, None, None, None, 0, 0, 0, None) == 1
    assert L.sdtgpu_lookup_reads_device(None, buf, None, None, 1, 100, 28, buf) == 1


def test_hit_layout(pkg):
    assert pkg.HIT_DTYPE.itemsize == 16 and pkg.HIT_DTYPE.names == ("count", "l_links", "rword", "status")
    assert (pkg.HIT_WINDOW, pkg.HIT_FOUND, pkg.HIT_RC) == (1, 2, 4)
    raw = np.arange(24, dtype=np.int32).reshape(2, 3, 4)
    h = pkg.hits_numpy(raw)
    assert h.shape == (2, 3) and h[1, 2]["status"] == 23 and h[0, 1]["count"] == 4
