"""B200-native pregraph k-mer hashing for SOAPdenovo-Trans — Python host side for tests and bench.

The product is the C-ABI shared library libsdtgpu.so (include/sdtgpu.h, csrc/).  The reference is a
C program, so its host-side integration is C (host/, INTEGRATION.md); this package only binds the
same C ABI with ctypes so that tests/ and bench.py drive exactly the entry points the C driver
would.  There is no CPU fallback anywhere in this package: if the CUDA library is missing or no
GPU is visible, calls raise.

The directory name contains a hyphen, so import it through `load()` in the repo-root helper
`sdt_pkg.py` (or importlib) under the module name `soapdenovo_trans_b200`.
"""
from . import synth  # noqa: F401
from .pregraph import (  # noqa: F401
    ARC_DTYPE, DeviceReadPacker, EDGE_COUNTS, EDGE_CYCLE, EDGE_DTYPE, EDGE_PALINDROME, HIT_DTYPE, HIT_FOUND, HIT_RC, HIT_WINDOW, LIB_PATH, NODE_DTYPE, PRUNE_COUNTS, PRUNE_MINOR_TIPS, PRUNE_SINGLE_TIPS, PregraphGPU, ReadPacker, STEP_DTYPE, STEP_NONE,
    SdtGpuError, build_library,
    edge_codes, hash_kmer, hits_numpy, library, nodes_to_records, read_kmersets, steps_numpy,
)
