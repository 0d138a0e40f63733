"""xpng_b200 — B200-native (sm_100a) implementation of the xPNG encode/decode hot path.

The product is the shared library `libxpng_b200.so` (hand-written CUDA kernels behind a C ABI,
include/xpng_b200.h, plus the reference-compatible C file API of include/xpng.h / include/seven.h).
This package is the thin ctypes mirror used by the tests and bench.py; it never falls back to a CPU
implementation: importing `codec` without the built library, or creating a Codec without a CUDA
device, raises.
"""
import os as _os

# A batch call keeps up to 24 CUDA streams busy; with the driver's default of 8 hardware queues they would wait on each
# other.  The driver reads this when CUDA initialises, so it must be in place before the process's first CUDA call.  It is
# taken out of the environment again once a codec context exists (codec.Codec): child processes (the one-image CLI) should
# not inherit it, 32 queues cost ~2.5 s of start-up (tools/ctx_time.py).
CONNECTIONS_SET_HERE = "CUDA_DEVICE_MAX_CONNECTIONS" not in _os.environ
_os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")

from .codec import Codec, LibraryMissing, inverse_op, lib, lib_path, region_tiles, xpng_store, xpng_load, load_7, store_7  # noqa: F401
