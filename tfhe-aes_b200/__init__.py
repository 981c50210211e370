"""tfhe-aes_b200 — B200-native WoPBS S-box engine behind the reference's `Server` / `sbox` API.

The directory name carries a hyphen (it is the name the build contract asks for), so import it
through `load_package()` in the repo-root `__graft_entry__.py`, or put this directory's parent on
`sys.path` and use `importlib` as the tests do.  The product is the C-ABI library
`libtfhe_aes_b200.so` (include/tfhe_aes_b200.h); this Python layer is a thin ctypes mirror of the
reference interface used by tests and bench.py.
"""
from .binding import (  # noqa: F401
    Engine, Params, TfaCtrStream, TfaCtrEncStream, TfaError, param_opt, param_test, param_test2, gen_lut, lut_size, lib_path, load_library,
    SBOX, INV_SBOX, mul2, mul3, mul9, mul11, mul13, mul14,
)
from .server import Server, sbox, many_sbox, many_wopbs_without_padding  # noqa: F401
from . import sharding  # noqa: F401
