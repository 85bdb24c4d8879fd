"""kyber-rs_b200 — host side of the B200-native edwards25519 hot path of teleconsys/kyber-rs.

Everything here is a thin ctypes binding over the C ABI in ``include/kyber_b200.h``
(``libkyber_b200.so``, built by ``csrc/Makefile``), plus a host-side mirror of the reference's
operator surface for this path (``host.py``: ``Point``, ``Scalar``, ``PubPoly``, ``eddsa`` /
``schnorr`` verify) so the parity tests read like the reference's own tests.

There is NO CPU implementation in this package: if the CUDA library is missing or no B200 is
visible, ``Context()`` raises.  Import name: the directory is literally ``kyber-rs_b200`` (the
layout the project asks for); use ``importlib.import_module("kyber-rs_b200")`` or the
``kyber_rs_b200`` alias module at the repository root.
"""
from .binding import (  # noqa: F401
    Context,
    KeySet,
    MultiContext,
    MultiKeySet,
    KBError,
    LIB_PATH,
    SIG_STATUS_NAMES,
    FLAG_SHARED_POINT,
    FLAG_VARTIME,
    load_library,
)
from . import host  # noqa: F401
from . import sharding  # noqa: F401

__all__ = ["Context", "KeySet", "MultiContext", "MultiKeySet", "KBError", "LIB_PATH", "SIG_STATUS_NAMES", "FLAG_VARTIME", "FLAG_SHARED_POINT", "load_library", "host", "sharding"]
