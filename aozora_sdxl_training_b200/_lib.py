"""ctypes binding of ``libaozora_b200.so``.

Signatures are parsed from ``include/aozora_b200.h`` (single source of truth for the C ABI).  There is no
CPU fallback: if the shared object is missing or a call fails, an exception is raised.
"""
from __future__ import annotations

import ctypes
import os
import re

HERE = os.path.dirname(os.path.abspath(__file__))
HEADER = os.path.join(os.path.dirname(HERE), "include", "aozora_b200.h")
LIB_PATH = os.path.join(HERE, "libaozora_b200.so")

_CTYPES = {
    "void*": ctypes.c_void_p, "const void*": ctypes.c_void_p, "int": ctypes.c_int, "long long": ctypes.c_longlong,
    "float": ctypes.c_float, "const char*": ctypes.c_char_p,
}


class AozoraError(RuntimeError):
    pass


def parse_header(path: str = HEADER):
    """Return {name: (restype_str, [argtype_str, ...])} for every function declared in the header."""
    text = open(path).read()
    text = re.sub(r"/\*.*?\*/", " ", text, flags=re.S)
    text = re.sub(r"^\s*#.*$", " ", text, flags=re.M)
    decls = {}
    for m in re.finditer(r"(const char\*|long long|int)\s+(aoz_\w+)\s*\(([^)]*)\)\s*;", text):
        ret, name, args = m.group(1), m.group(2), m.group(3).strip()
        argtypes = []
        if args and args != "void":
            for a in args.split(","):
                a = " ".join(a.split())
                tm = re.match(r"(const void\*|void\*|long long|int|float)\s*\w*$", a)
                if not tm:
                    raise ValueError(f"cannot parse argument {a!r} of {name}")
                argtypes.append(tm.group(1))
        decls[name] = (ret, argtypes)
    return decls


_lib = None
_decls = None


def load():
    """Load the shared library (once) and attach argtypes/restypes."""
    global _lib, _decls
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise AozoraError(
            f"{LIB_PATH} not found: build it with `python -m aozora_sdxl_training_b200.build` "
            "(there is no CPU fallback for the aozora-b200 kernels)")
    lib = ctypes.CDLL(LIB_PATH)
    _decls = parse_header()
    for name, (ret, args) in _decls.items():
        fn = getattr(lib, name)
        fn.restype = _CTYPES[ret]
        fn.argtypes = [_CTYPES[a] for a in args]
    _lib = lib
    # experiment switches (tools / A-B runs): AOZ_PDL=1 enables programmatic dependent launch, AOZ_GEMM_WIDE the 320-wide plan mode,
    # AOZ_GN_SLAB=0 selects the two-kernel GroupNorm path, AOZ_ATTN_BWD_MODE=0 the bit-reproducible two-kernel attention backward
    if os.environ.get("AOZ_PDL") is not None:
        lib.aoz_set_pdl(int(os.environ["AOZ_PDL"]))
    if os.environ.get("AOZ_GEMM_WIDE") is not None:
        lib.aoz_gemm_set_wide_mode(int(os.environ["AOZ_GEMM_WIDE"]))
    if os.environ.get("AOZ_ATTN_BWD_MODE") is not None:
        call("aoz_attn_set_bwd_mode", int(os.environ["AOZ_ATTN_BWD_MODE"]))     # refuses anything but 2 and 0
    if os.environ.get("AOZ_GN_SLAB") is not None:
        lib.aoz_groupnorm_set_slab(int(os.environ["AOZ_GN_SLAB"]))
    return lib


def last_error() -> str:
    return load().aoz_last_error().decode("utf-8", "replace")


def call(name: str, *args):
    """Call an int-returning entry point; raise AozoraError with the library's message on failure."""
    lib = load()
    rc = getattr(lib, name)(*args)
    if rc != 0:
        raise AozoraError(f"{name} failed ({rc}): {last_error()}")
    return rc


def query(name: str, *args):
    """Call a value-returning (size query) entry point."""
    return getattr(load(), name)(*args)
