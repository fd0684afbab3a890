"""ctypes binding of libpgica.so — the C ABI declared in include/pgica.h.

The prototypes are parsed from the header itself, so the binding cannot drift from the declared ABI.
The library is the product: if it is missing or fails to load every op raises — there is no
PyTorch/CPU fallback behind these calls.
"""
import ctypes
import os
import re
import threading

_HERE = os.path.dirname(os.path.abspath(__file__))
# PGICA_LIB_PATH selects another build of the same ABI (tools/ use it for the -DPGICA_TRACE diagnostics build)
LIB_PATH = os.environ.get("PGICA_LIB_PATH") or os.path.join(_HERE, "libpgica.so")
HEADER_PATH = os.path.join(os.path.dirname(_HERE), "include", "pgica.h")
DEBUG_HEADER_PATH = os.path.join(os.path.dirname(_HERE), "include", "pgica_debug.h")  # test / bring-up hooks

_lock = threading.Lock()
_lib = None

_SCALARS = {
    "int": ctypes.c_int,
    "int64_t": ctypes.c_int64,
    "int32_t": ctypes.c_int32,
    "uint32_t": ctypes.c_uint32,
    "float": ctypes.c_float,
    "double": ctypes.c_double,
    "size_t": ctypes.c_size_t,
}


class PgicaError(RuntimeError):
    pass


def _ctype(decl):
    decl = decl.strip()
    if decl == "void":
        return None
    if "*" in decl:
        base = decl.replace("const", "").replace("*", "").split()[0]
        if base == "size_t":
            return ctypes.POINTER(ctypes.c_size_t)
        if base == "char":
            return ctypes.c_char_p
        return ctypes.c_void_p
    base = decl.replace("const", "").split()[0]
    return _SCALARS[base]


def parse_header(path=None):
    """-> {name: (restype, [argtypes])} for every function prototype in the header (default: the product ABI plus the
    debug hooks)."""
    if path is None:
        protos = parse_header(HEADER_PATH)
        if os.path.exists(DEBUG_HEADER_PATH):
            protos.update(parse_header(DEBUG_HEADER_PATH))
        return protos
    text = open(path).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    text = re.sub(r"^\s*#.*$", "", text, flags=re.M)
    protos = {}
    for m in re.finditer(r"([A-Za-z_][\w\s\*]*?)\b(pgica_\w+)\s*\(([^)]*)\)\s*;", text):
        ret, name, args = m.group(1).strip(), m.group(2), m.group(3).strip()
        argtypes = [] if args in ("", "void") else [_ctype(a) for a in args.split(",")]
        protos[name] = (_ctype(ret) if ret != "const char*" and "char" not in ret else ctypes.c_char_p, argtypes)
    return protos


def _ensure_built(build_if_missing):
    """The in-tree library, rebuilt when csrc/ or the headers changed since it was made (source digest, _build.py).
    One process builds at a time (flock): under torchrun every rank arrives here at once."""
    from . import _build
    custom = bool(os.environ.get("PGICA_LIB_PATH"))
    if custom:
        return
    if _build.is_current():
        return
    if not build_if_missing and not os.path.exists(LIB_PATH):
        raise PgicaError(f"{LIB_PATH} is missing; run `python __graft_entry__.py build`")
    import fcntl
    with open(os.path.join(_HERE, ".libpgica.lock"), "w") as lock:
        fcntl.flock(lock, fcntl.LOCK_EX)
        try:
            if _build.is_current():
                return  # another rank built it while this one waited
            try:
                _build.build()
            except Exception as e:
                if not os.path.exists(LIB_PATH):
                    raise PgicaError(f"cannot build {LIB_PATH}: {e}") from e
                import warnings
                warnings.warn(f"libpgica.so is older than its sources and could not be rebuilt ({e}); using it as is")
        finally:
            fcntl.flock(lock, fcntl.LOCK_UN)


def load(build_if_missing=True):
    """Load the library (building it first if the in-tree .so is absent or stale and nvcc is available)."""
    global _lib
    with _lock:
        if _lib is not None:
            return _lib
        _ensure_built(build_if_missing)
        lib = ctypes.CDLL(LIB_PATH)
        for name, (restype, argtypes) in parse_header().items():
            fn = getattr(lib, name)  # AttributeError here == header/library mismatch: fail loudly
            fn.restype = restype
            fn.argtypes = argtypes
        if lib.pgica_abi_version() != 1:
            raise PgicaError("libpgica.so ABI version mismatch")
        _lib = lib
        return lib


def set_option(name, value):
    """Process-wide tuning option of the library (see pgica_set_option in include/pgica.h)."""
    check(load().pgica_set_option(name.encode(), int(value)))


def get_option(name):
    return int(load().pgica_get_option(name.encode()))


def check(rc):
    if rc != 0:
        msg = load().pgica_last_error()
        raise PgicaError(f"pgica error {rc}: {msg.decode() if msg else '?'}")
