"""ctypes binding of libsfb200.so (the C ABI declared in include/sfb200.h).

The prototypes are parsed from the header itself so the binding can never drift from the ABI; the library must have
been built in-tree (`python -c "import __graft_entry__ as g; g.build()"` or `make -C sample_factory_b200/csrc`).
There is NO fallback: if the shared library is missing, importing this module raises.
"""
from __future__ import annotations

import ctypes
import os
import re
from typing import Dict, List, Tuple

_HERE = os.path.dirname(os.path.abspath(__file__))
HEADER_PATH = os.path.join(os.path.dirname(_HERE), "include", "sfb200.h")
LIB_PATH = os.path.join(_HERE, "libsfb200.so")

_SCALARS = {
    "int": ctypes.c_int,
    "int32_t": ctypes.c_int32,
    "int64_t": ctypes.c_int64,
    "uint64_t": ctypes.c_uint64,
    "float": ctypes.c_float,
    "double": ctypes.c_double,
}


def parse_header(path: str = HEADER_PATH) -> Dict[str, Tuple[str, List[Tuple[str, str]]]]:
    """-> {function name: (return type, [(arg type, arg name), ...])} for every prototype in the header."""
    text = open(path).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    text = "\n".join(line for line in text.splitlines() if not line.lstrip().startswith("#"))
    protos = {}
    for m in re.finditer(r"([A-Za-z_][\w\s\*]*?)\b(sfb200_\w+)\s*\(([^)]*)\)\s*;", text):
        ret = " ".join(m.group(1).split())
        name = m.group(2)
        args = []
        arg_text = m.group(3).strip()
        if arg_text and arg_text != "void":
            for a in arg_text.split(","):
                a = " ".join(a.split())
                mm = re.match(r"(.*?)(\w+)$", a)
                args.append((mm.group(1).strip().replace(" *", "*"), mm.group(2)))
        protos[name] = (ret, args)
    return protos


def header_abi_version(path: str = HEADER_PATH) -> int:
    """SFB200_ABI_VERSION as defined in the header: the version the library built from it must report."""
    return int(re.search(r"^#define SFB200_ABI_VERSION (\d+)", open(path).read(), flags=re.M).group(1))


ABI_VERSION = header_abi_version()


def _ctype(t: str):
    if t.endswith("*"):
        return ctypes.c_char_p if t == "const char*" else ctypes.c_void_p
    return _SCALARS[t]


class SfbError(RuntimeError):
    pass


class _Lib:
    def __init__(self):
        if not os.path.isfile(LIB_PATH):
            raise ImportError(
                f"{LIB_PATH} not found: the CUDA extension has not been built. Run __graft_entry__.build() "
                "(or `make -C sample_factory_b200/csrc`). There is no CPU fallback."
            )
        self.cdll = ctypes.CDLL(LIB_PATH, mode=ctypes.RTLD_LOCAL)
        self.protos = parse_header()
        for name, (ret, args) in self.protos.items():
            fn = getattr(self.cdll, name)  # AttributeError if the symbol is not exported
            fn.restype = _ctype(ret)
            fn.argtypes = [_ctype(t) for t, _ in args]
        assert self.cdll.sfb200_abi_version() == ABI_VERSION, "libsfb200 ABI version mismatch"

    def call(self, name: str, *args):
        """Invoke an `int sfb200_*` entry point; raises SfbError with the library's message on failure."""
        rc = getattr(self.cdll, name)(*args)
        if rc != 0:
            msg = self.cdll.sfb200_last_error()
            raise SfbError(f"{name} failed (rc={rc}): {msg.decode() if msg else '?'}")

    def query(self, name: str, *args):
        """Invoke a value-returning entry point (workspace sizes, sm_count, ...)."""
        return getattr(self.cdll, name)(*args)


_lib = None


def lib() -> _Lib:
    global _lib
    if _lib is None:
        _lib = _Lib()
    return _lib
