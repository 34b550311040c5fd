"""ctypes loader for libvidar_b200.so (the C ABI declared in include/vidar_b200.h).

There is no CPU fallback anywhere in this package: if the library is missing or a call
fails, a RuntimeError is raised.
"""
import ctypes as C
import os
import re

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libvidar_b200.so")
HEADER = os.path.join(os.path.dirname(_HERE), "include", "vidar_b200.h")

_lib = None

_CTYPES = {
    "const float*": C.c_void_p, "float*": C.c_void_p, "const int64_t*": C.c_void_p,
    "const int32_t*": C.c_void_p, "int32_t*": C.c_void_p, "const unsigned char*": C.c_void_p, "unsigned char*": C.c_void_p, "int64_t*": C.c_void_p,
    "unsigned long long*": C.c_void_p, "double*": C.c_void_p,
    "void*": C.c_void_p, "int": C.c_int, "float": C.c_float, "long long": C.c_longlong,
}


def declared_symbols():
    """[(name, [ctype,...])] for every `int vidar_*(...)` prototype in the header."""
    with open(HEADER) as fh:
        src = re.sub(r"/\*.*?\*/", "", fh.read(), flags=re.S)
    out = []
    for m in re.finditer(r"\bint\s+(vidar_\w+)\s*\(([^)]*)\)\s*;", src):
        args = []
        for a in m.group(2).split(","):
            a = " ".join(a.split())
            ty = a.rsplit(" ", 1)[0] if " " in a else a
            ty = ty.replace(" *", "*")
            args.append(_CTYPES[ty])
        out.append((m.group(1), args))
    return out


def lib():
    """Load (once) and return the CDLL.  Raises if the CUDA library was not built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} is missing: build it with `python -m vidar_b200.build` "
            "(there is no CPU/PyTorch fallback for these ops)")
    L = C.CDLL(LIB_PATH)
    L.vidar_last_error.restype = C.c_char_p
    L.vidar_version.restype = C.c_char_p
    L.vidar_launch_count.restype = C.c_int64
    for name, argtypes in declared_symbols():
        fn = getattr(L, name)          # AttributeError here = header/library mismatch
        fn.argtypes = argtypes
        fn.restype = C.c_int
    _lib = L
    return L


def launch_count():
    return int(lib().vidar_launch_count())


def check(rc):
    if rc != 0:
        msg = lib().vidar_last_error().decode()
        raise RuntimeError(msg or f"libvidar_b200 error {rc}")


def stream_ptr(device=None):
    return C.c_void_p(torch.cuda.current_stream(device).cuda_stream)


def ptr(t):
    return C.c_void_p(t.data_ptr()) if t is not None else None


def require_cuda(**tensors):
    """Mirror of the reference CHECK_INPUT (third_lib/dvr/dvr.cpp:28-34): CUDA + contiguous."""
    for name, t in tensors.items():
        if t is None:
            continue
        if not t.is_cuda:
            raise RuntimeError(f"{name} must be a CUDA tensor")
        if not t.is_contiguous():
            raise RuntimeError(f"{name} must be contiguous")


def require_aligned(nbytes=16, **tensors):
    """The vector kernels use 16-byte loads / reductions (ld.global.v4, red.global.v4): a contiguous
    view with an odd storage offset would fault with a misaligned address."""
    for name, t in tensors.items():
        if t is not None and t.numel() and t.data_ptr() % nbytes:
            raise RuntimeError(f"{name} must be {nbytes}-byte aligned (data_ptr {t.data_ptr():#x}); "
                               f"pass a fresh tensor, e.g. `{name}.clone()`")


def aligned(t, nbytes=16):
    """t itself when its storage is `nbytes`-aligned, else a (fresh, aligned) copy."""
    return t if (t.numel() == 0 or t.data_ptr() % nbytes == 0) else t.clone()
