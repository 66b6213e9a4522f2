"""Test-side bindings for inverse dynamics: the oracle's mj_inverse (tests/native/ox_inverse_oracle.cpp, on top of the oracle's
own source) and the inverse kernel's per-env body on the host (tests/native/ox_inverse_hostcheck.cpp, on top of the host
instantiation). Both are compiled into one checker library, libox_inverse_check.so, the first time a test needs it: into
build/inverse_check/ when the tree is writable, else into a per-user temporary directory. Neither is reachable from the product."""
from __future__ import annotations

import ctypes as C
import glob
import os
import subprocess
import tempfile

import numpy as np

from support import HostBatch, OracleData

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NATIVE = os.path.join(ROOT, "tests", "native")
CSRC = os.path.join(ROOT, "oxide_control_b200", "csrc")
SOURCES = [os.path.join(NATIVE, "ox_inverse_oracle.cpp"), os.path.join(NATIVE, "ox_inverse_hostcheck.cpp"),
           os.path.join(CSRC, "ox_spec_registry.cpp")]
DEPS = SOURCES + [os.path.join(ROOT, "oracle", "ox_oracle.cpp"), os.path.join(NATIVE, "ox_hostcheck.cu"),
                  os.path.join(ROOT, "include", "ox_b200.h")] + glob.glob(os.path.join(CSRC, "*.cuh")) + glob.glob(os.path.join(CSRC, "*.h"))
CXXFLAGS = ["-std=c++17", "-O2", "-fPIC", "-shared", "-fvisibility=hidden", "-pthread", "-Wno-unknown-pragmas",
            "-Wno-aggressive-loop-optimizations", "-DOX_SPEC_HOST", "-I" + CSRC]


def _lib_dir() -> str:
    d = os.path.join(ROOT, "build", "inverse_check")
    try:
        os.makedirs(d, exist_ok=True)
        if os.access(d, os.W_OK):
            return d
    except OSError:
        pass
    d = os.path.join(tempfile.gettempdir(), f"ox_inverse_check_{os.getuid()}")
    os.makedirs(d, exist_ok=True)
    return d


def _build() -> str:
    path = os.path.join(_lib_dir(), "libox_inverse_check.so")
    if not os.path.exists(path) or os.path.getmtime(path) < max(os.path.getmtime(p) for p in DEPS):
        tmp = f"{path}.{os.getpid()}.tmp"     # concurrent test workers: each builds its own file, the rename is atomic
        subprocess.check_call([os.environ.get("CXX", "g++"), *CXXFLAGS, "-o", tmp, *SOURCES])
        os.replace(tmp, path)
    return path


_lib = None


def inverse_lib() -> C.CDLL:
    global _lib
    if _lib is None:
        L = C.CDLL(_build())
        P = C.c_void_p
        L.oxo_make_data.restype = P
        L.oxo_make_data.argtypes = [P]
        L.oxo_free_data.argtypes = [P]
        for f in ("oxo_reset", "oxo_forward", "oxo_step"):
            getattr(L, f).argtypes = [P, P]
        L.oxo_inverse.argtypes = [P, P, P]
        L.oxo_field.restype = C.POINTER(C.c_double)
        L.oxo_field.argtypes = [P, C.c_char_p, C.POINTER(C.c_int32)]
        L.oxo_int.restype = C.c_int32
        L.oxo_int.argtypes = [P, C.c_char_p]
        L.oxo_int_field.restype = C.POINTER(C.c_int32)
        L.oxo_int_field.argtypes = [P, C.c_char_p, C.POINTER(C.c_int32)]
        L.hc_create.restype = P
        L.hc_create.argtypes = [P, C.c_int, C.c_int, C.c_int, C.c_int, C.c_double]
        L.hc_free.argtypes = [P]
        L.hc_stride.argtypes = [P]
        L.hc_reset.argtypes = [P]
        L.hc_forward.argtypes = [P]
        L.hc_inverse.argtypes = [P]
        L.hc_field.restype = P
        L.hc_field.argtypes = [P, C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int)]
        _lib = L
    return _lib


class InverseOracle(OracleData):
    """One oracle env (the OracleData interface) with inverse(); field("qfrc_inverse") holds its result."""

    def __init__(self, model):
        self.model = model
        self.L = inverse_lib()
        self.t = C.c_void_p(model.tables_ptr)
        self.d = C.c_void_p(self.L.oxo_make_data(self.t))
        self.qfrc_inverse = np.zeros(model.nv)

    def field(self, name: str) -> np.ndarray:
        return self.qfrc_inverse if name == "qfrc_inverse" else super().field(name)

    def inverse(self):
        self.L.oxo_inverse(self.t, self.d, self.qfrc_inverse.ctypes.data_as(C.c_void_p))


class InverseHostBatch(HostBatch):
    """HostBatch (the product's stage templates on the CPU) with inverse(): the body of k_inverse for every env."""

    def __init__(self, model, nenv, precision="f64"):
        from oxide_control_b200 import _abi as A
        self.A = A
        self.L = inverse_lib()
        self.nenv = nenv
        self.precision = precision
        self.h = C.c_void_p(self.L.hc_create(C.c_void_p(model.tables_ptr), nenv, 1 if precision == "f64" else 0, 0, 0, -1.0))
        self.stride = self.L.hc_stride(self.h)
        self.L.hc_reset(self.h)

    def inverse(self):
        self.L.hc_inverse(self.h)
