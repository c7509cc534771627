"""ctypes binding of tests/scaled_oracle.c -- TEST INFRASTRUCTURE ONLY: the reduced-size decode's CPU restatement.

The library is compiled on first use into the system temporary directory (per user, keyed by the sources' contents),
so that the repository tree is never written to."""
from __future__ import annotations

import ctypes
import hashlib
import os
import subprocess
import tempfile

import numpy as np

from oracle import port

_HERE = os.path.dirname(os.path.abspath(__file__))
_SRC = os.path.join(_HERE, "scaled_oracle.c")
_DEPS = [_SRC, os.path.join(os.path.dirname(_HERE), "oracle", "jpeg_oracle.c")]
# the flags of oracle/Makefile: float results must not depend on contraction or fast-math
CFLAGS = ["-O2", "-ffp-contract=off", "-fno-fast-math", "-std=c99", "-Wall", "-Wextra", "-fPIC", "-shared"]
_lib = None


def build() -> str:
    h = hashlib.sha256()
    for p in _DEPS:
        with open(p, "rb") as fh:
            h.update(fh.read())
    h.update(" ".join(CFLAGS).encode())
    so = os.path.join(tempfile.gettempdir(), f"hjd_scaled_oracle_{os.getuid()}_{h.hexdigest()[:16]}.so")
    if not os.path.exists(so):
        tmp = f"{so}.{os.getpid()}.tmp"
        subprocess.check_call([os.environ.get("CC", "gcc")] + CFLAGS + [_SRC, "-o", tmp, "-lm"])
        os.replace(tmp, so)
    return so


def lib() -> ctypes.CDLL:
    global _lib
    if _lib is None:
        L = ctypes.CDLL(build())
        L.hjdo_scaled_block.restype = None
        L.hjdo_scaled_block.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p, ctypes.c_int]
        L.hjdo_decode_scaled.restype = ctypes.c_int
        L.hjdo_decode_scaled.argtypes = [ctypes.c_char_p, ctypes.c_size_t, ctypes.c_int, ctypes.c_void_p,
                                         ctypes.POINTER(ctypes.c_uint), ctypes.POINTER(ctypes.c_uint)]
        L.hjdo_ycc_cube.restype = None
        L.hjdo_ycc_cube.argtypes = [ctypes.c_int, ctypes.c_void_p]
        L.hjdo_dc_only.restype = ctypes.c_long
        L.hjdo_dc_only.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_long, ctypes.c_int, ctypes.c_void_p]
        _lib = L
    return _lib


def scaled_block(coef64: np.ndarray, q64: np.ndarray, n: int) -> np.ndarray:
    """One block through the reduced IDCT with n = 8, 4, 2 or 1 samples per side: uint8 [n, n] (row y, column x)."""
    coef64 = np.ascontiguousarray(coef64, dtype=np.int16)
    q64 = np.ascontiguousarray(q64, dtype=np.float32)
    out = np.zeros((n, n), dtype=np.uint8)
    lib().hjdo_scaled_block(coef64.ctypes.data, q64.ctypes.data, n, out.ctypes.data, n)
    return out


def ycc_cube(fma: bool = False) -> np.ndarray:
    """hjdo_ycc_to_rgb on every byte triple: uint8 [Y, Cb, Cr, channel] (256, 256, 256, 3).  fma: every product
    contracted into an FMA instead."""
    out = np.empty((256, 256, 256, 3), dtype=np.uint8)
    lib().hjdo_ycc_cube(int(fma), out.ctypes.data)
    return out


def dc_only(c0, q0, n: int) -> np.ndarray:
    """The sample of each DC-only block (quantised DC c0[i], DC table entry q0[i]) through the single-block decode
    (n = 8) or the reduced IDCT (n = 4, 2, 1): uint8 [len(c0)].  Asserts that every block decodes flat."""
    c0 = np.ascontiguousarray(c0, dtype=np.int32)
    q0 = np.ascontiguousarray(np.broadcast_to(q0, c0.shape), dtype=np.int32)
    out = np.empty(c0.shape, dtype=np.uint8)
    uneven = lib().hjdo_dc_only(c0.ctypes.data, q0.ctypes.data, c0.size, n, out.ctypes.data)
    assert uneven == 0, f"{uneven} samples of DC-only blocks differ from their block's first sample"
    return out


def decode_scaled(jpg: bytes, shift: int):
    """Decode at 1 / 2**shift of the source size (shift 0..3): dict(rc, width, height, rgb[ceil(H/d), ceil(W/d), 3])."""
    g = port.info(jpg)
    if g["rc"] != 0:
        return dict(rc=g["rc"], rgb=None)
    d = 1 << shift
    ow, oh = -(-g["width"] // d), -(-g["height"] // d)
    rgb = np.zeros((oh, ow, 3), dtype=np.uint8)
    w, h = ctypes.c_uint(), ctypes.c_uint()
    rc = lib().hjdo_decode_scaled(jpg, len(jpg), shift, rgb.ctypes.data, ctypes.byref(w), ctypes.byref(h))
    assert (w.value, h.value) == (ow, oh)
    return dict(rc=rc, width=w.value, height=h.value, rgb=rgb)
