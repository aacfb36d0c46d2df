"""ctypes loaders for the CPU oracle (oracle/liboracle.so) and the compiled reference (oracle/_ref). Test-only."""
import ctypes
import hashlib
import os
import subprocess

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ORACLE_DIR = os.path.join(ROOT, "oracle")
u32, sz, vp, ci = ctypes.c_uint32, ctypes.c_size_t, ctypes.c_void_p, ctypes.c_int
P = 0xFFF00001


def build_oracle():
    """(Re)build liboracle.so, and oracle/_ref when the reference tree is present."""
    subprocess.run(["make", "-C", ORACLE_DIR, "--no-print-directory"], check=True, capture_output=True)


def load_oracle():
    path = os.path.join(ORACLE_DIR, "liboracle.so")
    src = os.path.join(ORACLE_DIR, "gfp_oracle.c")
    if not os.path.exists(path) or os.path.getmtime(path) < os.path.getmtime(src):
        build_oracle()
    o = ctypes.CDLL(path)
    for f in ("gf_add", "gf_sub", "gf_mul", "gf_mul32", "gf_pow"):
        getattr(o, "oracle_" + f).restype = u32; getattr(o, "oracle_" + f).argtypes = [u32, u32]
    for f in ("gf_root", "gf_inv"):
        getattr(o, "oracle_" + f).restype = u32; getattr(o, "oracle_" + f).argtypes = [u32]
    o.oracle_hash.restype = u32; o.oracle_hash.argtypes = [vp, sz, sz, sz]
    o.oracle_slow_ntt.restype = None; o.oracle_slow_ntt.argtypes = [vp, sz, sz, ci]
    o.oracle_ntt.restype = ci; o.oracle_ntt.argtypes = [vp, sz, sz, ci]
    o.oracle_rs_encode.restype = ci; o.oracle_rs_encode.argtypes = [vp, sz, sz]
    o.oracle_rs_encode_by_definition.restype = None; o.oracle_rs_encode_by_definition.argtypes = [vp, vp, sz, sz]
    o.oracle_fill_A.restype = None; o.oracle_fill_A.argtypes = [vp, sz]
    o.oracle_fill_B.restype = None; o.oracle_fill_B.argtypes = [vp, sz]
    o.oracle_num_threads.restype = ci; o.oracle_num_threads.argtypes = []
    return o


def load_ref():
    path = os.path.join(ORACLE_DIR, "_ref", "libfastecc_ref.so")
    if not os.path.exists(path):
        if os.path.exists("/root/reference/ntt.cpp"):
            build_oracle()
        if not os.path.exists(path):
            return None
    r = ctypes.CDLL(path)
    for f in ("gf_add", "gf_sub", "gf_mul", "gf_pow"):
        getattr(r, "ref_" + f).restype = u32; getattr(r, "ref_" + f).argtypes = [u32, u32]
    for f in ("gf_root", "gf_inv"):
        getattr(r, "ref_" + f).restype = u32; getattr(r, "ref_" + f).argtypes = [u32]
    r.ref_mfa_ntt_flat.restype = None; r.ref_mfa_ntt_flat.argtypes = [vp, sz, sz, ci]
    r.ref_rs_encode_flat.restype = None; r.ref_rs_encode_flat.argtypes = [vp, sz, sz]
    r.ref_slow_ntt.restype = None; r.ref_slow_ntt.argtypes = [vp, sz, sz, ci]
    r.ref_num_threads.restype = ci; r.ref_num_threads.argtypes = []
    r.ref_build_flavour.restype = ctypes.c_char_p; r.ref_build_flavour.argtypes = []
    return r


def fill_A(o, N, S):
    a = np.empty((N, S), dtype=np.uint32); o.oracle_fill_A(a.ctypes.data, N * S); return a


def fill_B(o, N, S):
    a = np.empty((N, S), dtype=np.uint32); o.oracle_fill_B(a.ctypes.data, N * S); return a


def sha256(a):
    """Digest of a uint32 array's words (little-endian, row-major): stands for an output buffer too large to store."""
    return hashlib.sha256(np.ascontiguousarray(a, dtype="<u4").tobytes()).hexdigest()


def ohash(o, a):
    a = np.ascontiguousarray(a)
    return o.oracle_hash(a.ctypes.data, a.shape[0], a.shape[1], a.shape[1])


def o_ntt(o, a, inverse):
    b = np.ascontiguousarray(a).copy()
    assert o.oracle_ntt(b.ctypes.data, b.shape[0], b.shape[1], 1 if inverse else 0) == 0
    return b


def o_encode(o, a):
    b = np.ascontiguousarray(a).copy()
    assert o.oracle_rs_encode(b.ctypes.data, b.shape[0], b.shape[1]) == 0
    return b
