"""ctypes driver for tests/csrc/k1_host_harness.cpp (the K1 scalar core compiled for the CPU; test-only)."""
import ctypes
import os
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
SRC = os.path.join(HERE, "csrc", "k1_host_harness.cpp")
LIB = os.path.join(HERE, "csrc", "libk1_host_harness.so")
MERGES = os.path.join(ROOT, "leaf_b200", "data", "clip_bpe_merges.bin")

_lib = None


def _deps_mtime():
    deps = [SRC] + [os.path.join(ROOT, "leaf_b200", "csrc", f) for f in
                    ("k1_core.cuh", "k1_tables_host.h", "k1_tables.inc", "constrain_core.cuh")]
    return max(os.path.getmtime(d) for d in deps)


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB) or os.path.getmtime(LIB) < _deps_mtime():
            subprocess.check_call(["g++", "-O2", "-shared", "-fPIC", "-o", LIB, SRC])
        L = ctypes.CDLL(LIB)
        pairs = np.fromfile(MERGES, dtype="<u4")
        L.k1h_load(pairs.ctypes.data_as(ctypes.c_void_p), ctypes.c_int(len(pairs)))
        _lib = L
    return _lib


def pack_captions(caps, encoding="utf-8"):
    blobs = [c.encode(encoding) for c in caps]
    off = np.zeros(len(caps) + 1, dtype=np.int32)
    off[1:] = np.cumsum([len(b) for b in blobs])
    data = np.frombuffer(b"".join(blobs) + b"\0", dtype=np.uint8).copy()
    return data, off


def expand_tokenize(caps, n=0, pos=None, chr_=None, sel=None, valid=None, encoding="utf-8", hf=False):
    """Returns (tokens [R,77] int32, lengths [R] int32, flags)."""
    L = lib()
    L.k1h_set_mode(1 if hf else 0)
    data, off = pack_captions(caps, encoding)
    B = len(caps)
    R = B * max(n, 1)
    tok = np.zeros((R, 77), dtype=np.int32)
    ln = np.zeros(R, dtype=np.int32)
    p = lambda a, dt: None if a is None else np.ascontiguousarray(a, dtype=dt)
    pos, chr_, sel, valid = p(pos, np.int32), p(chr_, np.int32), p(sel, np.int32), p(valid, np.uint8)
    ptr = lambda a: None if a is None else a.ctypes.data_as(ctypes.c_void_p)
    flags = L.k1h_expand_tokenize(ptr(data), ptr(off), B, n, ptr(pos), ptr(chr_), ptr(sel), ptr(valid), ptr(tok), ptr(ln))
    return tok, ln, flags


def load_words(words, abbrev=()):
    L = lib()
    def pack(ws):
        blobs = [w.encode("ascii") for w in ws if w.isascii()]
        off = np.zeros(len(blobs) + 1, dtype=np.int32)
        off[1:] = np.cumsum([len(b) for b in blobs])
        return np.frombuffer(b"".join(blobs) + b"\0", dtype=np.uint8).copy(), off, len(blobs)
    wb, wo, nw = pack(words)
    ab, ao, na = pack(abbrev)
    p = lambda a: a.ctypes.data_as(ctypes.c_void_p)
    L.cnh_load(p(wb), p(wo), nw, p(ab), p(ao), na)


def constrain_counts(caps, n, pos, chr_, sel=None):
    """Dictionary-word counts [B*n + B] (candidates, then the sentences) from the CPU-compiled filter core; flags."""
    L = lib()
    data, off = pack_captions(caps)
    B = len(caps)
    out = np.zeros(B * n + B, dtype=np.int32)
    q = lambda a, dt: None if a is None else np.ascontiguousarray(a, dtype=dt)
    pos, chr_, sel = q(pos, np.int32), q(chr_, np.int32), q(sel, np.int32)
    ptr = lambda a: None if a is None else a.ctypes.data_as(ctypes.c_void_p)
    flags = L.cnh_counts(ptr(data), ptr(off), B, n, ptr(pos), ptr(chr_), ptr(sel), ptr(out))
    return out, flags
