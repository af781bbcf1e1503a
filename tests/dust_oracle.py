"""ctypes face of tests/native/dust_oracle.c, the CPU restatement of dustmasker's symmetric DUST that the GPU
masking is checked against.  TEST INFRASTRUCTURE ONLY.  The shared object is compiled on first use into the
system's temporary directory, named after a hash of the source, so the repository tree is never written."""
from __future__ import annotations

import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

SRC = os.path.join(os.path.dirname(os.path.abspath(__file__)), "native", "dust_oracle.c")
_lib = None


def lib() -> C.CDLL:
    global _lib
    if _lib is not None:
        return _lib
    digest = hashlib.sha1(open(SRC, "rb").read()).hexdigest()[:16]
    so = os.path.join(tempfile.gettempdir(), f"nh_dust_oracle_{os.getuid()}_{digest}.so")
    if not os.path.exists(so):
        fd, tmp = tempfile.mkstemp(suffix=".so", dir=os.path.dirname(so))
        os.close(fd)
        cc = "/usr/bin/gcc" if os.path.exists("/usr/bin/gcc") else "gcc"
        subprocess.check_call([cc, "-O3", "-fopenmp", "-fPIC", "-shared", "-Wall", "-Wextra", "-std=c11", "-o", tmp,
                               SRC])
        os.replace(tmp, so)  # atomic: concurrent first users each compile, one copy wins
    L = C.CDLL(so)
    L.dust_oracle_mask.restype = C.c_int
    L.dust_oracle_mask.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.c_int, C.c_int, C.c_int, C.c_void_p]
    _lib = L
    return L


def dust_mask_batch(bases: np.ndarray, offsets: np.ndarray, window: int = 64, level: int = 20,
                    threads: int = 0) -> np.ndarray:
    """Records concatenated in `bases` (offsets[n+1]): masked bases lower-cased, every other byte upper-cased."""
    bases = np.ascontiguousarray(bases, dtype=np.uint8)
    offsets = np.ascontiguousarray(offsets, dtype=np.uint64)
    out = np.empty(len(bases), np.uint8)
    if lib().dust_oracle_mask(bases.ctypes.data, offsets.ctypes.data, len(offsets) - 1, int(window), int(level),
                              int(threads), out.ctypes.data):
        raise ValueError(f"dust_oracle_mask refused window={window} level={level}")
    return out


def dust_mask(seqs, window: int = 64, level: int = 20, threads: int = 0) -> list[bytes]:
    """The same over a list of sequences (bytes or str)."""
    seqs = [s.encode() if isinstance(s, str) else bytes(s) for s in seqs]
    offsets = np.zeros(len(seqs) + 1, np.uint64)
    np.cumsum([len(s) for s in seqs], out=offsets[1:])
    data = np.frombuffer(b"".join(seqs) or b"\0", np.uint8)[:int(offsets[-1])]
    out = dust_mask_batch(data, offsets, window, level, threads).tobytes()
    return [out[int(offsets[i]):int(offsets[i + 1])] for i in range(len(seqs))]
