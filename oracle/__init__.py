"""oracle/ -- CPU restatement of the reference hot path (TEST INFRASTRUCTURE).

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline /
``--impl reference`` legs may import this package, and only as the checker or
the timed CPU baseline.  The product (pfrl_b200/) never imports it and has no
CPU fallback: its GPU classes raise if the CUDA library is missing.

Contents
  per_oracle.c      dense-heap restatement of the reference's sliding-window
                    sum/min trees and prioritized sampling (bit exact, fp64)
  replay.py         Python restatement of the n-step replay buffers, PER
                    weights and batch_experiences
  losses.py         numpy restatement of the loss / GAE arithmetic
  pyport.py         pure-Python port with the reference's cost profile, used
                    by bench.py as the timed "reference CPU path" (kind=port)
  gen_golden.py     imports the REAL reference (with gym_shim/) in the build
                    container and writes tests/golden/*.npz
  gen_golden_differential.py  the reference's side of the randomised
                    differential tests, as tests/golden/ref_*.npz
  digest.py         bit-exact fixture arrays stored by SHA-256 when large
  refimport.py      helper that puts the reference tree + gym_shim on sys.path

Parity status: pinned.  Every restatement here is checked against fixtures
generated from the real reference (tests/golden/, scripts committed).
"""
import ctypes
import os
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
_BUILD = os.path.join(_HERE, "_build")
_LIB = os.path.join(_BUILD, "libper_oracle.so")


def build(force=False):
    """Compile per_oracle.c with gcc (no FMA contraction)."""
    src = os.path.join(_HERE, "per_oracle.c")
    if (
        not force
        and os.path.exists(_LIB)
        and os.path.getmtime(_LIB) >= os.path.getmtime(src)
    ):
        return _LIB
    os.makedirs(_BUILD, exist_ok=True)
    cmd = [
        "gcc", "-O2", "-ffp-contract=off", "-fno-fast-math", "-shared", "-fPIC",
        "-o", _LIB, src, "-lm",
    ]
    subprocess.check_call(cmd)
    return _LIB


_lib = None


def lib():
    global _lib
    if _lib is None:
        path = build()
        L = ctypes.CDLL(path)
        c_i64, c_dbl, vp = ctypes.c_int64, ctypes.c_double, ctypes.c_void_p
        L.ora_per_create.restype = vp
        L.ora_per_create.argtypes = [c_i64]
        L.ora_per_destroy.argtypes = [vp]
        L.ora_per_len.restype = c_i64
        L.ora_per_len.argtypes = [vp]
        for name in ("ora_per_max_priority", "ora_per_total", "ora_per_min"):
            getattr(L, name).restype = c_dbl
            getattr(L, name).argtypes = [vp]
        for name in ("ora_per_napp", "ora_per_npop"):
            getattr(L, name).restype = c_i64
            getattr(L, name).argtypes = [vp]
        L.ora_per_append.argtypes = [vp, c_dbl]
        L.ora_per_popleft.argtypes = [vp]
        L.ora_per_sample.restype = ctypes.c_int
        L.ora_per_sample.argtypes = [vp, c_i64, vp, vp, vp, vp, vp]
        L.ora_per_set_last_priority.restype = ctypes.c_int
        L.ora_per_set_last_priority.argtypes = [vp, c_i64, vp]
        L.ora_per_leaf.restype = c_dbl
        L.ora_per_leaf.argtypes = [vp, c_i64]
        _lib = L
    return _lib
