"""TEST INFRASTRUCTURE ONLY -- ctypes binding of oracle/locate_oracle.c (wso_locate)."""
import ctypes
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SRC = os.path.join(_HERE, 'locate_oracle.c')
_SO = os.path.join(_HERE, 'liblocate_oracle.so')
_lib = None


def build(force: bool = False) -> str:
    if force or not os.path.exists(_SO) or os.path.getmtime(_SO) < os.path.getmtime(_SRC):
        tmp = _SO + f'.{os.getpid()}.tmp'
        subprocess.check_call(['gcc', '-O2', '-fPIC', '-ffp-contract=off', '-fno-fast-math', '-shared', '-o', tmp,
                               _SRC, '-lm'])
        os.replace(tmp, _SO)
    return _SO


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(_SO):
            build()
        f = ctypes.CDLL(_SO).wso_locate
        f.restype = ctypes.c_int
        f.argtypes = [ctypes.POINTER(ctypes.c_double), ctypes.c_int64, ctypes.POINTER(ctypes.c_double),
                      ctypes.POINTER(ctypes.c_int32), ctypes.POINTER(ctypes.c_int32), ctypes.c_int, ctypes.c_int,
                      ctypes.c_int, ctypes.c_double, ctypes.POINTER(ctypes.c_int64),
                      ctypes.POINTER(ctypes.c_int64), ctypes.POINTER(ctypes.c_double)]
        _lib = f
    return _lib


def _p(a, ty):
    return a.ctypes.data_as(ctypes.POINTER(ty))


def locate(x, tb, mv, offset=0.35):
    """wso_locate: (lo, hi, score, status) of the STR window search in the whole read ``x``."""
    x = np.ascontiguousarray(x, dtype=np.float64)
    v = np.ascontiguousarray(tb.values, dtype=np.float64)
    ip = np.ascontiguousarray(tb.in_ptr, dtype=np.int32)
    ii = np.ascontiguousarray(tb.in_idx, dtype=np.int32)
    lo, hi, score = ctypes.c_int64(), ctypes.c_int64(), ctypes.c_double()
    st = lib()(_p(x, ctypes.c_double), len(x), _p(v, ctypes.c_double), _p(ip, ctypes.c_int32),
               _p(ii, ctypes.c_int32), len(v), int(tb.endstate), int(mv), float(offset), ctypes.byref(lo),
               ctypes.byref(hi), ctypes.byref(score))
    if st == 3:
        raise MemoryError('wso_locate')
    return int(lo.value), int(hi.value), float(score.value), int(st)


def locate_batch(signals, tbs, mv, offset=0.35, threads=8):
    """``locate`` for every read (``tbs[r]`` its automaton) over ``threads`` Python threads (the C call
    releases the GIL).  Returns lo, hi (int64), score (float64), status (int32) arrays."""
    from concurrent.futures import ThreadPoolExecutor
    with ThreadPoolExecutor(max(1, int(threads))) as ex:
        res = list(ex.map(lambda a: locate(a[0], a[1], mv, offset), zip(signals, tbs)))
    lo, hi, score, status = (np.array(c) for c in zip(*res)) if res else (np.zeros(0),) * 4
    return lo.astype(np.int64), hi.astype(np.int64), score.astype(np.float64), status.astype(np.int32)
