"""ctypes binding of oracle/iph_oracle.c -- TEST INFRASTRUCTURE ONLY (see the header of that file)."""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB = os.path.join(HERE, "libiph_oracle.so")
_REF = os.environ.get("B200RT_REFERENCE")                      # the reference's source tree, where one is at hand
REF_TABLE = os.path.join(_REF, "src", "quemerais_IPH_model", "fsm99td12v20t80") if _REF else None

_fp = np.ctypeslib.ndpointer(dtype=np.float32, flags="C_CONTIGUOUS")
_dp = np.ctypeslib.ndpointer(dtype=np.float64, flags="C_CONTIGUOUS")
_lib = None


def build():
    if not os.path.exists(LIB) or os.path.getmtime(LIB) < os.path.getmtime(os.path.join(HERE, "iph_oracle.c")):
        subprocess.check_call(["make", "-C", HERE, "oracle"], stdout=subprocess.DEVNULL)


def _load():
    global _lib
    if _lib is None:
        build()
        lib = C.CDLL(LIB)
        lib.iph_oracle_create.restype = C.c_void_p
        lib.iph_oracle_create.argtypes = [C.c_int, C.c_int, C.c_int, C.c_float] + [_fp] * 7
        lib.iph_oracle_create_from_file.restype = C.c_void_p
        lib.iph_oracle_create_from_file.argtypes = [C.c_char_p]
        lib.iph_oracle_destroy.argtypes = [C.c_void_p]
        lib.iph_oracle_get_table.argtypes = [C.c_void_p, np.ctypeslib.ndpointer(np.int32), C.POINTER(C.c_float)] + [_fp] * 7
        lib.iph_oracle_background.argtypes = [C.c_void_p] + [C.c_float] * 4 + [C.c_int, _fp, _fp, _fp, _fp, C.c_void_p]
        lib.iph_oracle_model.argtypes = [C.c_void_p, C.c_double, _dp, C.c_int, _dp, _dp, _dp]
        _lib = lib
    return _lib


class IphOracle:
    def __init__(self, table=None, fname=None):
        self.lib = _load()
        if fname is not None:
            self.h = self.lib.iph_oracle_create_from_file(os.fsencode(fname))
        else:
            f = lambda k: np.ascontiguousarray(table[k], dtype=np.float32)
            self.h = self.lib.iph_oracle_create(int(table["kmax"]), int(table["lmax"]), int(table["ninf"]),
                                                float(table["temp"]), f("alt_au"), f("ang"), f("dans"), f("sot"),
                                                f("so"), f("sn"), f("dinf_cm3"))
        if not self.h:
            raise RuntimeError("iph oracle: bad table")

    def __del__(self):
        if getattr(self, "h", None):
            self.lib.iph_oracle_destroy(self.h)
            self.h = None

    def table(self):
        dims = np.zeros(3, np.int32)
        temp = C.c_float(0)
        NR, NK, NI = 60, 19, 5
        alt, ang, dinf = np.zeros(NR, np.float32), np.zeros(NK, np.float32), np.zeros(NI, np.float32)
        dans, sot = np.zeros(NR * NK, np.float32), np.zeros(NR * NK, np.float32)
        so, sn = np.zeros(NI * NR * NK, np.float32), np.zeros(NI * NR * NK, np.float32)
        self.lib.iph_oracle_get_table(self.h, dims, C.byref(temp), alt, ang, dans, sot, so, sn, dinf)
        k, l, n = (int(x) for x in dims)
        return dict(kmax=k, lmax=l, ninf=n, temp=float(temp.value), alt_au=alt[:k].copy(), ang=ang[:l].copy(),
                    dans=dans[:k * l].reshape(k, l).copy(), sot=sot[:k * l].reshape(k, l).copy(),
                    so=so[:n * k * l].reshape(n, k, l).copy(), sn=sn[:n * k * l].reshape(n, k, l).copy(),
                    dinf_cm3=dinf[:n].copy())

    def background(self, fs, pos, u, v, w, want_steps=False):
        n = len(u)
        fln = np.zeros(n, np.float32)
        steps = np.zeros(n, np.int32) if want_steps else None
        a = [np.ascontiguousarray(x, dtype=np.float32) for x in (u, v, w)]
        self.lib.iph_oracle_background(self.h, fs, pos[0], pos[1], pos[2], n, *a, fln,
                                       steps.ctypes.data_as(C.c_void_p) if want_steps else None)
        return (fln, steps) if want_steps else fln

    def model(self, g_lya, marspos, ra, dec):
        n = len(ra)
        out = np.zeros(n)
        self.lib.iph_oracle_model(self.h, g_lya, np.ascontiguousarray(marspos, dtype=np.float64), n,
                                  np.ascontiguousarray(ra, dtype=np.float64), np.ascontiguousarray(dec, dtype=np.float64), out)
        return out
