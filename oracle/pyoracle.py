"""TEST INFRASTRUCTURE ONLY. ctypes wrapper of oracle/liboracle.so (restatement) and
oracle/_ref/libpalace_qf_ref.so (the reference's own QFunction headers compiled in place).
Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference leg import this."""
from __future__ import annotations

import atexit
import ctypes as C
import os
import shutil
import subprocess
import tempfile

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = None
_REF = None

CURLCURL, ND_MASS, CURLCURL_MASS, H1_DIFFUSION, ND_WEAKCURL, ND_MIXEDCURL = 0, 1, 2, 3, 4, 5

_dp = np.ctypeslib.ndpointer(dtype=np.float64, flags="C_CONTIGUOUS")
_ip = np.ctypeslib.ndpointer(dtype=np.int32, flags="C_CONTIGUOUS")


def build():
    subprocess.check_call(["make", "-s", "-C", _HERE], stdout=subprocess.DEVNULL)


def lib():
    global _LIB
    if _LIB is None:
        path = os.path.join(_HERE, "liboracle.so")
        if not os.path.exists(path):
            build()
        _LIB = C.CDLL(path)
        _LIB.orc_nd_hex_ndof.restype = C.c_int
    return _LIB


def use_native_build():
    """Timed CPU baseline only (bench.py): rebuild the oracle with -march=native ON THIS HOST into a temporary
    directory (the source tree may be read-only) and switch to it, so the baseline is not handicapped by the portable
    ISA level of the prebuilt library. Returns True when the native build is in use."""
    global _LIB
    try:
        out = tempfile.mkdtemp(prefix="b2p_oracle_native_")
        atexit.register(shutil.rmtree, out, ignore_errors=True)
        subprocess.check_call(["make", "-s", "-C", _HERE, "native", "NATIVE_DIR=" + out], stdout=subprocess.DEVNULL,
                              stderr=subprocess.DEVNULL, timeout=300)
        _LIB = C.CDLL(os.path.join(out, "liboracle.so"))
        _LIB.orc_nd_hex_ndof.restype = C.c_int
        return True
    except Exception:
        return False


def ref():
    """The compiled reference QFunctions, or None when oracle/_ref was never built."""
    global _REF
    if _REF is None:
        path = os.path.join(_HERE, "_ref", "libpalace_qf_ref.so")
        if not os.path.exists(path):
            return None
        _REF = C.CDLL(path)
    return _REF


def _p(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def gauss_legendre(n):
    x = np.empty(n); w = np.empty(n)
    lib().orc_gauss_legendre(n, _p(x), _p(w))
    return x, w


def gauss_lobatto(n):
    x = np.empty(n)
    lib().orc_gauss_lobatto(n, _p(x))
    return x


def nd_hex_dofmap(p):
    m = np.empty(3 * p * (p + 1) ** 2, dtype=np.int32)
    lib().orc_nd_hex_dofmap(p, _p(m))
    return m


def nd_hex_1d(p, q1d):
    Bo = np.empty((q1d, p)); Bc = np.empty((q1d, p + 1)); Gc = np.empty((q1d, p + 1)); qw = np.empty(q1d)
    lib().orc_nd_hex_1d(p, q1d, _p(Bo), _p(Bc), _p(Gc), _p(qw))
    return Bo, Bc, Gc, qw


def nd_hex_tables(p, q1d):
    P = 3 * p * (p + 1) ** 2
    Q = q1d ** 3
    interp = np.empty((3, Q, P)); curl = np.empty((3, Q, P)); qw = np.empty(Q)
    lib().orc_nd_hex_tables(p, q1d, _p(interp), _p(curl), _p(qw))
    return interp, curl, qw


def h1_hex_tables(p, q1d):
    P = (p + 1) ** 3
    Q = q1d ** 3
    interp = np.empty((Q, P)); grad = np.empty((3, Q, P)); qw = np.empty(Q)
    lib().orc_h1_hex_tables(p, q1d, _p(interp), _p(grad), _p(qw))
    return interp, grad, qw


def geom_hex_qdata(xe, attr, k, q1d):
    xe = np.ascontiguousarray(xe, dtype=np.float64)
    attr = np.ascontiguousarray(attr, dtype=np.int32)
    ne = xe.shape[0]
    qd = np.empty((ne, 11, q1d ** 3))
    lib().orc_geom_hex_qdata(ne, k, q1d, _p(xe), _p(attr), _p(qd))
    return qd


def apply_D(kind, ctx, qdata, u, c):
    Q = qdata.shape[-1]
    v = np.zeros((3, Q)); w = np.zeros((3, Q))
    lib().orc_apply_D(kind, _p(ctx), Q, _p(np.ascontiguousarray(qdata)), _p(u), _p(c), _p(v), _p(w))
    return v, w


def apply_add(kind, interp, deriv, idx, orient, qdata, ctx, x, y):
    ne, P = idx.shape
    Q = qdata.shape[-1]
    assert idx.dtype == np.int32 and (orient is None or orient.dtype == np.int8)
    lib().orc_apply_add(kind, ne, P, Q, _p(interp), _p(deriv), _p(idx), _p(orient), _p(qdata), _p(ctx), _p(x), _p(y))
    return y


def apply_add_co(kind, interp, deriv, idx, curl_orient, qdata, ctx, x, y):
    """y += A x with the tridiagonal curl-oriented restriction (int8 [ne][P][3], row-major)."""
    ne, P = idx.shape
    Q = qdata.shape[-1]
    co = np.ascontiguousarray(curl_orient, dtype=np.int8)
    lib().orc_apply_add_co(kind, ne, P, Q, _p(interp), _p(deriv), _p(idx), _p(co), _p(qdata), _p(ctx), _p(x), _p(y))
    return y


def element_matrices(kind, interp, deriv, orient, qdata, ctx, P):
    ne = qdata.shape[0]
    Q = qdata.shape[-1]
    Ae = np.empty((ne, P, P))
    lib().orc_element_matrices(kind, ne, P, Q, _p(interp), _p(deriv), _p(orient), _p(qdata), _p(ctx), _p(Ae))
    return Ae


def diag_add(kind, interp, deriv, idx, qdata, ctx, diag):
    ne, P = idx.shape
    Q = qdata.shape[-1]
    lib().orc_diag_add(kind, ne, P, Q, _p(interp), _p(deriv), _p(idx), _p(qdata), _p(ctx), _p(diag))
    return diag


def apply_add_mt(nthreads, kind, interp, deriv, idx, orient, qdata, ctx, x, y):
    ne, P = idx.shape
    Q = qdata.shape[-1]
    lib().orc_apply_add_mt(int(nthreads), kind, ne, P, Q, _p(interp), _p(deriv), _p(idx), _p(orient), _p(qdata), _p(ctx), _p(x),
                           _p(y), C.c_longlong(y.size))
    return y


def physical_cores():
    lib().orc_physical_cores.restype = C.c_int
    return int(lib().orc_physical_cores())


class BlockedApply:
    """The reference arm of bench.py: dense-basis apply in blocks of 8 elements (one SIMD lane per element, libCEED
    /cpu/self/opt/blocked style) on a persistent pool of threads pinned one per physical core, with a precomputed
    transposed restriction for the scatter-add. Same arithmetic per element as apply_add (tests/test_oracle_identities.py)."""

    def __init__(self, kind, interp, deriv, idx, orient, qdata, ctx, lsize, nthreads=0):
        L = lib()
        L.orc_pool_create.restype = C.c_void_p
        L.orc_blocked_setup.restype = C.c_void_p
        L.orc_pool_threads.restype = C.c_int
        self.kind, self.interp, self.deriv, self.idx, self.orient, self.qdata, self.ctx = kind, interp, deriv, idx, orient, qdata, ctx
        self.ne, self.P = idx.shape
        self.Q = qdata.shape[-1]
        self.pool = C.c_void_p(L.orc_pool_create(int(nthreads)))
        self.threads = int(L.orc_pool_threads(self.pool))
        self.setup = C.c_void_p(L.orc_blocked_setup(self.ne, self.P, _p(idx), C.c_longlong(int(lsize))))

    def apply_add(self, x, y):
        lib().orc_apply_add_blocked(self.pool, self.setup, self.kind, self.ne, self.P, self.Q, _p(self.interp), _p(self.deriv),
                                    _p(self.idx), _p(self.orient), _p(self.qdata), _p(self.ctx), _p(x), _p(y))
        return y

    def close(self):
        if self.pool:
            lib().orc_blocked_destroy(self.setup)
            lib().orc_pool_destroy(self.pool)
            self.pool = self.setup = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
