"""Generates tests/golden/qf_golden.npz by running the REFERENCE's own QFunction headers
(compiled in place from /root/reference by oracle/Makefile into oracle/_ref) on seeded inputs.
Run in the build container only (needs /root/reference):  python tests/golden/make_golden.py
The fixture pins the oracle's restated pointwise arithmetic (tests/test_oracle_golden.py) on boxes
where /root/reference does not exist."""
import ctypes as C
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle import pyoracle as O  # noqa: E402
from palace_b200.host import coeff as cf  # noqa: E402


def main():
    ref = O.ref()
    assert ref is not None, "oracle/_ref not built (needs /root/reference)"
    rng = np.random.default_rng(20260923)
    Q = 96
    p = lambda a: a.ctypes.data_as(C.c_void_p)
    # Jacobians: random well-conditioned, column-major components [9][Q]
    J = np.empty((9, Q))
    for i in range(Q):
        M = np.eye(3) * (0.5 + rng.random()) + 0.3 * (rng.random((3, 3)) - 0.5)
        J[:, i] = M.ravel(order="F")
    n_attr = 5
    attr = (1 + rng.integers(0, n_attr, size=Q)).astype(np.float64)
    qw = 0.1 + rng.random(Q)
    qdata = np.empty((11, Q))
    assert ref.ref_build_geom_factor_33(Q, p(attr), p(qw), p(J), p(qdata)) == 0
    am, mc = cf.test_suite_coefficient(n_attr, "matrix")
    mc = mc + 0.05 * rng.random(mc.shape)  # non-symmetric on purpose
    am2 = am.copy()
    am2[1] = -1  # an unassigned attribute -> zero material (coefficient.cpp:78-88)
    ctx_mass = cf.coeff_ctx(am, mc, a=1.3)
    ctx_curl = cf.coeff_ctx(am2, mc[::-1].copy(), a=0.7, transpose=True)
    ctx_pair = cf.coeff_ctx_pair(ctx_mass, ctx_curl)
    ctx_id = cf.coeff_ctx(a=2.5)
    u = rng.random((3, Q)) - 0.5
    c = rng.random((3, Q)) - 0.5
    out = dict(J=J, attr=attr, qw=qw, qdata=qdata, ctx_mass=ctx_mass, ctx_curl=ctx_curl, ctx_pair=ctx_pair, ctx_id=ctx_id, u=u, c=c)
    v = np.empty((3, Q)); w = np.empty((3, Q))
    assert ref.ref_apply_hcurl_33(p(ctx_mass), Q, p(qdata), p(u), p(v)) == 0
    out["hcurl_v"] = v.copy()
    assert ref.ref_apply_hcurl_33(p(ctx_id), Q, p(qdata), p(u), p(v)) == 0
    out["hcurl_v_identity"] = v.copy()
    assert ref.ref_apply_hdiv_33(p(ctx_curl), Q, p(qdata), p(c), p(w)) == 0
    out["hdiv_w"] = w.copy()
    assert ref.ref_apply_hdivmass_33(p(ctx_pair), Q, p(qdata), p(u), p(c), p(v), p(w)) == 0
    out["hdivmass_v"], out["hdivmass_w"] = v.copy(), w.copy()
    qd1 = np.empty((9, Q)); qd2 = np.empty((18, Q))
    assert ref.ref_build_hcurl_33(p(ctx_mass), Q, p(qdata), p(qd1)) == 0
    out["build_hcurl"] = qd1.copy()
    assert ref.ref_build_hdiv_33(p(ctx_curl), Q, p(qdata), p(qd1)) == 0
    out["build_hdiv"] = qd1.copy()
    assert ref.ref_build_hdivmass_33(p(ctx_pair), Q, p(qdata), p(qd2)) == 0
    out["build_hdivmass"] = qd2.copy()
    path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "qf_golden.npz")
    np.savez_compressed(path, **out)
    print("wrote", path, os.path.getsize(path), "bytes")



def main32():
    """tests/golden/qf32_golden.npz: the reference's boundary (dim 2 in space_dim 3) geometry-factor and H(curl) mass
    QFunctions (qfunctions/32/geom_32_qf.h, hcurl_32_qf.h) on seeded inputs."""
    ref = O.ref()
    assert ref is not None, "oracle/_ref not built (needs /root/reference)"
    rng = np.random.default_rng(20260924)
    Q = 64
    p = lambda a: a.ctypes.data_as(C.c_void_p)
    J = np.ascontiguousarray(rng.random((6, Q)) - 0.5) + np.array([1.0, 0, 0, 0, 1.0, 0])[:, None]
    n_attr = 4
    attr = (1 + rng.integers(0, n_attr, size=Q)).astype(np.float64)
    qw = 0.1 + rng.random(Q)
    qd = np.empty((8, Q))
    assert ref.ref_build_geom_factor_32(Q, p(attr), p(qw), p(J), p(qd)) == 0
    am, mc = cf.test_suite_coefficient(n_attr, "matrix")
    mc = mc + 0.05 * rng.random(mc.shape)
    ctx = cf.coeff_ctx(am, mc, a=1.3)
    u = np.ascontiguousarray(rng.random((2, Q)) - 0.5)
    v = np.empty((2, Q))
    assert ref.ref_apply_hcurl_32(p(ctx), Q, p(qd), p(u), p(v)) == 0
    path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "qf32_golden.npz")
    np.savez_compressed(path, J=J, attr=attr, qw=qw, qdata=qd, ctx=ctx, u=u, v=v)
    print("wrote", path, os.path.getsize(path), "bytes")


def main31():
    """tests/golden/qf31_golden.npz: the reference's line-element (dim 1 in space_dim 3) geometry-factor and H(curl) mass QFunctions
    (qfunctions/31/geom_31_qf.h, hcurl_31_qf.h) on seeded inputs."""
    ref = O.ref()
    assert ref is not None, "oracle/_ref not built (needs /root/reference)"
    rng = np.random.default_rng(20260927)
    Q = 48
    p = lambda a: a.ctypes.data_as(C.c_void_p)
    J = np.ascontiguousarray(rng.random((3, Q)) - 0.5) + np.array([0.9, 0.0, 0.0])[:, None]
    n_attr = 4
    attr = (1 + rng.integers(0, n_attr, size=Q)).astype(np.float64)
    qw = 0.1 + rng.random(Q)
    qd = np.empty((5, Q))
    assert ref.ref_build_geom_factor_31(Q, p(attr), p(qw), p(J), p(qd)) == 0
    am, mc = cf.test_suite_coefficient(n_attr, "matrix")
    mc = mc + 0.05 * rng.random(mc.shape)
    ctx = cf.coeff_ctx(am, mc, a=0.7)
    u = np.ascontiguousarray(rng.random((1, Q)) - 0.5)
    v = np.empty((1, Q))
    assert ref.ref_apply_hcurl_31(p(ctx), Q, p(qd), p(u), p(v)) == 0
    path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "qf31_golden.npz")
    np.savez_compressed(path, J=J, attr=attr, qw=qw, qdata=qd, ctx=ctx, u=u, v=v)
    print("wrote", path, os.path.getsize(path), "bytes")


def main_mixed():
    """tests/golden/qf_mixed_golden.npz: the reference's mixed H(curl) / H(div) QFunctions (qfunctions/33/hcurlhdiv_33_qf.h:
    MixedVectorWeakCurl / MixedVectorCurl integrators and the FluxProjector's mixed mass) and the element error integrands of
    the flux error estimators (hcurlhdiv_error_33_qf.h, pair context) on the seeded q-data of qf_golden.npz."""
    ref = O.ref()
    assert ref is not None, "oracle/_ref not built (needs /root/reference)"
    G = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "qf_golden.npz"))
    rng = np.random.default_rng(20260925)
    qdata = np.ascontiguousarray(G["qdata"])
    Q = qdata.shape[1]
    p = lambda a: a.ctypes.data_as(C.c_void_p)
    n_attr = 5
    am, mc = cf.test_suite_coefficient(n_attr, "matrix")
    mc = mc + 0.05 * rng.random(mc.shape)  # non-symmetric: the two QFunctions place the coefficient differently
    ctx_weak = cf.coeff_ctx(am, mc, a=-1.0)                                # MixedVectorWeakCurlIntegrator scales by -1
    ctx_curl = cf.coeff_ctx(am, mc, a=1.0, transpose=True)                 # MixedVectorCurlIntegrator(Q, transpose = true)
    ctx_err = cf.coeff_ctx_pair(cf.coeff_ctx(am, mc, a=1.0), cf.coeff_ctx(am, mc[::-1].copy(), a=0.8))
    u1 = np.ascontiguousarray(rng.random((3, Q)) - 0.5)
    u2 = np.ascontiguousarray(rng.random((3, Q)) - 0.5)
    v = np.empty((3, Q)); s = np.empty(Q)
    out = dict(ctx_weak=ctx_weak, ctx_curl=ctx_curl, ctx_err=ctx_err, u1=u1, u2=u2)
    assert ref.ref_apply_hcurlhdiv_33(p(ctx_weak), Q, p(qdata), p(u1), p(v)) == 0
    out["hcurlhdiv_v"] = v.copy()
    assert ref.ref_apply_hdivhcurl_33(p(ctx_curl), Q, p(qdata), p(u2), p(v)) == 0
    out["hdivhcurl_v"] = v.copy()
    assert ref.ref_apply_hcurlhdiv_error_33(p(ctx_err), Q, p(qdata), p(u1), p(u2), p(s)) == 0
    out["hcurlhdiv_error"] = s.copy()
    assert ref.ref_apply_hdivhcurl_error_33(p(ctx_err), Q, p(qdata), p(u1), p(u2), p(s)) == 0
    out["hdivhcurl_error"] = s.copy()
    path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "qf_mixed_golden.npz")
    np.savez_compressed(path, **out)
    print("wrote", path, os.path.getsize(path), "bytes")


def main32curl():
    """tests/golden/qf32_curl_golden.npz: the reference's boundary curl-curl QFunction (scalar curl of a 2-D element in 3-D:
    integ/curlcurl.cpp case 32 -> f_apply_l2_1, qfunctions/1/l2_1_qf.h, coefficient context of dimension 1) on the q-data of
    qf32_golden.npz."""
    ref = O.ref()
    assert ref is not None, "oracle/_ref not built (needs /root/reference)"
    G = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "qf32_golden.npz"))
    rng = np.random.default_rng(20260926)
    qd, qw = np.ascontiguousarray(G["qdata"]), np.ascontiguousarray(G["qw"])
    Q = qd.shape[1]
    p = lambda a: a.ctypes.data_as(C.c_void_p)
    n_attr = 4
    am = np.arange(n_attr) % 3
    ctx1 = cf.coeff_ctx(am, np.array([1.5, 0.25, 7.0]), a=0.9, dim=1)
    u = np.ascontiguousarray(rng.random(Q) - 0.5)
    v = np.empty(Q)
    assert ref.ref_apply_l2_1(p(ctx1), Q, p(qd), p(qw), p(u), p(v)) == 0
    path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "qf32_curl_golden.npz")
    np.savez_compressed(path, ctx1=ctx1, u=u, v=v)
    print("wrote", path, os.path.getsize(path), "bytes")


def main_direct():
    """tests/golden/qf_direct_golden.npz: the reference's f_apply_hdivmass_33 and f_build_geom_factor_32 on the seeded inputs of
    test_oracle_golden.test_against_compiled_reference_headers and test_bdr_cpu.test_against_compiled_reference_32_headers, so
    that both compare the oracle with the reference's own output where oracle/_ref cannot be built."""
    ref = O.ref()
    assert ref is not None, "oracle/_ref not built (needs the reference checkout)"
    G = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "qf_golden.npz"))
    p = lambda a: a.ctypes.data_as(C.c_void_p)
    Q = 40
    rng = np.random.default_rng(7)
    qdata = np.ascontiguousarray(G["qdata"][:, :Q])
    u, c = rng.random((3, Q)), rng.random((3, Q))
    v, w = np.empty((3, Q)), np.empty((3, Q))
    assert ref.ref_apply_hdivmass_33(p(np.ascontiguousarray(G["ctx_pair"])), Q, p(qdata), p(u), p(c), p(v), p(w)) == 0
    rng = np.random.default_rng(3)
    J = np.ascontiguousarray(rng.random((6, Q)) - 0.5) + np.array([0.8, 0, 0, 0, 1.2, 0])[:, None]
    attr, qw = np.ones(Q), 0.2 + rng.random(Q)
    qd = np.empty((8, Q))
    assert ref.ref_build_geom_factor_32(Q, p(attr), p(qw), p(J), p(qd)) == 0
    path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "qf_direct_golden.npz")
    np.savez_compressed(path, hdivmass_u=u, hdivmass_c=c, hdivmass_v=v, hdivmass_w=w, geom32_J=J, geom32_attr=attr, geom32_qw=qw,
                        geom32_qdata=qd)
    print("wrote", path, os.path.getsize(path), "bytes")


if __name__ == "__main__":
    if len(sys.argv) > 1 and sys.argv[1] == "direct":
        main_direct()
    elif len(sys.argv) > 1 and sys.argv[1] == "32":
        main32()
    elif len(sys.argv) > 1 and sys.argv[1] == "31":
        main31()
    elif len(sys.argv) > 1 and sys.argv[1] == "32curl":
        main32curl()
    elif len(sys.argv) > 1 and sys.argv[1] == "mixed":
        main_mixed()
    else:
        main()
