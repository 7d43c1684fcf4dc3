"""CPU: pins the oracle's restated pointwise arithmetic (geometry factors, D for hcurl / hdiv /
hdivmass) to golden vectors produced by the REFERENCE's own QFunction headers
(tests/golden/make_golden.py; the reference's palace/fem/qfunctions/33/*.h), including the compiled reference's output on
the seeded inputs of test_against_compiled_reference_headers."""
import os

import numpy as np
import pytest

from oracle import pyoracle as O

G = np.load(os.path.join(os.path.dirname(__file__), "golden", "qf_golden.npz"))
TOL = 2e-15


def _rel(a, b):
    return np.abs(a - b).max() / np.abs(b).max()


def test_geom_factor_matches_reference_golden():
    # oracle geometry from J: restated in orc_geom_hex_qdata; here re-derive q-data from the golden J
    J, qw, attr = G["J"], G["qw"], G["attr"]
    Q = J.shape[1]
    qd = np.empty((11, Q))
    for i in range(Q):
        M = J[:, i].reshape(3, 3, order="F")
        det = np.linalg.det(M)
        qd[0, i] = attr[i]
        qd[1, i] = qw[i] * det
        qd[2:, i] = np.linalg.inv(M).T.ravel(order="F")  # adj(J)^T/detJ = J^-T
    assert _rel(qd, G["qdata"]) < 1e-13


@pytest.mark.parametrize("case", ["hcurl", "hcurl_identity", "hdiv", "hdivmass"])
def test_pointwise_D_matches_reference_golden(case):
    qdata, u, c = np.ascontiguousarray(G["qdata"]), np.ascontiguousarray(G["u"]), np.ascontiguousarray(G["c"])
    if case == "hcurl":
        v, _ = O.apply_D(O.ND_MASS, np.ascontiguousarray(G["ctx_mass"]), qdata, u, None)
        assert _rel(v, G["hcurl_v"]) < TOL
    elif case == "hcurl_identity":
        v, _ = O.apply_D(O.ND_MASS, np.ascontiguousarray(G["ctx_id"]), qdata, u, None)
        assert _rel(v, G["hcurl_v_identity"]) < TOL
        # H1 diffusion uses the same QFunction on the gradient (integ/diffusion.cpp:37-42)
        _, w = O.apply_D(O.H1_DIFFUSION, np.ascontiguousarray(G["ctx_id"]), qdata, None, u)
        assert _rel(w, G["hcurl_v_identity"]) < TOL
    elif case == "hdiv":
        _, w = O.apply_D(O.CURLCURL, np.ascontiguousarray(G["ctx_curl"]), qdata, None, c)
        assert _rel(w, G["hdiv_w"]) < TOL
    else:
        v, w = O.apply_D(O.CURLCURL_MASS, np.ascontiguousarray(G["ctx_pair"]), qdata, u, c)
        assert _rel(v, G["hdivmass_v"]) < TOL and _rel(w, G["hdivmass_w"]) < TOL


def test_build_qfunctions_are_consistent_with_apply():
    """The reference's assembled-q-data QFunctions (f_build_*_33 + f_apply_33) give the same v as
    the on-the-fly ones: checks the golden build outputs against the golden apply outputs."""
    u, c = G["u"], G["c"]
    qd = G["build_hdivmass"]
    v = np.einsum("rcq,cq->rq", qd[:9].reshape(3, 3, -1, order="F"), u)
    w = np.einsum("rcq,cq->rq", qd[9:].reshape(3, 3, -1, order="F"), c)
    assert _rel(v, G["hdivmass_v"]) < 1e-14 and _rel(w, G["hdivmass_w"]) < 1e-14
    assert _rel(np.einsum("rcq,cq->rq", G["build_hcurl"].reshape(3, 3, -1, order="F"), u), G["hcurl_v"]) < 1e-14
    assert _rel(np.einsum("rcq,cq->rq", G["build_hdiv"].reshape(3, 3, -1, order="F"), c), G["hdiv_w"]) < 1e-14


def test_against_compiled_reference_headers():
    """The compiled reference's f_apply_hdivmass_33 on seeded inputs, as stored by tests/golden/make_golden.py direct."""
    D = np.load(os.path.join(os.path.dirname(__file__), "golden", "qf_direct_golden.npz"))
    u, c, v, w = D["hdivmass_u"], D["hdivmass_c"], D["hdivmass_v"], D["hdivmass_w"]
    qdata = np.ascontiguousarray(G["qdata"][:, :u.shape[1]])
    ctx = np.ascontiguousarray(G["ctx_pair"])
    vo, wo = O.apply_D(O.CURLCURL_MASS, ctx, qdata, np.ascontiguousarray(u), np.ascontiguousarray(c))
    assert _rel(vo, v) < TOL and _rel(wo, w) < TOL


# ---- mixed H(curl) / H(div) QFunctions: MixedVectorWeakCurl / MixedVectorCurl integrators (integ/mixedveccurl.cpp), the mixed mass
# of the FluxProjector and the element error integrands of the flux estimators (linalg/errorestimator.cpp) ----
GM = np.load(os.path.join(os.path.dirname(__file__), "golden", "qf_mixed_golden.npz"))


def _decode_ctx(ctx):
    """attr (1-based) -> 3x3 matrix of a single coefficient context (qfunctions/coeff/coeff_qf.h:7-43); returns (lookup, entries)."""
    ints = np.ascontiguousarray(ctx).view(np.int32)[::2]
    n_attr = int(ints[0])
    n_mat = int(ints[1 + n_attr])
    base = 2 + n_attr
    mats = [np.asarray(ctx[base + 9 * k: base + 9 * (k + 1)]).reshape(3, 3, order="F") for k in range(n_mat)]

    def lookup(attr):
        return mats[int(ints[1 + (int(attr) - 1)]) if n_attr > 0 else 0]

    return lookup, base + 9 * n_mat


def test_mixed_curl_pointwise_D_matches_reference_golden():
    qdata = np.ascontiguousarray(G["qdata"])
    u1, u2 = np.ascontiguousarray(GM["u1"]), np.ascontiguousarray(GM["u2"])
    _, w = O.apply_D(O.ND_WEAKCURL, np.ascontiguousarray(GM["ctx_weak"]), qdata, u1, None)
    assert _rel(w, GM["hcurlhdiv_v"]) < TOL
    v, _ = O.apply_D(O.ND_MIXEDCURL, np.ascontiguousarray(GM["ctx_curl"]), qdata, None, u2)
    assert _rel(v, GM["hdivhcurl_v"]) < TOL


def test_estimator_oracle_matches_reference_golden():
    """oracle/estimator.py (mixed mass matrix, element error integrals) on one-point 'elements' with identity tables: the block
    of point q is the reference's pointwise D / integrand at q."""
    from oracle import estimator as E

    qdata = np.ascontiguousarray(G["qdata"])
    Q = qdata.shape[1]
    qd1 = np.ascontiguousarray(qdata.T.reshape(Q, 11, 1))            # ne = Q elements of one point each
    eye = np.eye(3).reshape(3, 1, 3)                                  # interp[3][1][3]: dof j = component j
    idx = np.arange(3 * Q).reshape(Q, 3)
    one = np.ones((Q, 3))
    u1, u2 = GM["u1"], GM["u2"]
    # f_apply_hdivhcurl_33: H(div) trial, H(curl) test
    look, _ = _decode_ctx(GM["ctx_curl"])
    coef = [look(a) for a in qdata[0]]
    M = E.mixed_mass_matrix(qd1, eye, E.HDIV, idx, one, 3 * Q, eye, E.HCURL, idx, one, 3 * Q, coef)
    assert _rel((M @ u2.T.ravel()).reshape(Q, 3).T, GM["hdivhcurl_v"]) < 1e-14
    # f_apply_hcurlhdiv_33: H(curl) trial, H(div) test
    look, _ = _decode_ctx(GM["ctx_weak"])
    coef = [look(a) for a in qdata[0]]
    M = E.mixed_mass_matrix(qd1, eye, E.HCURL, idx, one, 3 * Q, eye, E.HDIV, idx, one, 3 * Q, coef)
    assert _rel((M @ u1.T.ravel()).reshape(Q, 3).T, GM["hcurlhdiv_v"]) < 1e-14
    # error integrands with the pair context: first part scales field 1, second part field 2
    look1, n1 = _decode_ctx(GM["ctx_err"])
    look2, _ = _decode_ctx(GM["ctx_err"][n1:])
    c1 = [look1(a) for a in qdata[0]]
    c2 = [look2(a) for a in qdata[0]]
    x1, x2 = u1.T.ravel(), u2.T.ravel()
    e = E.element_errors(qd1, eye, E.HCURL, idx, one, x1, c1, eye, E.HDIV, idx, one, x2, c2)
    assert _rel(e, GM["hcurlhdiv_error"]) < 1e-13
    e = E.element_errors(qd1, eye, E.HDIV, idx, one, x1, c1, eye, E.HCURL, idx, one, x2, c2)
    assert _rel(e, GM["hdivhcurl_error"]) < 1e-13
