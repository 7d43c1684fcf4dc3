"""CPU checks of the boundary-integrator path (quadrilateral Nedelec faces embedded in 3-D; Palace's dim = 2,
space_dim = 3 QFunctions, /root/reference/palace/fem/qfunctions/32/{geom,hcurl}_32_qf.h): the embedding of the 3 x 2
geometry factor and the 2-component field into the 3-D ND mass path is pinned against golden vectors produced by the
reference's own headers (tests/golden/qf32_golden.npz, generator tests/golden/make_golden.py 32), and the assembled
boundary mass against exact surface integrals."""
import os

import numpy as np
import pytest

from oracle import pyoracle as O
from palace_b200.host import bdrspace as bs
from palace_b200.host import coeff as cf
from palace_b200.host import hexmesh as hm
from palace_b200.host import hexspace as hs
from tests import common

G = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "qf32_golden.npz"))


def _rel(a, b):
    return np.abs(a - b).max() / np.abs(b).max()


def test_geom32_restatement_matches_reference_golden():
    assert _rel(bs.geom32_qdata(G["attr"], G["qw"], G["J"]), G["qdata"]) < 1e-13


def test_padded_3d_mass_map_is_the_reference_hcurl_32():
    """v = w|J| A^T C A u with A = adj(J)^T/|J| (3 x 2): the 3-D pointwise map on [A | 0] and (u, 0) returns (v, 0)."""
    qd11 = bs.pad32_to_33(G["qdata"])
    u3 = np.concatenate([G["u"], np.zeros((1, G["u"].shape[1]))], axis=0)
    v, _ = O.apply_D(O.ND_MASS, np.ascontiguousarray(G["ctx"]), np.ascontiguousarray(qd11), np.ascontiguousarray(u3), None)
    assert _rel(v[:2], G["v"]) < 2e-15 * 10 and np.abs(v[2]).max() == 0.0


G31 = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "qf31_golden.npz"))


def test_line_elements_in_3d_are_the_padded_3d_map_too():
    """qfunctions/31 (1-D elements in 3-D space: the boundary edges of the wave ports' 2-D submeshes, integ/vecfemass.cpp case 31):
    the restated geometry factor against the reference's golden q-data, and f_apply_hcurl_31 = the 3-D H(curl) mass map on
    [A | 0 | 0] and (u, 0, 0) (tests/golden/qf31_golden.npz, generator tests/golden/make_golden.py 31). On a straight edge with a
    constant field the quadratic form is the line integral of (E . t)^2 t^T C t."""
    assert _rel(bs.geom31_qdata(G31["attr"], G31["qw"], G31["J"]), G31["qdata"]) < 1e-13
    Q = G31["u"].shape[1]
    u3 = np.concatenate([G31["u"], np.zeros((2, Q))], axis=0)
    v, _ = O.apply_D(O.ND_MASS, np.ascontiguousarray(G31["ctx"]), np.ascontiguousarray(bs.pad31_to_33(G31["qdata"])),
                     np.ascontiguousarray(u3), None)
    assert _rel(v[:1], G31["v"]) < 2e-14 and np.abs(v[1:]).max() == 0.0
    a, b = np.array([0.2, -0.1, 0.4]), np.array([1.1, 0.7, -0.3])
    Cm = np.array([[2.0, 0.3, 0.1], [0.3, 1.5, -0.2], [0.1, -0.2, 1.0]])
    Ev = np.array([0.5, -1.2, 0.8])
    x, w = np.polynomial.legendre.leggauss(3)
    t = np.repeat((b - a)[:, None], 3, axis=1)
    qd = bs.pad31_to_33(bs.geom31_qdata(np.ones(3), 0.5 * w, t))
    ut = np.zeros((3, 3))
    ut[0] = Ev @ (b - a)                                        # covariant component of the constant field
    ctx = cf.coeff_ctx(np.zeros(1, dtype=int), Cm[None], a=1.0)
    v, _ = O.apply_D(O.ND_MASS, ctx, np.ascontiguousarray(qd), ut, None)
    th = (b - a) / np.linalg.norm(b - a)
    assert abs((ut * v).sum() - np.linalg.norm(b - a) * (Ev @ th) ** 2 * (th @ Cm @ th)) < 1e-13


def test_against_compiled_reference_32_headers():
    """The compiled reference's f_build_geom_factor_32 on seeded inputs, as stored by tests/golden/make_golden.py direct."""
    D = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "qf_direct_golden.npz"))
    J, attr, qw, qd = D["geom32_J"], D["geom32_attr"], D["geom32_qw"], D["geom32_qdata"]
    Q = J.shape[1]
    assert _rel(bs.geom32_qdata(attr, qw, J), qd) < 1e-13
    # |J| is the area element and A the pseudo-inverse transposed: A^T Jm = I
    for i in range(Q):
        Jm = J[:, i].reshape(3, 2, order="F")
        A = qd[2:, i].reshape(3, 2, order="F")
        assert np.abs(A.T @ Jm - np.eye(2)).max() < 1e-12
        assert abs(qd[1, i] / qw[i] - np.linalg.norm(np.cross(Jm[:, 0], Jm[:, 1]))) < 1e-12


@pytest.mark.parametrize("p", [1, 2, 3])
def test_boundary_mass_energy_of_a_constant_field(p):
    """x = G phi with phi the nodal interpolant of a . x  (so E = a exactly) on a box mesh with scrambled element frames:
    x^T M_bdr x = sum over boundary faces of area * |a - (a . n) n|^2."""
    size = (1.0, 0.7, 0.9)
    mesh = hm.box_mesh((3, 2, 2), size, warp_amp=0.0, scramble_seed=3, n_attr=1)
    topo = hs.build_topology(mesh)
    nd, h1 = hs.build_nd_space(mesh, topo, p), hs.build_h1_space(mesh, topo, p)
    a = np.array([0.7, -1.1, 0.4])
    nodes = hs.gauss_lobatto(p + 1)
    xh = mesh.node_coords(p, nodes)                             # [ne][3][(p+1)^3] lexicographic
    phi = np.zeros(h1.ndofs)
    phi[h1.lex_gid] = np.einsum("c,ecn->en", a, xh)
    Gm = common.oracle_interp(h1, nd, hs.discrete_gradient_matrix(p))
    x = Gm @ phi
    faces = bs.boundary_faces(topo)
    assert faces.shape[0] == 2 * (3 * 2 + 3 * 2 + 2 * 2)
    sp = bs.build_nd_bdr_space(nd, faces)
    interp, qw2 = bs.nd_quad_tables(p)
    q1d = p + 1
    xe = mesh.node_coords(1, hs.gauss_lobatto(2))
    qd = bs.pad32_to_33(bs.bdr_qdata(xe, faces, 1, q1d))
    assert np.isclose(qd[:, 1, :].sum(), 2 * (size[0] * size[1] + size[0] * size[2] + size[1] * size[2]), rtol=1e-13)
    y = O.apply_add(O.ND_MASS, interp, None, sp.idx, sp.orient, qd, cf.coeff_ctx(a=1.0), x, np.zeros(nd.ndofs))
    want = 0.0
    for n_ax, area in ((0, size[1] * size[2]), (1, size[0] * size[2]), (2, size[0] * size[1])):
        want += 2 * area * (a @ a - a[n_ax] ** 2)
    assert abs(x @ y - want) < 1e-12 * want
    # a boundary mass with a material coefficient is symmetric positive semi-definite and touches boundary dofs only
    z = np.random.default_rng(1).random(nd.ndofs)
    yz = O.apply_add(O.ND_MASS, interp, None, sp.idx, sp.orient, qd, cf.coeff_ctx(a=2.0), z, np.zeros(nd.ndofs))
    interior = np.setdiff1d(np.arange(nd.ndofs), nd.ess_dofs)
    assert np.abs(yz[interior]).max() == 0.0 and z @ yz > 0


# ---- boundary curl-curl (scalar curl of the face element; integ/curlcurl.cpp case 32 -> f_apply_l2_1) ----
GC = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "qf32_curl_golden.npz"))


def test_padded_3d_curlcurl_map_is_the_reference_l2_1():
    """w = w' Jd^T C Jd c with the identity geometry factor, w' = qw^2 / (w |J|), C = coeff I and c = (curl, 0, 0)."""
    qd11 = bs.curl32_qdata(G["qdata"], G["qw"])
    c3 = np.zeros((3, GC["u"].size))
    c3[0] = GC["u"]
    ctx3 = cf.widen_scalar_ctx(GC["ctx1"])
    _, w = O.apply_D(O.CURLCURL, np.ascontiguousarray(ctx3), np.ascontiguousarray(qd11), None, np.ascontiguousarray(c3))
    assert _rel(w[0], GC["v"]) < 1e-14 and np.abs(w[1:]).max() == 0.0


@pytest.mark.parametrize("p", [2, 3])
def test_boundary_curlcurl_energy_of_a_rigid_rotation(p):
    """E = omega x r (in ND_p for p >= 2, curl E = 2 omega): x^T K_bdr x = sum over boundary faces of area (2 omega . n)^2."""
    size = (1.0, 0.7, 0.9)
    mesh = hm.box_mesh((3, 2, 2), size, warp_amp=0.0, scramble_seed=4, n_attr=1)
    topo = hs.build_topology(mesh)
    nd = hs.build_nd_space(mesh, topo, p)
    om = np.array([0.3, -0.8, 0.5])
    # ND dofs of E: tangential reference component at the dof's node (interpolatory tensor basis): u^_c = (J^T E)_c
    op_, _ = hs.gauss_legendre(p)
    cp_ = hs.gauss_lobatto(p + 1)
    x = np.zeros(nd.ndofs)
    for e in range(mesh.ne):
        v = mesh.verts[mesh.elems[e]]
        J = np.stack([v[1] - v[0], v[2] - v[0], v[4] - v[0]], axis=1)
        for l, (c, i, j, k) in enumerate(hs._nd_lex_layout(p)):
            ix = (i, j, k)
            xi = np.array([op_[ix[d]] if d == c else cp_[ix[d]] for d in range(3)])
            E = np.cross(om, v[0] + J @ xi)
            x[nd.lex_gid[e, l]] = nd.lex_sign[e, l] * (J[:, c] @ E)
    faces = bs.boundary_faces(topo)
    sp = bs.build_nd_bdr_space(nd, faces)
    deriv = bs.nd_quad_curl_tables(p)
    _, qw2 = bs.nd_quad_tables(p)
    xe = mesh.node_coords(1, hs.gauss_lobatto(2))
    qd = bs.curl32_qdata(bs.bdr_qdata(xe, faces, 1, p + 1), qw2)
    ctx3 = cf.widen_scalar_ctx(cf.coeff_ctx(np.array([0]), np.array([1.0]), a=1.0, dim=1))
    y = O.apply_add(O.CURLCURL, None, deriv, sp.idx, sp.orient, qd, ctx3, x, np.zeros(nd.ndofs))
    want = sum(2 * area * (2 * om[n_ax]) ** 2 for n_ax, area in ((0, size[1] * size[2]), (1, size[0] * size[2]), (2, size[0] * size[1])))
    assert abs(x @ y - want) < 1e-11 * want
