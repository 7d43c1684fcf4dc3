"""END-TO-END pin of the TETRAHEDRAL geometry / space path against numbers produced by the reference itself: the
capacitance matrix of the two-spheres electrostatics example (the reference's examples/spheres/spheres.json: 14,362
curved cubic tetrahedra TET20, H1 order 3, 66,328 dofs) that Palace's regression suite stores in
test/data/regression/ref/spheres/terminal-C.csv. The oracle-side path -- the example mesh as palace_b200/host/gmsh.py reads it, order-3
tet geometry q-data and the H1 tet space of palace_b200/host/tetspace.py, the reference QFunction arithmetic of the oracle,
a Jacobi-preconditioned CG solve to 1e-13 -- reproduces all four entries to 1.4e-10 relative when the forms are integrated with the rule
the reference uses (q_order = 2 p = 6 -> the 24-point symmetric rule, tetspace.tet_quadrature_symmetric6); with the 64-point conical
rule of the same degree the entries sit 4e-8 ... 7e-8 away: on curved elements the integrand is not a polynomial, and the choice of
rule is what round 1's looser pin was seeing. The remaining 1.3e-10 is uniform over the four entries (the physical constants' digits). The example's
mesh (3.4 MB as a .msh file) is stored compactly in tests/golden/spheres_mesh.npz (generator and loader:
tests/golden/make_spheres_fixture.py): corners, connectivity and the curved lattice nodes; the straight ones are rebuilt.

The same run's error-indicators.csv pins the GRAD-FLUX estimator on these curved tetrahedra (GradFluxErrorEstimator,
palace/linalg/errorestimator.cpp:272-398 and drivers/electrostaticsolver.cpp:77-86): E = -grad V in ND_3 by the element-local
discrete gradient, D = eps E projected onto RT_2 (mass CG to 1e-12), eta_K^2 = int_K |D - E|^2 scaled by 0.5 / E_elec per terminal,
e_K = sqrt(mean over the two terminals). Global norm 2.9e-8 and mean 4.8e-8 relative to the stored values, minimum 6.1e-5 and maximum 1.2e-5
(single elements; the reference's projection stops at 1e-6)."""
import numpy as np
import pytest
import scipy.sparse as sp
import scipy.sparse.linalg as spla

from oracle import estimator as E

from oracle import pyoracle as O
from palace_b200.host import coeff as cf
from palace_b200.host import tetspace as ts
from tests.golden import make_spheres_fixture

RULE = ts.tet_quadrature_symmetric6
# test/data/regression/ref/spheres/terminal-C.csv (farads)
# test/data/regression/ref/spheres/error-indicators.csv: Norm, Minimum, Maximum, Mean
IND_REF = (6.910139872411e-03, 1.217546964778e-06, 5.028157468369e-04, 3.383123588483e-05)
C_REF = np.array([[+1.237445610357e-12, -4.770975738888e-13], [-4.770975738888e-13, +2.478413459856e-12]])


@pytest.fixture(scope="module")
def spheres():
    m = make_spheres_fixture.load_fixture()
    assert m.order == 3 and m.ne == 14362
    p = 3                                                            # spheres.json "Order": 3
    mesh = ts.TetMesh(m.verts, m.elems, m.attr)
    nd = ts.build_nd_tet_space(mesh, p)                              # edge / face numbering; E = -grad V lives here
    h1 = ts.build_h1_tet_space(mesh, nd, p)
    assert h1.ndofs == 66328                                         # = the node count of the order-3 mesh file
    qpts, qw = RULE() if RULE else ts.tet_quadrature(2 * p)
    qd = ts.geom_qdata(m.xe, np.ones(m.ne, dtype=np.int32), m.order, qpts, qw)
    assert (qd[:, 1, :] > 0).all()
    _, grad = ts.h1_tet_element(p).tabulate(qpts)
    Ae = O.element_matrices(O.H1_DIFFUSION, None, np.ascontiguousarray(grad), None, qd, cf.coeff_ctx(a=1.0), h1.P)
    I = np.repeat(h1.idx, h1.P, axis=1).ravel()
    J = np.tile(h1.idx, (1, h1.P)).ravel()
    K = sp.csr_matrix((Ae.ravel(), (I, J)), shape=(h1.ndofs, h1.ndofs))
    nv, n_e, n_f = m.verts.shape[0], p - 1, (p - 1) * (p - 2) // 2
    edge_base, face_base = nv, nv + n_e * nd.n_edges

    def boundary_dofs(attr):
        s = set()
        for tri in m.bdr_verts[m.bdr_attr == attr]:
            g = sorted(int(x) for x in tri)
            s.update(g)
            for a, b in ((0, 1), (0, 2), (1, 2)):
                eb = edge_base + n_e * nd.edges[(g[a], g[b])]
                s.update(range(eb, eb + n_e))
            fb = face_base + n_f * nd.faces[tuple(g)]
            s.update(range(fb, fb + n_f))
        return np.array(sorted(s))

    D = {a: boundary_dofs(a) for a in (2, 3, 4)}                     # ground (far field), sphere A, sphere B
    free = np.setdiff1d(np.arange(h1.ndofs), np.concatenate(list(D.values())))
    Kff = K[free][:, free].tocsr()
    dinv = 1.0 / Kff.diagonal()
    prec = spla.LinearOperator(Kff.shape, matvec=lambda r: dinv * r, dtype=np.float64)
    V = []
    for a in (3, 4):                                                  # unit potential on one terminal, zero on the rest
        x = np.zeros(h1.ndofs)
        x[D[a]] = 1.0
        sol, info = spla.cg(Kff, -(K[free] @ x), rtol=1e-13, atol=0.0, maxiter=20000, M=prec)
        assert info == 0
        x[free] = sol
        V.append(x)
    return dict(m=m, mesh=mesh, nd=nd, h1=h1, p=p, qpts=qpts, qd=qd, K=K, V=V)


def test_capacitance_matrix_of_the_spheres_example(spheres):
    K, V = spheres["K"], spheres["V"]
    mu0, c0, L0 = 1.25663706127e-6, 299792458.0, 1.0e-2              # palace/utils/constants.hpp:22-30, "L0": 1e-2
    C = np.array([[V[i] @ (K @ V[j]) for j in range(2)] for i in range(2)]) * L0 / (mu0 * c0 * c0)
    rel = np.abs(C - C_REF) / np.abs(C_REF)
    print("capacitance matrix (F):", C, "rel. error vs the reference's terminal-C.csv:", rel)
    assert rel.max() < 1e-9


def test_error_indicators_of_the_spheres_example(spheres):
    """Vectorised over the 14,362 elements (the oracle's per-point loops, oracle/estimator.py, are held to it on a handful of them)."""
    m, mesh, nd, h1, p, qpts, qd, K = (spheres[k] for k in ("m", "mesh", "nd", "h1", "p", "qpts", "qd", "K"))
    ne, Q = m.ne, qd.shape[2]
    rt = ts.build_rt_tet_space(mesh, nd, p - 1)
    A = np.transpose(qd[:, 2:, :].reshape(ne, 3, 3, Q), (0, 3, 2, 1))          # adj(J)^T / det J = J^-T at the points [e][q][row][col]
    Jd = np.transpose(np.linalg.inv(A), (0, 1, 3, 2)) * np.linalg.det(A)[..., None, None]   # J / det J
    w = qd[:, 1, :]
    nd_i = ts.nd_tet_element(p).tabulate(qpts)[0]
    rt_i = ts.rt_tet_element(p - 1).tabulate(qpts)
    Psi = np.einsum("eqcd,dqj->eqcj", Jd, rt_i)                               # physical RT basis
    so = rt.orient.astype(float)
    Me = np.einsum("eqci,eqcj,eq->eij", Psi, Psi, w, optimize=True)
    sub = np.array([0, 1, 777, 5000, ne - 1])                                 # the oracle's loops on a few elements
    ds = np.arange(sub.size * rt.P).reshape(sub.size, rt.P)
    one = np.ones((sub.size, rt.P))
    Mo = E.mixed_mass_matrix(qd[sub], rt_i, E.HDIV, ds, one, ds.size, rt_i, E.HDIV, ds, one, ds.size, [np.eye(3)] * sub.size).toarray()
    for k, e in enumerate(sub):
        assert np.abs(Mo[k * rt.P:(k + 1) * rt.P, k * rt.P:(k + 1) * rt.P] - Me[e]).max() < 1e-12 * np.abs(Me[e]).max()
    Me = so[:, :, None] * Me * so[:, None, :]
    Mrt = sp.csr_matrix((Me.ravel(), (np.repeat(rt.idx, rt.P, axis=1).ravel(), np.tile(rt.idx, (1, rt.P)).ravel())), shape=(rt.ndofs, rt.ndofs))
    md = 1.0 / Mrt.diagonal()
    pm = spla.LinearOperator(Mrt.shape, matvec=lambda r: md * r, dtype=np.float64)
    G = ts.tet_discrete_gradient(p)
    acc = np.zeros(ne)
    for x in spheres["V"]:
        ve = -(x[h1.idx] @ G.T)                                               # E = -grad V, element-frame ND vectors
        Eph = np.einsum("eqcd,dqi,ei->eqc", A, nd_i, ve, optimize=True)
        Et = 0.5 * x @ (K @ x)
        assert abs(0.5 * np.einsum("eqc,eqc,eq->", Eph, Eph, w) / Et - 1) < 1e-12   # the ND field carries the energy of V
        rhs = np.zeros(rt.ndofs)
        np.add.at(rhs, rt.idx.ravel(), (np.einsum("eqci,eqc,eq->ei", Psi, Eph, w, optimize=True) * so).ravel())
        Dv, info = spla.cg(Mrt, rhs, rtol=1e-12, atol=0.0, maxiter=5000, M=pm)
        assert info == 0
        De = so * Dv[rt.idx]
        Dph = np.einsum("eqci,ei->eqc", Psi, De, optimize=True)
        eta2 = np.einsum("eqc,eqc,eq->e", Dph - Eph, Dph - Eph, w)
        dn = np.arange(sub.size * nd.P).reshape(sub.size, nd.P)
        eo = E.element_errors(qd[sub], nd_i, E.HCURL, dn, np.ones((sub.size, nd.P)), ve[sub].ravel(), [np.eye(3)] * sub.size,
                              rt_i, E.HDIV, ds, one, De[sub].ravel(), [np.eye(3)] * sub.size)
        assert np.abs(eo - eta2[sub]).max() < 1e-10 * eta2[sub].max()
        acc += eta2 * 0.5 / Et
    e_ = np.sqrt(acc / 2)
    got = (np.linalg.norm(e_), e_.min(), e_.max(), e_.mean())
    rel = [g / r - 1 for g, r in zip(got, IND_REF)]
    print("error indicators (norm, min, max, mean):", got, "rel. to the reference's error-indicators.csv:", rel)
    assert abs(rel[0]) < 1e-6 and abs(rel[3]) < 1e-6 and abs(rel[1]) < 5e-4 and abs(rel[2]) < 1e-4


def test_probe_field_of_the_spheres_example(spheres):
    """probe-E.csv: E = -grad V at (-1.49, 0, 0) cm, "just above the surface of the smaller sphere", for both terminals. The point is
    located in its curved cubic tetrahedron by Newton's method on the order-3 geometry map, E = -J^-T grad_ref V there; volts per metre
    are sqrt(Z0) / L0 times the value in mesh units (utils/units.hpp:27-34,115-117: E_c = H_c Z0 with H_c^2 Z0 L_c^2 = 1 W, and one
    nondimensional length is L_c). The large component agrees to 8e-8, the vector to 5e-7 of its length."""
    m, h1, p = spheres["m"], spheres["h1"], spheres["p"]
    ref = np.array([[+2.337300901858e+03, +1.334018133064e+01, -1.974701031155e+01],
                    [-1.587529647745e+03, -1.151288542522e+01, +1.802818191385e+01]])
    x0, order = np.array([-1.49, 0.0, 0.0]), m.order
    expo = [(a, b, c) for c in range(order + 1) for b in range(order + 1 - c) for a in range(order + 1 - b - c)]
    vand = lambda X: np.stack([X[:, 0] ** a * X[:, 1] ** b * X[:, 2] ** c for (a, b, c) in expo], axis=1)
    Vinv = np.linalg.inv(vand(ts.tet_lattice(order)))                # nodal basis of the geometry: N(xi) = mono(xi) Vinv
    found = None
    for e in np.argsort(np.linalg.norm(m.xe.mean(axis=2) - x0, axis=1))[:40]:
        xi = np.full(3, 0.25)
        for _ in range(30):
            J = m.xe[e] @ ts._lagrange_tet_grad(order, xi[None])[:, 0, :]
            xi = xi - np.linalg.solve(J, m.xe[e] @ (vand(xi[None]) @ Vinv)[0] - x0)
        if np.linalg.norm(m.xe[e] @ (vand(xi[None]) @ Vinv)[0] - x0) < 1e-12 and xi.min() > -1e-10 and xi.sum() < 1 + 1e-10:
            found = (e, xi)
            break
    assert found is not None
    e, xi = found
    J = m.xe[e] @ ts._lagrange_tet_grad(order, xi[None])[:, 0, :]
    _, grad = ts.h1_tet_element(p).tabulate(xi[None])
    mu0, c0, L0 = 1.25663706127e-6, 299792458.0, 1.0e-2
    for k, x in enumerate(spheres["V"]):
        Ev = -np.linalg.solve(J.T, grad[:, 0, :] @ x[h1.idx[e]]) * np.sqrt(mu0 * c0) / L0
        print("probe E (V/m), terminal", k + 1, Ev, "reference", ref[k])
        assert abs(Ev[0] / ref[k, 0] - 1) < 5e-7 and np.linalg.norm(Ev - ref[k]) < 2e-6 * np.linalg.norm(ref[k])


def test_surface_charges_of_the_spheres_example(spheres):
    """surface-F.csv: the electric flux through each sphere for each terminal's field, Q = int eps E . n dS with n pointing into the
    domain, integrated on the CURVED boundary triangles -- each as a face of its parent cubic tetrahedron: points on the reference
    face, n dS = (J e_s x J e_t) w, E = -J^-T grad_ref V of the parent (the construction of host/tetbdr.py with the cubic geometry
    map). Coulombs are eps0 sqrt(Z0) L0 times the mesh-unit value (utils/units.hpp:115-121). All four entries agree to 4e-7 (they
    are 1.7 % away from C V, which is why the reference prefers the energy formula; the comparison is of the same discrete field)."""
    from palace_b200.host import tetbdr as tb

    m, h1, p = spheres["m"], spheres["h1"], spheres["p"]
    ref = np.array([[+2.361114386696e-11, -9.140234297242e-12], [-9.102953898712e-12, +4.734636562291e-11]])
    pts2, w2 = tb.tri_quadrature(10)
    face_of = {}
    for e in range(m.ne):
        v = m.elems[e][:4]
        for fc in range(4):
            face_of[tuple(sorted(int(v[t]) for t in range(4) if t != fc))] = (e, fc)
    h1el = ts.h1_tet_element(p)
    out = np.zeros((2, 2))
    for s_i, attr in enumerate((3, 4)):
        byf = {fc: [] for fc in range(4)}
        for tri in m.bdr_verts[m.bdr_attr == attr]:
            e, fc = face_of[tuple(sorted(int(x) for x in tri))]
            byf[fc].append(e)
        for fc, els in byf.items():
            if not els:
                continue
            els = np.array(els)
            others = [t for t in range(4) if t != fc]
            es, et = tb.REF_VERTS[others[1]] - tb.REF_VERTS[others[0]], tb.REF_VERTS[others[2]] - tb.REF_VERTS[others[0]]
            rpts = tb.REF_VERTS[others[0]][None] + pts2[:, :1] * es[None] + pts2[:, 1:] * et[None]
            J = np.einsum("ecn,nqd->eqcd", m.xe[els], ts._lagrange_tet_grad(m.order, rpts))
            nv = np.cross(J @ es, J @ et)
            X = m.verts[m.elems[els][:, :4]]
            nv *= -np.sign(np.einsum("eqc,ec->eq", nv, X[:, others].mean(axis=1) - X[:, fc]))[..., None]   # towards the parent: into the domain
            _, grad = h1el.tabulate(rpts)
            for k, x in enumerate(spheres["V"]):
                g = np.einsum("dqi,ei->eqd", grad, x[h1.idx[els]])
                Eph = -np.einsum("eqdc,eqd->eqc", np.linalg.inv(J), g)
                out[k, s_i] += np.einsum("eqc,eqc,q->", Eph, nv, w2)
    mu0, c0, L0 = 1.25663706127e-6, 299792458.0, 1.0e-2
    Qs = out * np.sqrt(mu0 * c0) * L0 / (mu0 * c0 * c0)
    print("surface charges (C):", Qs, "rel. to the reference's surface-F.csv:", Qs / ref - 1)
    assert np.abs(Qs / ref - 1).max() < 2e-6
