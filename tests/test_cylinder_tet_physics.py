"""Physics check of the Nedelec TETRAHEDRON path on an unstructured curved mesh: the cylinder cavity of the reference's
example on its tetrahedral mesh (examples/cylinder/mesh/cylinder_tet.msh, quadratic tets, as stored without the periodic
identification in tests/golden/cylinder_waveguide_tet.npz) with the oracle's
order-3 ND tet discretisation (element tables, curl-oriented restrictions of arbitrarily ordered neighbours, order-2 geometry
q-data) must give the closed-form TM/TE frequencies of docs/src/examples/cylinder.md:36-120 to discretisation accuracy, with
the doubly degenerate modes degenerate to round-off -- which fails for any conformity / orientation error on shared faces.
(The reference stores regression output for the hexahedral mesh only; that one is pinned in tests/test_cylinder_golden.py.)"""
import os

import numpy as np
import scipy.sparse as sp
import scipy.sparse.linalg as spla

from oracle import pyoracle as O
from palace_b200.host import coeff as cf
from palace_b200.host import gmsh
from palace_b200.host import tetspace as ts

FIX = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "cylinder_waveguide_tet.npz"))
# cylinder.md table (GHz): TM010, TE111 (x2), TM011, TE211 (x2), TE112 (x2)
ANALYTIC = np.array([2.903605, 2.922212, 2.922212, 3.468149, 4.146842, 4.146842, 4.396673, 4.396673])


def test_tet_cylinder_cavity_frequencies():
    m = gmsh.HighOrderTetMesh(int(FIX["geom_order"]), FIX["verts"], FIX["elems"], FIX["attr"], FIX["xe"], None, None)
    assert m.order == 2
    p = 3
    mesh = ts.TetMesh(m.verts, m.elems, m.attr)
    nd = ts.build_nd_tet_space(mesh, p)
    interp, curl, qpts, qw = ts.nd_tet_tables(p, 2 * p + 2)
    qd = ts.geom_qdata(m.xe, np.ones(m.ne, dtype=np.int32), m.order, qpts, qw)
    assert (qd[:, 1, :] > 0).all() and abs(qd[:, 1, :].sum() / (np.pi * 2.74 ** 2 * 5.48) - 1) < 5e-4
    one = cf.coeff_ctx(a=1.0)

    def assemble(kind):
        Ae = O.element_matrices(kind, interp, curl, None, qd, one, nd.P)
        rows, cols, vals = [], [], []
        for e in range(m.ne):
            T = nd.dense_T(e)
            r, c = np.meshgrid(nd.idx[e], nd.idx[e], indexing="ij")
            rows.append(r.ravel())
            cols.append(c.ravel())
            vals.append((T.T @ Ae[e] @ T).ravel())
        return sp.csr_matrix((np.concatenate(vals), (np.concatenate(rows), np.concatenate(cols))), shape=(nd.ndofs, nd.ndofs))

    K, M = assemble(O.CURLCURL), assemble(O.ND_MASS)
    free = np.setdiff1d(np.arange(nd.ndofs), nd.ess_dofs)
    c0, L0, er = 299792458.0, 1.0e-2, 2.08
    sigma = (2 * np.pi * 2.0e9 * L0) ** 2 * er / c0 ** 2
    from tests import common

    lam = common.eigsh_above(K[free][:, free].tocsc(), M[free][:, free].tocsc(), 8, sigma, tol=1e-12)
    f = c0 * np.sqrt(lam / er) / (2 * np.pi * L0) / 1e9
    rel = np.abs(f - ANALYTIC) / ANALYTIC
    print("ND tet p=3 frequencies (GHz):", f, "rel. error vs closed form:", rel)
    assert rel.max() < 5e-4
    for a, b in ((1, 2), (4, 5), (6, 7)):                       # TE_1ml / TE_2ml pairs
        assert abs(f[a] - f[b]) < 1e-7 * f[a]
