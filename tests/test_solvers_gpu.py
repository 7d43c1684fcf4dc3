"""GPU parity of the device-resident linear algebra / smoother / multigrid / Krylov layer against
the NumPy restatement of the reference algorithms (oracle/solvers.py) on explicitly assembled oracle
matrices. Vector and Gram-Schmidt cases follow the reference's own unit tests
(/root/reference/test/unit/test-vector.cpp:17-134, test-orthog.cpp:99-374); the smoothers, multigrid
and Krylov solvers have no direct unit tests upstream (SURVEY §4), so they are pinned to the
algorithm restatement with a tight FP64 tolerance."""
import numpy as np
import pytest
import scipy.sparse.linalg as spla

from oracle import pyoracle as O
from oracle import solvers as S
from palace_b200.host import assemble as asm
from palace_b200.host import hexspace as hs
from tests import common

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu


def _dev(a):
    return torch.from_numpy(np.ascontiguousarray(a, dtype=np.float64)).cuda()


def _rel(a, b):
    return np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-300)


@pytest.fixture(scope="module")
def capi_mod():
    from palace_b200 import capi

    return capi


def test_vector_reductions_and_updates(b2p_ctx, capi_mod):
    capi = capi_mod
    rng = np.random.default_rng(0)
    n = 100003  # odd size, not a multiple of any block shape
    x, y, z = rng.standard_normal(n), rng.standard_normal(n), rng.standard_normal(n)
    xd, yd, zd = _dev(x), _dev(y), _dev(z)
    assert abs(capi.vec_dot(b2p_ctx, xd, yd) - x @ y) < 1e-10 * np.sqrt(n)
    assert abs(capi.vec_sum(b2p_ctx, xd) - x.sum()) < 1e-10 * np.sqrt(n)
    # test-vector.cpp: Sum of [1, 2, 3, 4] = 10
    assert capi.vec_sum(b2p_ctx, _dev([1.0, 2.0, 3.0, 4.0])) == 10.0
    capi.vec_axpby(b2p_ctx, 0.3, xd, -1.7, yd)
    assert _rel(yd.cpu().numpy(), 0.3 * x - 1.7 * y) < 1e-15
    capi.vec_axpbypcz(b2p_ctx, 2.0, xd, 0.5, yd, -1.0, zd)
    assert _rel(zd.cpu().numpy(), 2.0 * x + 0.5 * (0.3 * x - 1.7 * y) - z) < 1e-15


@pytest.mark.parametrize("kind", [0, 1, 2])
def test_gram_schmidt_matches_reference_algorithms(b2p_ctx, capi_mod, kind):
    """orthog.hpp:41-89; as in test-orthog.cpp the result must be orthogonal to the basis and H must
    hold the projection coefficients."""
    rng = np.random.default_rng(1)
    n, m = 5000, 11
    Q, _ = np.linalg.qr(rng.standard_normal((n, m)))
    V = [np.ascontiguousarray(Q[:, j]) for j in range(m)]
    w = rng.standard_normal(n)
    H_ref, w_ref = S.orthogonalize(kind, V, w)
    Vd = [_dev(v) for v in V]
    wd = _dev(w)
    H = capi_mod.vec_orthogonalize(b2p_ctx, kind, Vd, wd)
    assert np.abs(H - H_ref).max() < 1e-12 * np.abs(H_ref).max()
    assert _rel(wd.cpu().numpy(), w_ref) < 1e-12
    assert np.abs(Q.T @ wd.cpu().numpy()).max() < 1e-12 * np.linalg.norm(w)


@pytest.fixture(scope="module")
def hier(b2p_ctx):
    """p = 3 problem with its LOGARITHMIC p-hierarchy {1, 2, 3} (multigrid.hpp:44-70), ND + H1 aux."""
    prob = common.make_problem(n=(3, 2, 2), p=3)
    geom = common.gpu_geom(b2p_ctx, prob)
    orders = asm.p_sequence(3)
    assert orders == [1, 2, 3]
    blob = common.coefficient(O.CURLCURL_MASS, 3, "matrix", a_mass=1.0, a_curl=0.5)
    blob_h1 = common.coefficient(O.H1_DIFFUSION, 3, "matrix", a_mass=1.0)
    nd = {p: hs.build_nd_space(prob.mesh, prob.topo, p) for p in orders}
    h1 = {p: hs.build_h1_space(prob.mesh, prob.topo, p) for p in orders}
    fineA = common.gpu_par_operator(b2p_ctx, geom, prob, O.CURLCURL_MASS, blob, space=nd[3])
    fineG = common.gpu_par_operator(b2p_ctx, geom, prob, O.H1_DIFFUSION, blob_h1, space=h1[3])
    A, AG, Aor, AGor, Gop, Gor = {}, {}, {}, {}, {}, {}
    for p in orders:
        A[p] = fineA if p == 3 else common.gpu_par_operator(b2p_ctx, geom, prob, O.CURLCURL_MASS, blob, space=nd[p], fine_op=fineA.local_op)
        AG[p] = fineG if p == 3 else common.gpu_par_operator(b2p_ctx, geom, prob, O.H1_DIFFUSION, blob_h1, space=h1[p], fine_op=fineG.local_op)
        Aor[p] = common.oracle_matrix(prob, O.CURLCURL_MASS, blob, space=nd[p])
        AGor[p] = common.oracle_matrix(prob, O.H1_DIFFUSION, blob_h1, space=h1[p])
        Gop[p] = common.gpu_interp(b2p_ctx, h1[p], nd[p], asm.gradient_comps(p))
        Gor[p] = common.oracle_interp(h1[p], nd[p], hs.discrete_gradient_matrix(p))
    P, Por = {}, {}
    for pc, pf in zip(orders[:-1], orders[1:]):
        P[(pc, pf)] = common.gpu_interp(b2p_ctx, nd[pc], nd[pf], asm.nd_prolongation_comps(pc, pf))
        Por[(pc, pf)] = common.oracle_interp(nd[pc], nd[pf], hs.nd_prolongation_matrix(pc, pf))
    return dict(prob=prob, geom=geom, orders=orders, nd=nd, h1=h1, A=A, AG=AG, Aor=Aor, AGor=AGor, G=Gop, Gor=Gor, P=P, Por=Por,
                blob=blob)


def test_par_operator_matches_eliminated_matrix(b2p_ctx, hier):
    A, Ao = hier["A"][3], hier["Aor"][3]
    n = Ao.shape[0]
    rng = np.random.default_rng(2)
    x, y0 = rng.standard_normal(n), rng.standard_normal(n)
    yd = torch.empty(n, dtype=torch.float64, device="cuda")
    A.mult(_dev(x), yd)
    assert _rel(yd.cpu().numpy(), Ao @ x) < 1e-12
    yd = _dev(y0)
    A.add_mult(_dev(x), yd, -0.5)
    assert _rel(yd.cpu().numpy(), y0 - 0.5 * (Ao @ x)) < 1e-12
    dd = torch.empty(n, dtype=torch.float64, device="cuda")
    A.assemble_diagonal(dd)
    assert _rel(dd.cpu().numpy(), Ao.diagonal()) < 1e-12


@pytest.mark.parametrize("p", [1, 2, 3])
def test_discrete_gradient_and_prolongation(b2p_ctx, hier, p):
    rng = np.random.default_rng(3)
    G, Go = hier["G"][p], hier["Gor"][p]
    x = rng.standard_normal(Go.shape[1])
    yd = torch.empty(Go.shape[0], dtype=torch.float64, device="cuda")
    G.mult(_dev(x), yd)
    assert _rel(yd.cpu().numpy(), Go @ x) < 1e-13
    r = rng.standard_normal(Go.shape[0])
    xd = torch.empty(Go.shape[1], dtype=torch.float64, device="cuda")
    G.mult_transpose(_dev(r), xd)
    assert _rel(xd.cpu().numpy(), Go.T @ r) < 1e-13
    y0 = rng.standard_normal(Go.shape[0])
    yd = _dev(y0)
    G.add_mult(_dev(x), yd, 1.0)
    assert _rel(yd.cpu().numpy(), y0 + Go @ x) < 1e-13
    if p > 1:
        key = (hier["orders"][hier["orders"].index(p) - 1], p)
        Pm, Po = hier["P"][key], hier["Por"][key]
        xc = rng.standard_normal(Po.shape[1])
        yf = torch.empty(Po.shape[0], dtype=torch.float64, device="cuda")
        Pm.mult(_dev(xc), yf)
        assert _rel(yf.cpu().numpy(), Po @ xc) < 1e-13
        rf = rng.standard_normal(Po.shape[0])
        xcd = torch.empty(Po.shape[1], dtype=torch.float64, device="cuda")
        Pm.mult_transpose(_dev(rf), xcd)
        assert _rel(xcd.cpu().numpy(), Po.T @ rf) < 1e-13


def test_h1_prolongation(b2p_ctx, hier):
    h1 = hier["h1"]
    Pm = common.gpu_interp(b2p_ctx, h1[1], h1[2], asm.h1_prolongation_comps(1, 2))
    Po = common.oracle_interp(h1[1], h1[2], hs.h1_prolongation_matrix(1, 2))
    x = np.random.default_rng(4).standard_normal(Po.shape[1])
    yd = torch.empty(Po.shape[0], dtype=torch.float64, device="cuda")
    Pm.mult(_dev(x), yd)
    assert _rel(yd.cpu().numpy(), Po @ x) < 1e-13


def test_jacobi_smoother(b2p_ctx, capi_mod, hier):
    A, Ao = hier["A"][2], hier["Aor"][2]
    J = capi_mod.Solver.jacobi(b2p_ctx, omega=0.8)
    J.set_operator(A)
    x = np.random.default_rng(5).standard_normal(Ao.shape[0])
    yd = torch.empty_like(_dev(x))
    J.mult(_dev(x), yd)
    assert _rel(yd.cpu().numpy(), 0.8 * x / Ao.diagonal()) < 1e-13


@pytest.mark.parametrize("fourth_kind", [True, False])
@pytest.mark.parametrize("initial_guess", [False, True])
def test_chebyshev_smoother(b2p_ctx, capi_mod, hier, fourth_kind, initial_guess):
    A, Ao = hier["A"][3], hier["Aor"][3]
    n = Ao.shape[0]
    order = 6  # max(2p, 4) for p = 3 (iodata.cpp:533-536)
    C = capi_mod.Solver.chebyshev(b2p_ctx, smooth_it=1, order=order, sf_max=1.0, sf_min=0.0, fourth_kind=fourth_kind)
    C.set_operator(A)
    lam = C.lambda_max()
    dinv = 1.0 / Ao.diagonal()
    lam_ref = S.power_iteration(Ao, dinv, tol=1e-7, max_it=5000)
    assert abs(lam - lam_ref) < 2e-2 * lam_ref  # power iteration stopped at 1e-4 relative change from a random start
    rng = np.random.default_rng(6)
    x, y0 = rng.standard_normal(n), rng.standard_normal(n)
    yd, rd = _dev(y0), torch.empty(n, dtype=torch.float64, device="cuda")
    C.set_initial_guess(initial_guess)
    C.mult2(_dev(x), yd, rd)
    y_ref = S.chebyshev(Ao, dinv, lam, order, x, y0, initial_guess, fourth_kind)
    assert _rel(yd.cpu().numpy(), y_ref) < 1e-11


def _lams(capi, ctx, hier, p, order):
    """lambda_max of the ND and aux level operators as estimated on the device (fed to the oracle so
    that both sides run the same polynomial)."""
    c1 = capi.Solver.chebyshev(ctx, 1, order)
    c1.set_operator(hier["A"][p])
    c2 = capi.Solver.chebyshev(ctx, 1, order)
    c2.set_operator(hier["AG"][p])
    return c1.lambda_max(), c2.lambda_max()


def test_distributive_relaxation_smoother(b2p_ctx, capi_mod, hier):
    p, order = 2, 4
    A, AG, G = hier["A"][p], hier["AG"][p], hier["G"][p]
    Ao, AGo, Go = hier["Aor"][p], hier["AGor"][p], hier["Gor"][p]
    D = capi_mod.Solver.distrelax(b2p_ctx, G, smooth_it=1, cheby_smooth_it=1, cheby_order=order)
    D.distrelax_set_operators(A, AG)
    # The device smoother ran its own power iterations; rebuild the oracle with the same estimates.
    # (lambda_max is a property of the operator, so two estimates agree to the 1e-4 stopping
    # tolerance; the comparison below therefore uses a matching tolerance.)
    lam, lamG = _lams(capi_mod, b2p_ctx, hier, p, order)
    ref = S.DistRelax(Ao, AGo, Go, hier["h1"][p].ess_dofs, lam, lamG, order)
    rng = np.random.default_rng(7)
    n = Ao.shape[0]
    x, y0 = rng.standard_normal(n), rng.standard_normal(n)
    x[hier["nd"][p].ess_dofs] = 0.0
    for transpose in (False, True):
        yd, rd = _dev(y0), torch.empty(n, dtype=torch.float64, device="cuda")
        D.set_initial_guess(True)
        if transpose:
            D.mult_transpose2(_dev(x), yd, rd)
            y_ref = ref.mult_transpose2(x, y0, True)
        else:
            D.mult2(_dev(x), yd, rd)
            y_ref = ref.mult2(x, y0, True)
        assert _rel(yd.cpu().numpy(), y_ref) < 5e-3  # limited by the two independent lambda_max estimates


@pytest.mark.parametrize("kind,orth,side", [(0, 0, 0), (1, 0, 0), (1, 1, 1), (1, 2, 0), (2, 0, 0), (2, 2, 0)])
def test_krylov_solvers_match_reference_recurrences(b2p_ctx, capi_mod, hier, kind, orth, side):
    """CG / GMRES / FGMRES with a Jacobi preconditioner: same iterates as iterative.cpp's recurrences
    (iteration count and solution), including restarts."""
    # mass-dominated operator (well conditioned under Jacobi) so that restarted GMRES(10) converges
    prob, nd2 = hier["prob"], hier["nd"][2]
    blob = common.coefficient(O.CURLCURL_MASS, 3, "matrix", a_mass=1.0, a_curl=1e-3)
    A = common.gpu_par_operator(b2p_ctx, hier["geom"], prob, O.CURLCURL_MASS, blob, space=nd2)
    Ao = common.oracle_matrix(prob, O.CURLCURL_MASS, blob, space=nd2, q1d=prob.q1d)
    n = Ao.shape[0]
    b = np.random.default_rng(8).standard_normal(n)
    b[nd2.ess_dofs] = 0.0
    dinv = 1.0 / Ao.diagonal()
    Bref = lambda r: dinv * r
    J = capi_mod.Solver.jacobi(b2p_ctx)
    J.set_operator(A)
    K = capi_mod.Solver.krylov(b2p_ctx, kind, rel_tol=1e-8, max_it=300, max_dim=10, orthog=orth, pc_side=side)
    K.set_operator(A)
    K.set_preconditioner(J)
    xd = torch.zeros(n, dtype=torch.float64, device="cuda")
    K.mult(_dev(b), xd)
    st = K.stats()
    if kind == 0:
        x_ref, it_ref, _ = S.cg(Ao, b, Bref, rel_tol=1e-8, max_it=300)
    else:
        x_ref, it_ref, _ = S.gmres(Ao, b, Bref, rel_tol=1e-8, max_it=300, max_dim=10, orthog=orth, flexible=(kind == 2),
                                   right=(side == 0))
    assert st["converged"]
    # long Krylov recurrences amplify rounding differences (atomic scatter order): allow 10 % drift in the count
    assert abs(st["its"] - it_ref) <= max(1, it_ref // 10)
    x_direct = spla.spsolve(Ao.tocsc(), b)
    assert _rel(xd.cpu().numpy(), x_direct) < 1e-6
    assert _rel(xd.cpu().numpy(), x_ref) < 1e-7


def test_gmres_with_initial_guess(b2p_ctx, capi_mod, hier):
    A, Ao = hier["A"][1], hier["Aor"][1]
    n = Ao.shape[0]
    rng = np.random.default_rng(9)
    b, x0 = rng.standard_normal(n), rng.standard_normal(n)
    K = capi_mod.Solver.krylov(b2p_ctx, 1, rel_tol=1e-10, max_it=200, max_dim=200)
    K.set_operator(A)
    K.set_initial_guess(True)
    xd = _dev(x0)
    K.mult(_dev(b), xd)
    assert _rel(xd.cpu().numpy(), spla.spsolve(Ao.tocsc(), b)) < 1e-8


def _build_gmg(capi, ctx, hier, use_aux, order_of):
    orders = hier["orders"]
    coarse = capi.Solver.krylov(ctx, 0, rel_tol=1e-13, max_it=2000)
    cj = capi.Solver.jacobi(ctx)
    cj.set_operator(hier["A"][orders[0]])
    coarse.set_preconditioner(cj)
    coarse.set_operator(hier["A"][orders[0]])
    P = [hier["P"][(a, b)] for a, b in zip(orders[:-1], orders[1:])]
    G = [hier["G"][p] for p in orders] if use_aux else None
    M = capi.Solver.gmg(ctx, coarse, P, G, cycle_it=1, smooth_it=1, cheby_order=order_of, sf_max=1.0, sf_min=0.0, fourth_kind=True)
    M.gmg_set_operators([hier["A"][p] for p in orders], [hier["AG"][p] for p in orders] if use_aux else None)
    M._keep.append(cj)
    return M


@pytest.mark.parametrize("use_aux", [False, True])
def test_geometric_multigrid_vcycle(b2p_ctx, capi_mod, hier, use_aux):
    """One V-cycle (gmg.cpp:172-205) against the NumPy restatement, coarse level solved exactly."""
    orders, order = hier["orders"], 4
    M = _build_gmg(capi_mod, b2p_ctx, hier, use_aux, order)
    Aor = [hier["Aor"][p] for p in orders]
    Por = [hier["Por"][(a, b)] for a, b in zip(orders[:-1], orders[1:])]
    ess = [hier["nd"][p].ess_dofs for p in orders]
    smoothers = [None]
    for p in orders[1:]:
        lam, lamG = _lams(capi_mod, b2p_ctx, hier, p, order)
        if use_aux:
            smoothers.append(S.DistRelax(hier["Aor"][p], hier["AGor"][p], hier["Gor"][p], hier["h1"][p].ess_dofs, lam, lamG, order))
        else:
            smoothers.append(S.ChebSmoother(hier["Aor"][p], lam, order))
    lu = spla.splu(Aor[0].tocsc())
    ref = S.Gmg(Aor, Por, smoothers, lambda x: lu.solve(x), ess)
    n = Aor[-1].shape[0]
    x = np.random.default_rng(10).standard_normal(n)
    x[ess[-1]] = 0.0
    yd = torch.empty(n, dtype=torch.float64, device="cuda")
    M.mult(_dev(x), yd)
    assert _rel(yd.cpu().numpy(), ref.mult(x)) < 5e-3  # lambda_max estimates differ at the 1e-4 level per smoother


def test_fgmres_with_multigrid_preconditioner_solves_the_system(b2p_ctx, capi_mod, hier):
    """The reference's production configuration in miniature (iodata.cpp:453-466,519-536): flexible GMRES,
    p-multigrid V-cycle with Chebyshev + Hiptmair auxiliary-space smoothing."""
    M = _build_gmg(capi_mod, b2p_ctx, hier, True, 6)
    A, Ao = hier["A"][3], hier["Aor"][3]
    n = Ao.shape[0]
    b = np.random.default_rng(11).standard_normal(n)
    b[hier["nd"][3].ess_dofs] = 0.0
    K = capi_mod.Solver.krylov(b2p_ctx, 2, rel_tol=1e-10, max_it=60, max_dim=60)
    K.set_operator(A)
    K.set_preconditioner(M)
    xd = torch.zeros(n, dtype=torch.float64, device="cuda")
    K.mult(_dev(b), xd)
    st = K.stats()
    assert st["converged"] and st["its"] <= 25, st
    assert _rel(xd.cpu().numpy(), spla.spsolve(Ao.tocsc(), b)) < 1e-8


def test_multigrid_with_the_coarse_level_assembled_on_the_device(b2p_ctx, capi_mod, hier):
    """The reference's coarse-level flow (MfemWrapperSolver::SetOperator, linalg/solver.cpp:13-30): the multigrid hands its
    level-0 ParOperator to a solver that assembles it; here a Jacobi-PCG on the device CSR matrix. Same V-cycle as with the
    matrix-free coarse solve, and the FGMRES solve converges to the direct solution."""
    orders = hier["orders"]
    cg = capi_mod.Solver.krylov(b2p_ctx, 0, rel_tol=1e-13, max_it=2000)
    coarse = capi_mod.Solver.assembled(b2p_ctx, cg, capi_mod.Solver.jacobi(b2p_ctx))
    assert coarse.assembled_nnz() == -1
    P = [hier["P"][(a, b)] for a, b in zip(orders[:-1], orders[1:])]
    G = [hier["G"][p] for p in orders]
    M = capi_mod.Solver.gmg(b2p_ctx, coarse, P, G, cycle_it=1, smooth_it=1, cheby_order=6, sf_max=1.0, sf_min=0.0, fourth_kind=True)
    M.gmg_set_operators([hier["A"][p] for p in orders], [hier["AG"][p] for p in orders])
    assert M.assembled_nnz() >= hier["Aor"][1].tocsr().nnz  # the symbolic pattern keeps structural zeros
    Mref = _build_gmg(capi_mod, b2p_ctx, hier, True, 6)
    n = hier["Aor"][3].shape[0]
    x = np.random.default_rng(12).standard_normal(n)
    x[hier["nd"][3].ess_dofs] = 0.0
    y1, y2 = torch.empty(n, dtype=torch.float64, device="cuda"), torch.empty(n, dtype=torch.float64, device="cuda")
    M.mult(_dev(x), y1)
    Mref.mult(_dev(x), y2)
    assert _rel(y1.cpu().numpy(), y2.cpu().numpy()) < 1e-7  # two PCG solves to 1e-13 of different representations of level 0

    A, Ao = hier["A"][3], hier["Aor"][3]
    b = np.random.default_rng(11).standard_normal(n)
    b[hier["nd"][3].ess_dofs] = 0.0
    K = capi_mod.Solver.krylov(b2p_ctx, 2, rel_tol=1e-10, max_it=60, max_dim=60)
    K.set_operator(A)
    K.set_preconditioner(M)
    xd = torch.zeros(n, dtype=torch.float64, device="cuda")
    K.mult(_dev(b), xd)
    st = K.stats()
    assert st["converged"] and st["its"] <= 25, st
    assert _rel(xd.cpu().numpy(), spla.spsolve(Ao.tocsc(), b)) < 1e-8


def test_ksp_composer_builds_the_reference_configuration(b2p_ctx, capi_mod, hier):
    """BaseKspSolver (linalg/ksp.cpp:29-239,256-328): one configuration record -> FGMRES + p-multigrid (Chebyshev order
    max(2p, 4) + Hiptmair smoothing, coarse level assembled on the device) -- the same solve as the hand-composed objects, and
    the reference's counters NumTotalMult / NumTotalMultIts across two solves."""
    orders = hier["orders"]
    P = [hier["P"][(a, b)] for a, b in zip(orders[:-1], orders[1:])]
    G = [hier["G"][p] for p in orders]
    ksp = capi_mod.Ksp(b2p_ctx, order=3, P=P, G=G, krylov_solver=2, tol=1e-10, max_it=60, coarse_tol=1e-12, coarse_max_it=2000)
    assert ksp.cfg.mg_smooth_order == 6 and ksp.cfg.mg_smooth_aux == 1 and ksp.cfg.mg_cycle_it == 1  # iodata.cpp:519-536
    ksp.set_operators(hier["A"][3], [hier["A"][p] for p in orders], [hier["AG"][p] for p in orders])
    Ao = hier["Aor"][3]
    n = Ao.shape[0]
    sol = spla.splu(Ao.tocsc())
    its = 0
    for seed in (11, 12):
        b = np.random.default_rng(seed).standard_normal(n)
        b[hier["nd"][3].ess_dofs] = 0.0
        xd = torch.zeros(n, dtype=torch.float64, device="cuda")
        ksp.mult(_dev(b), xd)
        st = ksp.stats()
        assert st["converged"] and st["its"] <= 25, st
        its += st["its"]
        assert _rel(xd.cpu().numpy(), sol.solve(b)) < 1e-8
    assert st["num_total_mult"] == 2 and st["num_total_mult_its"] == its
    # one level: the coarse solver alone preconditions (ksp.cpp:232-237); Jacobi-PCG through the same record
    k1 = capi_mod.Ksp(b2p_ctx, order=1, krylov_solver=0, tol=1e-10, max_it=2000, coarse_type=0)
    k1.set_operators(hier["A"][1], [hier["A"][1]])
    A1 = hier["Aor"][1]
    b = np.random.default_rng(13).standard_normal(A1.shape[0])
    b[hier["nd"][1].ess_dofs] = 0.0
    xd = torch.zeros(A1.shape[0], dtype=torch.float64, device="cuda")
    k1.mult(_dev(b), xd)
    assert k1.stats()["converged"] and _rel(xd.cpu().numpy(), spla.spsolve(A1.tocsc(), b)) < 1e-7


def test_multi_gpu_partition_independence():
    """Runs tools/dist_check.py under torchrun on 2 GPUs when the machine has them."""
    import os
    import subprocess
    import sys

    if torch.cuda.device_count() < 2:
        pytest.skip("needs >= 2 GPUs")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr",
                          "127.0.0.1", "--master-port", "29611", os.path.join(root, "tools", "dist_check.py")],
                         capture_output=True, text=True, timeout=600)
    assert "DIST_CHECK OK" in out.stdout, out.stdout[-2000:] + out.stderr[-2000:]
