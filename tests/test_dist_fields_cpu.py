"""Sharded Burgers / Eikonal on the CPU: the Theta^-1 sub-block plans of three-field Hessians (blocks that straddle the
boundary between two unknown fields, odd segment offsets) checked on the host through the C ABI, and the Burgers class
flow through the fake engine (tests/fake_engine.py, backed by the oracle)."""
import numpy as np
import pytest

from fake_engine import FakeEngine
from oracle import gp_oracle as o

DOM = np.array([[0.0, 1.0], [0.0, 1.0]])
DOM_T = np.array([[0.0, 1.0], [-1.0, 1.0]])
GRIDS = ((1, 1), (2, 1), (3, 1), (2, 2), (8, 1), (2, 4), (4, 2))


@pytest.fixture()
def fake(monkeypatch):
    from nonlinpdes_gpsolver_b200 import _lib
    monkeypatch.setattr(_lib, "Engine", lambda *a, **k: FakeEngine())
    monkeypatch.setattr(_lib, "_default_engine", None)
    return _lib


@pytest.mark.parametrize("pde", ["Burgers", "Eikonal"])
@pytest.mark.parametrize("N,NB", [(700, 128), (701, 128), (1024, 256), (1500, 512)])
def test_three_field_hessian_plans_are_consistent(pde, N, NB):
    """Every lower block of the 3N x 3N Hessian has one owner; every element gets each term of its field pair exactly once,
    from the right rows of U and the right K range."""
    from nonlinpdes_gpsolver_b200 import _lib
    for P, Q in GRIDS:
        assert _lib.dist_hess_plan_check(N, NB, P, Q, pde, nb_extra=99) == 0, (pde, N, NB, P, Q)


def test_elliptic_hessian_plans_through_the_field_check():
    from nonlinpdes_gpsolver_b200 import _lib
    for N, NB in ((700, 128), (701, 128), (1300, 128), (2048, 256), (1500, 512)):
        for P, Q in GRIDS:
            assert _lib.dist_hess_plan_check(N, NB, P, Q, "Nonlinear_elliptic", nb_extra=96) == 0, (N, NB, P, Q)


def test_hessian_plan_check_refuses_what_does_not_shard():
    from nonlinpdes_gpsolver_b200 import _lib
    for pde in ("Darcy_flow2d", "Nonlinear_elliptic_relaxed"):
        assert _lib.dist_hess_plan_check(700, 128, 2, 1, pde, nb_extra=99) == -1
    assert _lib.dist_hess_plan_check(700, 100, 2, 1, "Burgers") == -1        # block size must be a multiple of 64


def test_sharded_burgers_class_flow_on_fake_engine(fake):
    """PDEs.Burgers(...).shard(): assembly, nugget, factorisation, inverse and GN steps go through the dist_* calls only,
    the reference's RNG order holds (points, then the initial guess) and the loss history is the oracle's."""
    from nonlinpdes_gpsolver_b200 import InverseProblems, PDEs
    N, Nb, steps, seed = 60, 20, 3, 7
    np.random.seed(seed)
    p = PDEs.Burgers(alpha=1.0, nu=0.02, bdy=o.burgers_bdy, rhs=lambda a, b: 0, domain=DOM_T)
    p.sampled_pts(N, Nb)
    assert p.shard(virtual_ranks=4, Q=2) is p
    assert p._engine().dist_info() == dict(rank=0, world=4, P=2, Q=2)
    p.Gram_matrix("anisotropic_Gaussian", (0.3, 0.05), 1e-5, "adaptive")
    p.Gram_Cholesky()
    p.GN_method(steps, 1, "rdm", print_hist=False)
    calls = p._engine().calls
    assert "dist_gram_assemble" in calls and "dist_potrf" in calls and "dist_inverse" in calls and calls.count("dist_gn_step") == steps
    assert not any(c.startswith("inverse[") for c in calls)
    np.random.seed(seed)
    Xd, Xb = o.sampled_pts_rdm(N, Nb, DOM_T, time_dependent=True)
    init = np.random.normal(0.0, 1.0, 3 * N)
    ref = o.Burgers(1.0, 0.02)
    ref.set_points(Xd, Xb, p.rhs_f, p.bdy_g)
    ref.Gram_matrix("anisotropic_Gaussian", (0.3, 0.05), 1e-5, "adaptive")
    ref.Gram_Cholesky("tri")
    ref.GN_method(steps, 1, init)
    assert np.array_equal(p.X_domain, Xd) and np.array_equal(p.X_boundary, Xb)
    assert np.array_equal(p.init_sol, init)
    assert list(np.atleast_1d(p.ratio)) == list(np.atleast_1d(ref.ratio))
    np.testing.assert_allclose(p.loss_hist, ref.loss_hist, rtol=1e-9)
    np.testing.assert_allclose(p.sol_sampled_pts, ref.sol_sampled_pts, rtol=1e-7, atol=1e-9)
    with pytest.raises(NotImplementedError):
        InverseProblems.Darcy_flow2d(bdy=lambda a, b: 0, rhs=lambda a, b: 1, domain=DOM).shard(virtual_ranks=2)
