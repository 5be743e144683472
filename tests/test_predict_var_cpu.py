"""Posterior variance, host side, on the CPU: extend_sol_var / solver_GP.test_var driven through a fake engine whose
predict_var / dist_predict_var come from the oracle.  Checks the class flow (which engine call, which slot), attribute
names, state errors, Darcy's two fields and the console lines; the numbers themselves are checked on the GPU
(tests/test_predict_var.py)."""
from types import SimpleNamespace

import numpy as np
import pytest
import scipy.linalg as sla

from fake_engine import FakeEngine
from oracle import gp_oracle as o

DOM = np.array([[0.0, 1.0], [0.0, 1.0]])
DOM_T = np.array([[0.0, 1.0], [-1.0, 1.0]])


class VarFakeEngine(FakeEngine):
    """FakeEngine plus the posterior-variance calls: kappa(x, x) - |L^{-1} theta(x)|^2 with the oracle's theta."""

    def predict_var(self, slot, X_test):
        s = self.slots[slot]
        Xb = self.Xb if s["layout"] != "Darcy_flow2d_a" else np.zeros((0, 2))
        X = np.asarray(X_test, float)
        W = sla.solve_triangular(s["L"], o._theta_test(X, self.Xd, Xb, s["layout"], s["kernel"], s["kp"]).T, lower=True)
        self.calls.append(f"predict_var[{slot}]")
        kxx = o.functional(s["kernel"], s["kp"], "id", "id", X[:, 0], X[:, 1], X[:, 0], X[:, 1])
        return kxx - np.sum(W * W, axis=0)

    def dist_predict_var(self, X_test):
        out = self.predict_var(0, X_test)
        self.calls[-1] = "dist_predict_var"
        return out


@pytest.fixture()
def fake(monkeypatch):
    from nonlinpdes_gpsolver_b200 import _lib
    monkeypatch.setattr(_lib, "Engine", lambda *a, **k: VarFakeEngine())
    monkeypatch.setattr(_lib, "_default_engine", None)
    return _lib


def _oracle_var(Xd, Xb, layout, kernel, kp, add, X):
    theta = o._assemble(Xd, Xb, layout, kernel, kp) + np.diag(add)
    W = sla.solve_triangular(np.linalg.cholesky(theta), o._theta_test(X, Xd, Xb, layout, kernel, kp).T, lower=True)
    return 1.0 - np.sum(W * W, axis=0)


@pytest.mark.parametrize("name", ["elliptic", "burgers"])
def test_extend_sol_var_flow_and_state_errors(fake, name):
    from nonlinpdes_gpsolver_b200 import PDEs
    if name == "elliptic":
        p = PDEs.Nonlinear_elliptic2d(alpha=1.0, m=3, bdy=o.elliptic_u, rhs=o.elliptic_f, domain=DOM)
        kernel, kp, dom, layout = "Gaussian", 0.2, DOM, "Nonlinear_elliptic"
    else:
        p = PDEs.Burgers(alpha=1.0, nu=0.02, bdy=o.burgers_bdy, rhs=lambda a, b: 0, domain=DOM_T)
        kernel, kp, dom, layout = "anisotropic_Gaussian", (0.3, 0.05), DOM_T, "Burgers"
    Xt = np.random.RandomState(2).uniform(dom[:, 0], dom[:, 1], (13, 2))
    with pytest.raises(RuntimeError, match="Gram_Cholesky"):
        p.extend_sol_var(Xt)                            # no points yet
    np.random.seed(1)
    p.sampled_pts(50, 16)
    with pytest.raises(RuntimeError, match="Gram_Cholesky"):
        p.extend_sol_var(Xt)
    p.Gram_matrix(kernel, kp, 1e-5, "adaptive")
    with pytest.raises(RuntimeError, match="Gram_Cholesky"):
        p.extend_sol_var(Xt)
    assert not hasattr(p, "extended_var")
    p.Gram_Cholesky()
    p.extend_sol_var(Xt)                                # allowed in state 'chol'
    ref = _oracle_var(p.X_domain, p.X_boundary, layout, kernel, kp, p._nugget_add, Xt)
    np.testing.assert_allclose(p.extended_var, ref, rtol=0, atol=1e-10)
    assert p._engine().calls[-1] == "predict_var[0]"
    assert not hasattr(p, "X_test") and not hasattr(p, "N_test")     # extend_sol's attributes stay its own
    p.GN_method(2, 1, "rdm", print_hist=False)
    p.extend_sol_var(Xt[:4])                            # and in state 'solved'
    np.testing.assert_allclose(p.extended_var, ref[:4], rtol=0, atol=1e-10)


def test_sharded_problem_uses_the_split_call(fake):
    from nonlinpdes_gpsolver_b200 import PDEs
    p = PDEs.Burgers(alpha=1.0, nu=0.02, bdy=o.burgers_bdy, rhs=lambda a, b: 0, domain=DOM_T)
    np.random.seed(1)
    p.sampled_pts(40, 12)
    p.shard(virtual_ranks=3)
    p.Gram_matrix("anisotropic_Gaussian", (0.3, 0.05), 1e-5, "adaptive")
    p.Gram_Cholesky()
    Xt = np.random.RandomState(2).uniform(DOM_T[:, 0], DOM_T[:, 1], (2, 2))
    p.extend_sol_var(Xt)
    assert p._engine().calls[-1] == "dist_predict_var"
    assert p.extended_var.shape == (2,)


def test_darcy_two_fields(fake):
    from nonlinpdes_gpsolver_b200.InverseProblems import Darcy_flow2d
    d = Darcy_flow2d(bdy=lambda a, b: 0, rhs=lambda a, b: 1, domain=DOM)
    np.random.seed(3)
    d.sampled_pts(40, 12, 10)
    d.Gram_matrix("Gaussian", 0.2, 1e-5, "adaptive")
    Xt = np.random.RandomState(4).uniform(0, 1, (9, 2))
    with pytest.raises(RuntimeError):
        d.extend_sol_var(Xt)
    d.Gram_Cholesky()
    d.extend_sol_var(Xt)
    assert d._engine().calls[-2:] == ["predict_var[0]", "predict_var[1]"]
    add_u, add_a = d._nugget_add
    np.testing.assert_allclose(d.extended_var_u, _oracle_var(d.X_domain, d.X_boundary, "Darcy_flow2d", "Gaussian", 0.2, add_u, Xt),
                               rtol=0, atol=1e-10)
    np.testing.assert_allclose(d.extended_var_a, _oracle_var(d.X_domain, np.zeros((0, 2)), "Darcy_flow2d_a", "Gaussian", 0.2, add_a, Xt),
                               rtol=0, atol=1e-10)
    assert not hasattr(d, "extended_var")


def _cfg():
    return SimpleNamespace(alpha=1.0, m=3, kernel="Gaussian", kernel_parameter=0.2, nugget=1e-5, nugget_type="adaptive",
                           GNsteps=2, step_size=1, initial_sol="rdm", print_hist=False)


def test_solver_test_var_console_lines(fake, capsys):
    from nonlinpdes_gpsolver_b200.solver import solver_GP
    s = solver_GP(_cfg(), PDE_type="Nonlinear_elliptic")
    s.set_equation(bdy=o.elliptic_u, rhs=o.elliptic_f, domain=DOM, print_option=False)
    np.random.seed(0)
    s.auto_sample(50, 16, print_option=False)
    s.solve(print_option=False)
    capsys.readouterr()
    Xt = np.concatenate([np.random.RandomState(5).uniform(0, 1, (11, 2)), [[8.0, 8.0]]])
    s.test_var(Xt)
    out = capsys.readouterr().out.splitlines()
    var = s.eqn.extended_var
    assert s.test_var_all is var
    assert out == [f'[Test variance] Max posterior standard deviation {np.sqrt(np.max(np.maximum(var, 0.0)))}']
    assert abs(np.sqrt(np.max(var)) - 1.0) < 1e-12      # the far point: the prior standard deviation
    s.test_var(Xt, print_option=False)
    assert capsys.readouterr().out == ''


def test_solver_test_var_darcy(fake, capsys):
    from nonlinpdes_gpsolver_b200.solver import solver_GP
    s = solver_GP(_cfg(), PDE_type="Darcy_flow2d")
    s.set_equation(bdy=lambda a, b: 0, rhs=lambda a, b: 1, domain=DOM, print_option=False)
    np.random.seed(0)
    s.auto_sample_IP(40, 12, 10, print_option=False)
    s.eqn.Gram_matrix("Gaussian", 0.2, 1e-5, "adaptive")
    s.eqn.Gram_Cholesky()
    capsys.readouterr()
    s.test_var(np.random.RandomState(6).uniform(0, 1, (7, 2)))
    out = capsys.readouterr().out.splitlines()
    su = np.sqrt(np.max(np.maximum(s.eqn.extended_var_u, 0.0)))
    sa = np.sqrt(np.max(np.maximum(s.eqn.extended_var_a, 0.0)))
    assert out == [f'[Test variance] Max posterior standard deviation of u {su}',
                   f'[Test variance] Max posterior standard deviation of a {sa}']
    assert s.test_var_all is s.eqn.extended_var_u and s.test_var_all_a is s.eqn.extended_var_a
