"""Posterior variance at test points (gpp_predict_var / gpp_dist_predict_var, PDEs.extend_sol_var) on the GPU:
against LAPACK on the oracle's matrices, against numpy on the device's own factor, its properties at collocation and
far-away points, the blocking edges (bit-identity across chunks, call splits and GEMM tile sizes), the call order, the
sharded paths on virtual ranks and the NCCL path on two GPUs."""
import os
import subprocess
import sys

import numpy as np
import pytest
import scipy.linalg as sla

from oracle import gp_oracle as o

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DOM = np.array([[0.0, 1.0], [0.0, 1.0]])
DOM_T = np.array([[0.0, 1.0], [-1.0, 1.0]])
NUG = 1e-5
BAND = max(1e-8, 10 * np.finfo(float).eps / NUG)       # the project's agreement band between two FP64 paths
# more than 10 kernel length scales (0.2, 0.3 and 0.05) outside both domains
FAR = np.array([[6.0, 6.0], [-5.0, 0.5], [0.5, -6.0], [7.0, -5.0], [-6.0, 6.0]])


def _problem(kind, NB=None, seed=0):
    from nonlinpdes_gpsolver_b200 import PDEs, InverseProblems
    np.random.seed(seed)
    if kind == "elliptic":
        p = PDEs.Nonlinear_elliptic2d(alpha=1.0, m=3, bdy=o.elliptic_u, rhs=o.elliptic_f, domain=DOM)
        args, gram = (300, 44), ("Gaussian", 0.2)
    elif kind == "burgers":
        p = PDEs.Burgers(alpha=1.0, nu=0.02, bdy=o.burgers_bdy, rhs=lambda a, b: 0, domain=DOM_T)
        args, gram = (200, 42), ("anisotropic_Gaussian", [0.3, 0.05])
    elif kind == "eikonal":
        p = PDEs.Eikonal(eps=1e-2, bdy=lambda a, b: 0, rhs=lambda a, b: 1, domain=DOM)
        args, gram = (200, 40), ("Gaussian", 0.2)
    else:
        p = InverseProblems.Darcy_flow2d(bdy=lambda a, b: 0, rhs=lambda a, b: 1, domain=DOM)
        args, gram = (150, 40, 20), ("Gaussian", 0.2)
    if NB:
        p._engine().set_option("NB", NB)
    p.sampled_pts(*args)
    p.Gram_matrix(gram[0], gram[1], NUG, "adaptive")
    return p, gram


def _test_points(p, dom, n=500, seed=11):
    rnd = np.random.RandomState(seed).uniform(dom[:, 0], dom[:, 1], (n, 2))
    return np.concatenate([rnd, p.X_domain, p.X_boundary, FAR])


def _oracle_var(p, gram, layout, add, X):
    """scipy.linalg.solve_triangular(cholesky(Theta_oracle), Theta_test_oracle^T): the LAPACK reference."""
    Xb = p.X_boundary if layout != "Darcy_flow2d_a" else np.zeros((0, 2))
    theta = o._assemble(p.X_domain, Xb, layout, gram[0], gram[1]) + np.diag(add)
    W = sla.solve_triangular(np.linalg.cholesky(theta), o._theta_test(X, p.X_domain, Xb, layout, gram[0], gram[1]).T, lower=True)
    kxx = o.functional(gram[0], gram[1], "id", "id", X[:, 0], X[:, 1], X[:, 0], X[:, 1])
    return kxx - np.sum(W * W, axis=0)


def _same_L_var(eng, slot, X):
    L, T = eng.gram_download(slot, 1), eng.theta_test(slot, X)
    W = sla.solve_triangular(L, T.T, lower=True)
    return 1.0 - np.sum(W * W, axis=0)


def _check_slot(p, gram, eng, slot, layout, add, X, var, n_coll):
    assert var.shape == (X.shape[0],)
    np.testing.assert_allclose(var, _oracle_var(p, gram, layout, add, X), rtol=0, atol=BAND)
    np.testing.assert_allclose(var, _same_L_var(eng, slot, X), rtol=0, atol=1e-12)
    coll = var[500:500 + n_coll]
    assert np.all(coll <= NUG + 1e-12), coll.max()
    assert np.all(var[-len(FAR):] >= 1 - 1e-12), var[-len(FAR):]
    assert np.all(var >= -1e-12), var.min()


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["elliptic", "burgers", "eikonal"])
def test_against_lapack_and_own_factor(kind):
    p, gram = _problem(kind)
    p.Gram_Cholesky()
    dom = DOM_T if kind == "burgers" else DOM
    X = _test_points(p, dom)
    p.extend_sol_var(X)
    layout = {"elliptic": "Nonlinear_elliptic", "burgers": "Burgers", "eikonal": "Eikonal"}[kind]
    _check_slot(p, gram, p._engine(), 0, layout, p._nugget_add, X, p.extended_var, p.N_domain + p.N_boundary)


@pytest.mark.gpu
def test_darcy_both_slots():
    p, gram = _problem("darcy")
    p.Gram_Cholesky()
    X = _test_points(p, DOM)
    p.extend_sol_var(X)
    eng = p._engine()
    _check_slot(p, gram, eng, 0, "Darcy_flow2d", p._nugget_add[0], X, p.extended_var_u, p.N_domain + p.N_boundary)
    # Theta_a has no boundary rows: its collocation points are the interior ones
    _check_slot(p, gram, eng, 1, "Darcy_flow2d_a", p._nugget_add[1], X, p.extended_var_a, p.N_domain)
    assert not np.array_equal(p.extended_var_u, p.extended_var_a)


@pytest.mark.gpu
def test_blocking_edges_bit_identical():
    """NB = 128 with M = 2N + Nb not a multiple of 128 (ragged last block), N_test = 1, 63, 65 and 20 000 (two chunks):
    the same points give the same bits whatever the call split and the GEMM tile size."""
    from nonlinpdes_gpsolver_b200 import PDEs
    np.random.seed(4)
    p = PDEs.Nonlinear_elliptic2d(alpha=1.0, m=3, bdy=o.elliptic_u, rhs=o.elliptic_f, domain=DOM)
    eng = p._engine()
    eng.set_option("NB", 128)
    p.sampled_pts(951, 101)
    p.Gram_matrix("Gaussian", 0.2, NUG, "adaptive")
    p.Gram_Cholesky()
    M = eng.gram_size(0)[0]
    assert M == 2002 and M % 128 != 0
    X = np.random.RandomState(3).uniform(0, 1, (20000, 2))
    full = eng.predict_var(0, X)
    cuts = [0, 1, 64, 129, 20000]                      # 1, 63, 65 and the 19 871 remaining rows
    parts = np.concatenate([eng.predict_var(0, X[a:b]) for a, b in zip(cuts[:-1], cuts[1:])])
    assert np.array_equal(parts, full)
    for tile in (64, 128):
        eng.set_option("gemm_tile", tile)
        assert np.array_equal(eng.predict_var(0, X), full)
        assert np.array_equal(eng.predict_var(0, X[:65]), full[:65])
    eng.set_option("gemm_tile", 0)
    sub = X[::50]
    np.testing.assert_allclose(full[::50], _same_L_var(eng, 0, sub), rtol=0, atol=1e-12)


@pytest.mark.gpu
def test_call_order():
    """Before GN_method (no U in the upper triangle of T) and after it (gpp_inverse wrote U there): the same bits.
    Before Gram_Cholesky: the class raises RuntimeError, the engine GppError."""
    from nonlinpdes_gpsolver_b200 import _lib
    p, gram = _problem("elliptic", NB=128)
    X = _test_points(p, DOM, n=200)
    with pytest.raises(RuntimeError, match="Gram_Cholesky"):
        p.extend_sol_var(X)
    with pytest.raises(_lib.GppError, match="potrf first"):
        p._engine().predict_var(0, X)
    p.Gram_Cholesky()
    p.extend_sol_var(X)
    before = p.extended_var.copy()
    p.GN_method(2, 1, np.zeros(p.N_domain), print_hist=False)
    p.extend_sol_var(X)
    assert np.array_equal(p.extended_var, before)


@pytest.mark.gpu
def test_refuses_bad_arguments():
    from nonlinpdes_gpsolver_b200 import _lib
    eng = _lib.Engine()
    with pytest.raises(_lib.GppError, match="not assembled"):
        eng.predict_var(0, np.zeros((3, 2)))
    with pytest.raises(ValueError):
        eng.predict_var(0, np.zeros((0, 2)))
    with pytest.raises(_lib.GppError):
        eng.dist_predict_var(np.zeros((3, 2)))          # not a sharded handle


def _sharded_and_single(kind, N, Nb, NB, nranks, Q):
    from nonlinpdes_gpsolver_b200 import PDEs
    make = {"burgers": lambda: PDEs.Burgers(alpha=1.0, nu=0.02, bdy=o.burgers_bdy, rhs=lambda a, b: 0, domain=DOM_T),
            "elliptic": lambda: PDEs.Nonlinear_elliptic2d(alpha=1.0, m=3, bdy=o.elliptic_u, rhs=o.elliptic_f, domain=DOM)}[kind]
    gram = ("anisotropic_Gaussian", [0.3, 0.05]) if kind == "burgers" else ("Gaussian", 0.2)
    out = []
    for shard in (False, True):
        np.random.seed(9)
        p = make()
        p._engine().set_option("NB", NB)
        p.sampled_pts(N, Nb)
        if shard:
            p.shard(virtual_ranks=nranks, Q=Q)
        p.Gram_matrix(gram[0], gram[1], NUG, "adaptive")
        p.Gram_Cholesky()
        out.append(p)
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("kind,nranks,Q,N,Nb", [
    ("burgers", 1, 1, 700, 99),
    ("burgers", 3, 1, 700, 99),
    ("burgers", 8, 1, 700, 99),
    ("elliptic", 4, 2, 600, 80),       # 2 x 2 grid
])
def test_virtual_sharded(kind, nranks, Q, N, Nb):
    single, sh = _sharded_and_single(kind, N, Nb, 128, nranks, Q)
    dom = DOM_T if kind == "burgers" else DOM
    X = np.random.RandomState(5).uniform(dom[:, 0], dom[:, 1], (1000, 2))
    sh.extend_sol_var(X)
    assert np.array_equal(sh.extended_var, sh._engine().predict_var(0, X))
    single.extend_sol_var(X)
    np.testing.assert_allclose(sh.extended_var, single.extended_var, rtol=0, atol=BAND)
    # fewer test points than ranks: some ranks own no rows
    few = X[:nranks - 1] if nranks > 1 else X[:1]
    sh.extend_sol_var(few)
    assert np.array_equal(sh.extended_var, sh._engine().predict_var(0, few))


@pytest.mark.gpu
def test_nccl_two_gpus_same_vector_on_every_rank():
    """torchrun on 2 GPUs (tools/dist_solve.py --var-points --check): every rank returns the same vector, bit-identical to
    gpp_predict_var on its own copy of the factor."""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs >= 2 GPUs")
    out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
                          "--master-addr", "127.0.0.1", "--master-port", "29631", os.path.join(ROOT, "tools", "dist_solve.py"),
                          "--pde", "burgers", "--N", "1200", "--Nb", "120", "--NB", "256", "--reps", "1", "--gn_steps", "1",
                          "--check", "--var-points", "777"], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stdout[-2000:] + out.stderr[-2000:]
    assert '"var_same_on_ranks_and_single_rank": true' in out.stdout
