"""Sharded GN path for the three-field problems (Burgers, Eikonal) on the GPU.
ONE GPU: the task plans of n "virtual" ranks run one after the other on the device (shared storage, no NCCL) -- Burgers
through the class against the unsharded path, Eikonal through the engine-level dist_* calls, the plan cache across
layouts, and the refusals.  >= 2 GPUs / one rank under torchrun: the real NCCL path (tools/dist_solve.py --pde burgers)."""
import os
import subprocess
import sys

import numpy as np
import pytest

from oracle import gp_oracle as o

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DOM = np.array([[0.0, 1.0], [0.0, 1.0]])
DOM_T = np.array([[0.0, 1.0], [-1.0, 1.0]])
NUG = 1e-5
BAND = max(1e-8, 10 * np.finfo(float).eps / NUG)       # the project's agreement band between two FP64 paths


def _burgers(PDEs, N, Nb, NB, seed=3):
    np.random.seed(seed)
    p = PDEs.Burgers(alpha=1.0, nu=0.02, bdy=o.burgers_bdy, rhs=lambda a, b: 0, domain=DOM_T)
    p._engine().set_option("NB", NB)
    p.sampled_pts(N, Nb)
    return p, np.random.normal(0.0, 1.0, 3 * N)


@pytest.mark.gpu
@pytest.mark.parametrize("nranks,Q,N,Nb,NB", [
    (1, 1, 500, 60, 128),
    (2, 1, 700, 99, 128),       # 3N = 2100: blocks straddle the field boundaries at 700 and 1400
    (3, 1, 701, 99, 128),       # odd segment offsets
    (4, 2, 700, 99, 128),       # 2 x 2 grid
    (8, 1, 900, 120, 128),
    (2, 1, 1500, 150, 512),
])
def test_virtual_sharded_burgers_matches_single_gpu(nranks, Q, N, Nb, NB):
    from nonlinpdes_gpsolver_b200 import PDEs
    steps = 3
    ref, init = _burgers(PDEs, N, Nb, NB)
    ref.Gram_matrix("anisotropic_Gaussian", [0.3, 0.05], NUG, "adaptive")
    theta = ref.Theta
    ref.Gram_Cholesky()
    ref.GN_method(steps, 1, init, print_hist=False)
    sh, init2 = _burgers(PDEs, N, Nb, NB)
    assert np.array_equal(init, init2)
    sh.shard(virtual_ranks=nranks, Q=Q)
    assert sh._engine().dist_info() == dict(rank=0, world=nranks, P=nranks // Q, Q=Q)
    sh.Gram_matrix("anisotropic_Gaussian", [0.3, 0.05], NUG, "adaptive")
    assert list(sh.ratio) == list(ref.ratio)
    sh.Gram_Cholesky()
    assert sh.chol_info == 0
    L, M = sh.L, theta.shape[0]
    assert np.max(np.abs(L @ L.T - theta)) <= 1e-13 * np.max(np.abs(theta)) * np.sqrt(M)
    sh.GN_method(steps, 1, init, print_hist=False)
    np.testing.assert_allclose(sh.loss_hist, ref.loss_hist, rtol=BAND)
    np.testing.assert_allclose(sh.sol, ref.sol, rtol=0, atol=BAND * np.max(np.abs(ref.sol)))
    Xt = np.random.RandomState(1).uniform(DOM_T[:, 0], DOM_T[:, 1], (40, 2))
    sh.extend_sol(Xt)
    ref.extend_sol(Xt)
    np.testing.assert_allclose(sh.extended_sol, ref.extended_sol, rtol=0, atol=BAND * np.max(np.abs(ref.extended_sol)))
    # a second solve on the same handle reuses the cached plans and buffers and repeats the first one exactly
    first = list(sh.loss_hist)
    sh.Gram_matrix("anisotropic_Gaussian", [0.3, 0.05], NUG, "adaptive")
    sh.Gram_Cholesky()
    sh.GN_method(steps, 1, init, print_hist=False)
    assert sh.loss_hist == first


def _adaptive_nugget(diag, N):
    """nugget * trace ratios of the four operator blocks (PDEs._GPProblem._nugget_vector)."""
    tr_last = np.sum(diag[3 * N:])
    r = np.ones(diag.shape[0])
    for p in range(3):
        r[p * N:(p + 1) * N] = np.sum(diag[p * N:(p + 1) * N]) / tr_last
    return NUG * r


def _engine_solve(eng, layout, kernel, kp, pde, params, rhs_f, bdy_g, z0, steps):
    """The sharded call sequence of the classes, on an engine whose points and ranks are set up."""
    eng.dist_gram_assemble(layout, kernel, kp)
    eng.dist_add_diag(_adaptive_nugget(eng.dist_get_diag(), eng.N))
    assert eng.dist_potrf() == 0
    eng.gn_setup(pde, params, rhs_f, bdy_g)
    eng.dist_inverse()
    eng.gn_set_z(z0)
    hist = [eng.gn_loss()] + [eng.dist_gn_step(1.0) for _ in range(steps)]
    return hist, eng.gn_get_z()


def _virtual_engine(Xd, Xb, NB, nranks, Q):
    from nonlinpdes_gpsolver_b200 import _lib
    eng = _lib.Engine()
    eng.set_option("NB", NB)
    eng.set_points(Xd, Xb)
    eng.dist_init_virtual(nranks)
    eng.dist_set_grid(nranks // Q, Q)
    return eng


@pytest.mark.gpu
@pytest.mark.parametrize("nranks,Q,N,Nb,NB", [(3, 1, 701, 100, 128), (4, 2, 700, 100, 128)])
def test_virtual_sharded_eikonal_engine_level_and_plan_cache(nranks, Q, N, Nb, NB):
    """Eikonal through the engine-level dist_* calls against the unsharded class; then, on the same engine, a Burgers-layout
    solve at the same N, Nb must give the results of a fresh engine (the sub-block plans are cached per layout)."""
    from nonlinpdes_gpsolver_b200 import PDEs
    steps, eps = 3, 1e-2
    np.random.seed(5)
    ref = PDEs.Eikonal(eps=eps, bdy=lambda a, b: 0, rhs=lambda a, b: 1, domain=DOM)
    ref._engine().set_option("NB", NB)
    ref.sampled_pts(N, Nb)
    ref.Gram_matrix("Gaussian", 0.2, NUG, "adaptive")
    ref.Gram_Cholesky()
    ref.GN_method(steps, 1, "zero", print_hist=False)
    eng = _virtual_engine(ref.X_domain, ref.X_boundary, NB, nranks, Q)
    hist, z = _engine_solve(eng, "Eikonal", "Gaussian", 0.2, "Eikonal", [eps], ref.rhs_f, ref.bdy_g, np.zeros(3 * N), steps)
    np.testing.assert_allclose(hist, ref.loss_hist, rtol=BAND)
    np.testing.assert_allclose(z, ref.sol, rtol=0, atol=BAND * np.max(np.abs(ref.sol)))
    # Burgers layout, same N and Nb (same M and operator offsets as Eikonal), on the same engine and on a fresh one
    bdy = o.burgers_bdy(ref.X_boundary[:, 0], ref.X_boundary[:, 1])
    z0 = np.random.RandomState(2).standard_normal(3 * N)
    args = ("Burgers", "anisotropic_Gaussian", [0.3, 0.05], "Burgers", [1.0, 0.02], np.zeros(N), bdy, z0, steps)
    hist_b, z_b = _engine_solve(eng, *args)
    fresh = _virtual_engine(ref.X_domain, ref.X_boundary, NB, nranks, Q)
    hist_f, z_f = _engine_solve(fresh, *args)
    assert hist_b == hist_f and np.array_equal(z_b, z_f)


@pytest.mark.gpu
def test_sharded_refusals():
    from nonlinpdes_gpsolver_b200 import _lib
    rng = np.random.RandomState(0)
    N, Nb = 300, 40
    Xd, Xb = rng.uniform(0, 1, (N, 2)), rng.uniform(0, 1, (Nb, 2))
    eng = _virtual_engine(Xd, Xb, 128, 2, 1)
    # Darcy's coefficient layout: no sharded Hessian
    eng.dist_gram_assemble("Darcy_flow2d_a", "Gaussian", 0.2)
    eng.dist_add_diag(np.full(3 * N, 1e-3))
    eng.dist_potrf()
    with pytest.raises(_lib.GppError):
        eng.dist_inverse()
    # the GN state is Burgers, the inverse was last planned for the Eikonal layout
    zero_bdy = np.zeros(Nb)
    eng.dist_gram_assemble("Burgers", "anisotropic_Gaussian", [0.3, 0.05])
    eng.dist_add_diag(_adaptive_nugget(eng.dist_get_diag(), N))
    assert eng.dist_potrf() == 0
    eng.gn_setup("Burgers", [1.0, 0.02], np.zeros(N), zero_bdy)
    eng.dist_inverse()
    eng.gn_set_z(np.zeros(3 * N))
    eng.dist_gram_assemble("Eikonal", "Gaussian", 0.2)
    eng.dist_add_diag(_adaptive_nugget(eng.dist_get_diag(), N))
    assert eng.dist_potrf() == 0
    eng.dist_inverse()
    with pytest.raises(_lib.GppError, match="another PDE"):
        eng.dist_gn_step(1.0)
    # the relaxed elliptic method stays on one GPU
    eng.dist_gram_assemble("Nonlinear_elliptic", "Gaussian", 0.2)
    eng.dist_add_diag(np.full(2 * N + Nb, 1e-6))
    assert eng.dist_potrf() == 0
    eng.dist_inverse()
    eng.gn_setup("Nonlinear_elliptic_relaxed", [1.0, 3.0, 1e-6], np.zeros(N), zero_bdy)
    eng.gn_set_z(np.zeros(2 * N))
    with pytest.raises(_lib.GppError):
        eng.dist_gn_step(1.0)


def _torchrun(nproc, port, args, env=None):
    return subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={nproc}",
                           "--master-addr", "127.0.0.1", "--master-port", str(port), os.path.join(ROOT, "tools", "dist_solve.py"),
                           "--pde", "burgers"] + args, capture_output=True, text=True, timeout=600, env=env)


@pytest.mark.gpu
@pytest.mark.parametrize("p2p", ["0", "1"])
def test_sharded_burgers_two_gpus(p2p):
    """The real exchange paths on 2 GPUs: NCCL all-gather / broadcast (default) and peer stores over NVLink (GPP_DIST_P2P=1)."""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs >= 2 GPUs")
    out = _torchrun(2, 29621, ["--N", "1500", "--Nb", "150", "--NB", "256", "--reps", "1", "--check"],
                    env=dict(os.environ, GPP_DIST_P2P=p2p))
    assert out.returncode == 0, out.stdout[-2000:] + out.stderr[-2000:]
    assert '"ok": true' in out.stdout
    assert ('"exchange": "p2p"' if p2p == "1" else '"exchange": "nccl"') in out.stdout


@pytest.mark.gpu
def test_sharded_burgers_single_rank_nccl():
    """world = 1 through torchrun: communicator creation and the whole sharded Burgers call sequence."""
    out = _torchrun(1, 29622, ["--N", "1200", "--Nb", "120", "--NB", "256", "--reps", "1", "--check"])
    assert out.returncode == 0, out.stdout[-2000:] + out.stderr[-2000:]
    assert '"ok": true' in out.stdout
