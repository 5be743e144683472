"""Problem classes with the reference's names, constructor arguments, methods and attributes
(src/PDEs.py:18-505).  The Python side only holds points, data vectors and the loop; Theta, its
Cholesky factor, the interior block of Theta^{-1} and the GN iterate live on the GPU."""
import numpy as onp
from numpy import random

from . import _dist, _lib
from .sample_points import sampled_pts_rdm, sampled_pts_grid


def eval_on_points(fun, X):
    """vmap(fun)(X[:,0], X[:,1]) of the reference (src/PDEs.py:44-45) without JAX: try a vectorised call,
    fall back to a per-point loop for callables that only take scalars."""
    x1, x2 = X[:, 0], X[:, 1]
    n = X.shape[0]
    if n == 0:
        return onp.zeros(0)
    try:
        v = onp.asarray(fun(x1, x2), dtype=onp.float64)
    except (TypeError, ValueError):
        v = None
    if v is not None and v.shape == (n,):
        return v
    if v is not None and v.shape == ():
        # a 0-d result is either a constant function (bdy = lambda x1, x2: 0) or a callable that reduces over its
        # inputs; only the former may be broadcast, so check it against per-point scalar calls at both ends
        ends = [float(fun(float(x1[k]), float(x2[k]))) for k in (0, n - 1)]
        if ends[0] == float(v) and ends[1] == float(v):
            return onp.full(n, float(v))
    return onp.array([float(fun(float(a), float(b))) for a, b in zip(x1, x2)], dtype=onp.float64)


class _GPProblem(object):
    """Shared host logic of the three PDE classes."""
    _eqn = None            # eqn string of Gram_matrix_assembly
    _time_dependent = False
    _nz = 1                # number of unknown blocks

    def __init__(self, bdy=None, rhs=None, domain=onp.array([[0, 1], [0, 1]])):
        self.bdy = bdy
        self.rhs = rhs
        self.domain = domain
        self._eng = None
        self._sharded = False
        self.timings = {}

    # reference helpers
    def get_bd(self, x1, x2):
        return self.bdy(x1, x2)

    def get_rhs(self, x1, x2):
        return self.rhs(x1, x2)

    def _engine(self):
        if self._eng is None:
            self._eng = _lib.Engine()
        return self._eng

    # ---- multi-GPU: ONE solve sharded over the GPUs of the box (no counterpart in the reference) ----
    def shard(self, dist=None, virtual_ranks=None, Q=None):
        """Shard this problem over the ranks of an initialised ``torch.distributed`` group (one process per GPU; every
        rank must construct the same problem with the same points and make the same calls).  Gram assembly, Cholesky,
        the inverse and the GN Hessian are then owner-computes over a P x Q block-cyclic grid with NCCL panel gathers
        (csrc/dist.cu); all results (loss history, solution, predictions) are identical on every rank.
        ``virtual_ranks=n`` instead emulates n ranks on this one GPU (tests)."""
        if self._eqn not in ('Nonlinear_elliptic', 'Burgers'):
            raise NotImplementedError("the sharded path covers Nonlinear_elliptic2d and Burgers (not Eikonal, "
                                      "Darcy_flow2d or the relaxed method)")
        eng = self._engine()
        if virtual_ranks is not None:
            eng.dist_init_virtual(virtual_ranks)
            eng.dist_set_grid(*_dist.grid_shape(virtual_ranks, Q))
        else:
            _dist.init_engine_distributed(eng, dist, Q)
        self._sharded = True
        return self

    # ---- sampling (src/PDEs.py:34-54) ----
    def sampled_pts(self, N_domain, N_boundary, sampled_type='random'):
        if sampled_type == 'random':
            X_domain, X_boundary = sampled_pts_rdm(N_domain, N_boundary, self.domain, time_dependent=self._time_dependent)
        elif sampled_type == 'grid':
            X_domain, X_boundary = sampled_pts_grid(N_domain, N_boundary, self.domain, time_dependent=self._time_dependent)
        else:
            raise ValueError(f"unknown sampled_type {sampled_type!r}")
        self.get_sampled_points(X_domain, X_boundary)

    def get_sampled_points(self, X_domain, X_boundary):
        self.X_domain = onp.ascontiguousarray(X_domain, dtype=onp.float64)
        self.N_domain = self.X_domain.shape[0]
        self.X_boundary = onp.ascontiguousarray(X_boundary, dtype=onp.float64).reshape(-1, 2)
        self.N_boundary = self.X_boundary.shape[0]
        self.rhs_f = eval_on_points(self.get_rhs, self.X_domain)
        self.bdy_g = eval_on_points(self.get_bd, self.X_boundary)
        self._engine().set_points(self.X_domain, self.X_boundary)
        self._state = 'points'

    # ---- Gram matrix + nugget (src/PDEs.py:56-73, :250-269, :391-409) ----
    def _nugget_vector(self, diag, n_blocks, nugget, nugget_type):
        """nugget * r with r from the trace ratios of the diagonal blocks; traces are summed on the
        host with numpy from the device-computed diagonal, like the reference's jnp/onp.trace."""
        N, M = self.N_domain, diag.shape[0]
        if nugget_type == 'adaptive':
            tr = [onp.sum(diag[p * N:(p + 1) * N]) for p in range(n_blocks - 1)]
            tr_last = onp.sum(diag[(n_blocks - 1) * N:])
            ratio = [t / tr_last for t in tr]
            r = onp.ones(M)
            for p, rt in enumerate(ratio):
                r[p * N:(p + 1) * N] = rt
            return nugget * r, ratio
        if nugget_type == 'identity':
            return nugget * onp.ones(M), None
        if nugget_type == 'none':
            return None, None
        raise ValueError(f"unknown nugget_type {nugget_type!r}")

    def _gram(self, kernel, kernel_parameter, nugget, nugget_type):
        eng = self._engine()
        self.nugget_type, self.nugget = nugget_type, nugget
        self.kernel, self.kernel_parameter = kernel, kernel_parameter
        eng.timer_start()
        if self._sharded:
            eng.dist_gram_assemble(self._eqn, kernel, kernel_parameter)
        else:
            eng.gram_assemble(0, self._eqn, kernel, kernel_parameter)
        self.timings['assembly_ms'] = eng.timer_stop()
        n_blocks = {'Nonlinear_elliptic': 2}.get(self._eqn, 4)
        diag = eng.dist_get_diag() if self._sharded else eng.gram_get_diag(0)
        add, ratio = self._nugget_vector(diag, n_blocks, nugget, nugget_type)
        if ratio is not None:
            self.ratio = ratio[0] if len(ratio) == 1 else ratio
        if add is not None:
            if self._sharded:
                eng.dist_add_diag(add)
            else:
                eng.gram_add_diag(0, add)
        self._nugget_add = add
        self._state = 'gram'

    # Theta / L are lazy: dense download only when somebody asks (tests, small problems)
    @property
    def Theta(self):
        """The reference keeps ``self.Theta`` (src/PDEs.py:69); here the device copy is overwritten in place by its
        Cholesky factor, so after Gram_Cholesky() a read re-assembles it (same kernel, same nugget) on a scratch handle."""
        if self._state == 'gram' and not self._sharded:
            return self._engine().gram_download(0, 0)
        if self._state in ('gram', 'chol', 'solved'):
            return self._reassemble(self._eqn, self._nugget_add)
        raise RuntimeError("call Gram_matrix() first")

    def _reassemble(self, layout, add):
        eng = _lib.default_engine()
        eng.set_points(self.X_domain, self.X_boundary)
        eng.gram_assemble(0, layout, self.kernel, self.kernel_parameter)
        if add is not None:
            eng.gram_add_diag(0, add)
        return eng.gram_download(0, 0)

    @property
    def L(self):
        if self._state not in ('chol', 'solved'):
            raise RuntimeError("call Gram_Cholesky() first")
        return self._engine().gram_download(0, 1)

    def Gram_Cholesky(self):
        """jnp.linalg.cholesky(self.Theta) (src/PDEs.py:75-80).  Like JAX, failure does not raise: the
        factor carries NaNs and the loss turns NaN; the pivot index is kept in ``self.chol_info``."""
        if self._state in ('chol', 'solved'):
            return                                  # already factored (the reference would recompute the same L)
        eng = self._engine()
        eng.timer_start()
        self.chol_info = eng.dist_potrf() if self._sharded else eng.potrf(0)
        self.chol_schedule = 'right-looking, block summation (sharded)' if self._sharded else 'default'
        if self.chol_info > 0 and not self._sharded and eng.gram_size(0)[0] > 4608:
            # the fast left-looking schedule subtracts entry by entry; near the edge of FP64 (nugget ~1e-13, N_domain >= 20 000)
            # the right-looking schedule with block summation still factors (profiles/r02_nugget_*.jsonl): rebuild Theta, retry
            eng.gram_assemble(0, self._eqn, self.kernel, self.kernel_parameter)
            if self._nugget_add is not None:
                eng.gram_add_diag(0, self._nugget_add)
            eng.set_option("rl_potrf", 1)
            try:
                info = eng.potrf(0)
            finally:
                eng.set_option("rl_potrf", 0)
            if info == 0:
                self.chol_info, self.chol_schedule = 0, 'right-looking, block summation (retry after a failed pivot)'
        self.timings['potrf_ms'] = eng.timer_stop()
        self._inverted = False
        self._state = 'chol'

    def _quad(self, slot, r):
        """r^T Theta^{-1} r = |L^{-1} r|^2 of the reference's linearised losses, by two triangular solves."""
        r = onp.ascontiguousarray(r, dtype=onp.float64)
        return float(onp.dot(r, self._engine().solve_vec(slot, r)))

    # ---- loss / GN ----
    def _gn_params(self):
        raise NotImplementedError

    def _setup_gn(self):
        eng = self._engine()
        eng.gn_setup(self._eqn, self._gn_params(), self.rhs_f, self.bdy_g)

    def loss(self, z):
        eng = self._engine()
        self._setup_gn()
        eng.gn_set_z(z)
        return eng.gn_loss()

    def _at(self, z):
        eng = self._engine()
        self._setup_gn()
        self._ensure_inverse()
        eng.gn_set_z(z)
        return eng

    def _ensure_inverse(self):
        if self._sharded:
            raise NotImplementedError("dense grad_loss / Hessian_GN read-outs are not available on a sharded problem")
        if not getattr(self, '_inverted', False):
            self._engine().inverse(0)
            self._inverted = True

    def grad_loss(self, z):
        """grad(self.loss)(z)  (src/PDEs.py:90-91)."""
        return self._at(z).gn_grad_hess(True, False)[0]

    def Hessian_GN(self, z, z_old=None):
        """hessian(GN_loss)(z, z_old) (src/PDEs.py:101-102); it depends on z_old only (Burgers takes one argument)."""
        return self._at(z if z_old is None else z_old).gn_grad_hess(False, True)[1]

    def _initial_guess(self, initial_sol):
        n = self._nz * self.N_domain
        if isinstance(initial_sol, str):
            if initial_sol == 'rdm':
                return random.normal(0.0, 1.0, (n))
            if initial_sol == 'zero' and self._eqn == 'Eikonal':
                return onp.zeros(n)
            # the reference leaves `sol` undefined here and dies with a NameError
            raise ValueError(f"initial_sol {initial_sol!r} not supported for {self._eqn}")
        return onp.array(initial_sol, dtype=onp.float64).reshape(n)

    def GN_method(self, max_iter=3, step_size=1, initial_sol='rdm', print_hist=True):
        """src/PDEs.py:104-135 (and :309-343, :457-498).  Loop on the host, all arithmetic on the GPU;
        one scalar (the loss) is read back per iteration because the reference prints it."""
        eng = self._engine()
        sol = self._initial_guess(initial_sol)
        self.init_sol = sol
        self._setup_gn()
        eng.timer_start()
        if self._sharded:
            eng.dist_inverse()
        else:
            eng.inverse(0)
            self._inverted = True
        self.timings['inverse_ms'] = eng.timer_stop()
        eng.gn_set_z(sol)
        loss_hist = []
        eng.timer_start()
        loss_now = eng.gn_loss()
        loss_hist.append(loss_now)
        if onp.isnan(loss_now):
            print('[Error] Loss is nan: maybe nugget is too small!')
        if print_hist:
            print('iter = 0', 'Loss =', loss_now)
        gn_step = eng.dist_gn_step if self._sharded else eng.gn_step
        for iter_step in range(1, max_iter + 1):
            loss_now = gn_step(step_size)
            if onp.isnan(loss_now):
                print('[Error] Loss is nan: maybe nugget is too small!')
            loss_hist.append(loss_now)
            if print_hist:
                print('iter = ', iter_step, 'Gauss-Newton step size =', step_size, ' Loss = ', loss_now)
        self.timings['gn_ms'] = eng.timer_stop()
        self.max_iter = max_iter
        self.step_size = step_size
        self.loss_hist = loss_hist
        sol = eng.gn_get_z()
        self.sol = sol
        self.sol_vec = eng.gn_residual(0)
        self.sol_sampled_pts = sol[:self.N_domain]
        self._state = 'solved'

    # ---- optional checkpoint of a finished solve (the reference only has commented-out np.savez calls)
    _STATE_KEYS = ('X_domain', 'X_boundary', 'rhs_f', 'bdy_g', 'sol', 'sol_vec', 'sol_sampled_pts', 'loss_hist', 'init_sol')

    def save_solution(self, path):
        """np.savez of the points, data vectors, iterate, loss history and kernel / nugget settings."""
        onp.savez(path, kernel=str(self.kernel), kernel_parameter=onp.asarray(self.kernel_parameter, dtype=onp.float64),
                  nugget=float(self.nugget), nugget_type=str(self.nugget_type),
                  **{k: onp.asarray(getattr(self, k)) for k in self._STATE_KEYS if hasattr(self, k)})

    def extend_sol(self, X_test):
        """src/PDEs.py:203-208: Theta_test @ (L^T \\ (L \\ sol_vec)); Theta_test is never formed."""
        eng = self._engine()
        X_test = onp.ascontiguousarray(X_test, dtype=onp.float64)
        temp = eng.solve_vec(0, self.sol_vec)
        self.X_test = X_test
        self.N_test = X_test.shape[0]
        self.extended_sol = eng.predict(0, X_test, temp)


class Nonlinear_elliptic2d(_GPProblem):
    """-Delta u + alpha*u^m = f in a box (src/PDEs.py:18-208)."""
    _eqn, _nz = 'Nonlinear_elliptic', 1

    def __init__(self, alpha=1.0, m=3, bdy=None, rhs=None, domain=onp.array([[0, 1], [0, 1]])):
        super().__init__(bdy, rhs, domain)
        self.alpha = alpha
        self.m = m

    def _gn_params(self):
        return [float(self.alpha), float(self.m)]

    def Gram_matrix(self, kernel='Gaussian', kernel_parameter=0.2, nugget=1e-8, nugget_type='adaptive'):
        self._gram(kernel, kernel_parameter, nugget, nugget_type)

    def GN_loss(self, z, z_old):
        """src/PDEs.py:94-98 (the linearised loss whose Hessian is Hessian_GN)."""
        z, z_old = onp.asarray(z, dtype=onp.float64), onp.asarray(z_old, dtype=onp.float64)
        zz = onp.append(self.alpha * self.m * (z_old ** (self.m - 1)) * (z - z_old), z)
        return self._quad(0, onp.append(zz, self.bdy_g))

    def _relaxed_at(self, z, pen_lambda):
        eng = self._engine()
        eng.gn_setup('Nonlinear_elliptic_relaxed', [float(self.alpha), float(self.m), float(pen_lambda)], self.rhs_f, self.bdy_g)
        eng.gn_set_z(z)
        return eng

    def loss_relaxed(self, z, pen_lambda):
        return self._relaxed_at(z, pen_lambda).gn_loss()

    def grad_loss_relaxed(self, z, pen_lambda):
        """src/PDEs.py:150-152."""
        self._ensure_inverse()
        return self._relaxed_at(z, pen_lambda).gn_grad_hess(True, False)[0]

    def GN_loss_relaxed(self, z, z_old, pen_lambda):
        """src/PDEs.py:155-165."""
        N = self.N_domain
        z, z_old = onp.asarray(z, dtype=onp.float64), onp.asarray(z_old, dtype=onp.float64)
        v, w, w_old = z[:N], z[N:], z_old[N:]
        ss2 = -v + self.alpha * self.m * (w_old ** (self.m - 1)) * (w - w_old) - self.rhs_f
        return self._quad(0, onp.append(onp.append(v, w), self.bdy_g)) + float(onp.dot(ss2, ss2)) / pen_lambda

    def Hessian_GN_relaxed(self, z, z_old, pen_lambda):
        """src/PDEs.py:168-169; depends on z_old only."""
        self._ensure_inverse()
        return self._relaxed_at(z_old, pen_lambda).gn_grad_hess(False, True)[1]

    def GN_relaxed_method(self, max_iter=3, step_size=1, initial_sol='rdm', pen_lambda=1e-10, print_hist=True):
        """src/PDEs.py:171-201: unknowns z = [v; w] (2N), penalised constraint -v + alpha w^m = f.
        H = 2 E^T Theta^{-1} E + (2/lambda) B^T B uses the same interior inverse block as the elimination path."""
        print(f'Relaxed approach: penalization parameter = {pen_lambda}')
        eng = self._engine()
        N = self.N_domain
        if isinstance(initial_sol, str):
            if initial_sol != 'rdm':
                raise ValueError(f"initial_sol {initial_sol!r} not supported")
            sol = random.normal(0.0, 1.0, (2 * N))
        else:
            sol = onp.array(initial_sol, dtype=onp.float64).reshape(2 * N)
        self.init_sol = sol
        eng.gn_setup('Nonlinear_elliptic_relaxed', [float(self.alpha), float(self.m), float(pen_lambda)], self.rhs_f, self.bdy_g)
        eng.timer_start()
        eng.inverse(0)
        self.timings['inverse_ms'] = eng.timer_stop()
        eng.gn_set_z(sol)
        eng.timer_start()
        loss_now = eng.gn_loss()
        loss_hist = [loss_now]
        if onp.isnan(loss_now):
            print('[Error] Loss is nan: maybe nugget is too small!')
        if print_hist:
            print('iter = 0', 'Loss =', loss_now)
        for iter_step in range(1, max_iter + 1):
            loss_now = eng.gn_step(step_size)
            if onp.isnan(loss_now):
                print('[Error] Loss is nan: maybe nugget is too small!')
            loss_hist.append(loss_now)
            if print_hist:
                print('iter = ', iter_step, 'Gauss-Newton step size =', step_size, ' Loss = ', loss_now)
        self.timings['gn_ms'] = eng.timer_stop()
        self.max_iter, self.step_size, self.loss_hist = max_iter, step_size, loss_hist
        sol = eng.gn_get_z()
        self.sol = sol
        self.sol_vec = onp.append(sol, self.bdy_g)        # :199
        self.sol_sampled_pts = sol[N:]                    # :201
        self._inverted = True
        self._state = 'solved'


class Burgers(_GPProblem):
    """u_t + alpha u u_x - nu u_xx = 0, (t, x) in [0,1] x [-1,1] (src/PDEs.py:211-350)."""
    _eqn, _nz, _time_dependent = 'Burgers', 3, True

    def __init__(self, alpha=1.0, nu=0.2, bdy=None, rhs=None, domain=onp.array([[0, 1], [-1, 1]])):
        super().__init__(bdy, rhs, domain)
        self.alpha = alpha
        self.nu = nu

    def _gn_params(self):
        return [float(self.alpha), float(self.nu)]

    def Gram_matrix(self, kernel='anisotropic_Gaussian', kernel_parameter=[1 / 3, 1 / 20], nugget=1e-5, nugget_type='adaptive'):
        self._gram(kernel, kernel_parameter, nugget, nugget_type)

    def GN_method(self, max_iter=10, step_size=1, initial_sol='rdm', print_hist=True):
        super().GN_method(max_iter, step_size, initial_sol, print_hist)


class Eikonal(_GPProblem):
    """|grad u|^2 = f^2 + eps Delta u (src/PDEs.py:352-505)."""
    _eqn, _nz = 'Eikonal', 3

    def __init__(self, eps=3, bdy=None, rhs=None, domain=onp.array([[0, 1], [0, 1]])):
        super().__init__(bdy, rhs, domain)
        self.eps = eps

    def _gn_params(self):
        return [float(self.eps)]

    def GN_loss(self, z, z_old):
        """src/PDEs.py:437-451."""
        N = self.N_domain
        z, z_old = onp.asarray(z, dtype=onp.float64), onp.asarray(z_old, dtype=onp.float64)
        v1_old, v2_old = z_old[N:2 * N], z_old[2 * N:]
        v0, v1, v2 = z[:N], z[N:2 * N], z[2 * N:]
        v3 = -(self.rhs_f ** 2 - 2 * v1 * v1_old - 2 * v2 * v2_old) / self.eps
        return self._quad(0, onp.concatenate((v1, v2, v3, v0, self.bdy_g)))

    def Gram_matrix(self, kernel='Gaussian', kernel_parameter=0.2, nugget=1e-8, nugget_type='adaptive'):
        self._gram(kernel, kernel_parameter, nugget, nugget_type)
