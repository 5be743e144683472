"""Darcy-flow inverse problem with the reference's interface (src/InverseProblems.py:16-196)."""
import numpy as onp
from numpy import random

from .PDEs import _GPProblem, eval_on_points
from .sample_points import sampled_pts_rdm, sampled_pts_grid


class Darcy_flow2d(_GPProblem):
    """-div(a grad u) = f, infer a from f and noisy observations of u.  Unknowns z = [w0 = log a; w1; w2;
    v0 = u; v1; v2] (6N); two Gram systems: slot 0 = Theta_u, slot 1 = Theta_a."""
    _eqn, _nz = 'Darcy_flow2d', 6

    def __init__(self, bdy=None, rhs=None, domain=onp.array([[0, 1], [0, 1]])):
        super().__init__(bdy, rhs, domain)

    # src/InverseProblems.py:32-47: the first N_data interior points carry the observations
    def sampled_pts(self, N_domain, N_boundary, N_data, sampled_type='random'):
        if sampled_type == 'random':
            X_domain, X_boundary = sampled_pts_rdm(N_domain, N_boundary, self.domain, time_dependent=False)
        elif sampled_type == 'grid':
            X_domain, X_boundary = sampled_pts_grid(N_domain, N_boundary, self.domain, time_dependent=False)
        else:
            raise ValueError(f"unknown sampled_type {sampled_type!r}")
        self.get_sampled_points(X_domain, X_boundary, X_domain[0:N_data, :])

    def get_sampled_points(self, X_domain, X_boundary, X_data):
        super().get_sampled_points(X_domain, X_boundary)
        self.X_data = onp.asarray(X_data)
        self.N_data = self.X_data.shape[0]

    def get_observation(self, data_u, noise_level):
        # src/InverseProblems.py:62-64 (the noise draw is part of the reference's RNG call order)
        self.data_u = data_u + noise_level * random.normal(0, 1.0, onp.shape(data_u)[0])
        self.noise_level = noise_level

    def Gram_matrix(self, kernel='Gaussian', kernel_parameter=0.2, nugget=1e-10, nugget_type='adaptive'):
        """src/InverseProblems.py:66-99: Theta_u (4N+Nb) and Theta_a (3N), separate trace ratios."""
        eng = self._engine()
        self.nugget_type, self.nugget = nugget_type, nugget
        self.kernel, self.kernel_parameter = kernel, kernel_parameter
        eng.timer_start()
        eng.gram_assemble(0, 'Darcy_flow2d', kernel, kernel_parameter)
        eng.gram_assemble(1, 'Darcy_flow2d_a', kernel, kernel_parameter)
        self.timings['assembly_ms'] = eng.timer_stop()
        add_u, self.ratio_u = self._nugget_vector(eng.gram_get_diag(0), 4, nugget, nugget_type)
        add_a, self.ratio_a = self._nugget_vector(eng.gram_get_diag(1), 3, nugget, nugget_type)
        if add_u is not None:
            eng.gram_add_diag(0, add_u)
            eng.gram_add_diag(1, add_a)
        self._nugget_add = (add_u, add_a)
        self._state = 'gram'

    @property
    def Theta_u(self):
        if self._state in ('chol', 'solved'):       # overwritten by L_u on the device: re-assemble on request
            return self._reassemble('Darcy_flow2d', self._nugget_add[0])
        return self._dense(0, 0, ('gram',))

    @property
    def Theta_a(self):
        if self._state in ('chol', 'solved'):
            return self._reassemble('Darcy_flow2d_a', self._nugget_add[1])
        return self._dense(1, 0, ('gram',))

    Theta = Theta_u

    @property
    def L_u(self):
        return self._dense(0, 1, ('chol', 'solved'))

    @property
    def L_a(self):
        return self._dense(1, 1, ('chol', 'solved'))

    def _dense(self, slot, what, states):
        if self._state not in states:
            raise RuntimeError("matrix not available in this state (Theta is overwritten by its Cholesky factor)")
        return self._engine().gram_download(slot, what)

    def Gram_Cholesky(self):
        if self._state in ('chol', 'solved'):
            return
        eng = self._engine()
        eng.timer_start()
        self.chol_info = (eng.potrf(0), eng.potrf(1))
        self.timings['potrf_ms'] = eng.timer_stop()
        self._inverted = False
        self._state = 'chol'

    def _setup_gn(self):
        self._engine().gn_setup('Darcy_flow2d', [], self.rhs_f, self.bdy_g, self.data_u, self.noise_level)

    def _ensure_inverse(self):
        if not getattr(self, '_inverted', False):
            self._engine().inverse(0)
            self._engine().inverse(1)
            self._inverted = True

    def GN_loss(self, z, z_old):
        """src/InverseProblems.py:127-147."""
        N = self.N_domain
        z, zo = onp.asarray(z, dtype=onp.float64), onp.asarray(z_old, dtype=onp.float64)
        w0_old, w1_old, w2_old, v1_old, v2_old = zo[:N], zo[N:2 * N], zo[2 * N:3 * N], zo[4 * N:5 * N], zo[5 * N:6 * N]
        w0, w1, w2, v0, v1, v2 = (z[k * N:(k + 1) * N] for k in range(6))
        v3 = (-self.rhs_f) * (-onp.exp(-w0_old)) * w0 + (-v1_old) * w1 + (-v2_old) * w2 + (-w1_old) * v1 + (-w2_old) * v2
        w_all = onp.concatenate((w1, w2, w0), axis=0)
        v_all = onp.concatenate((v1, v2, v3, v0, self.bdy_g), axis=0)
        return (self._quad(1, w_all) + self._quad(0, v_all)
                + (1 / self.noise_level ** 2) * float(onp.sum((v0[:self.N_data] - self.data_u) ** 2)))

    def GN_method(self, max_iter=3, step_size=1, initial_sol='rdm', print_hist=True):
        """src/InverseProblems.py:153-186."""
        eng = self._engine()
        N = self.N_domain
        sol = self._initial_guess(initial_sol)
        self.init_sol = sol
        self._setup_gn()
        eng.timer_start()
        eng.inverse(0)
        eng.inverse(1)
        self.timings['inverse_ms'] = eng.timer_stop()
        self._inverted = True
        eng.gn_set_z(sol)
        eng.timer_start()
        loss_now = eng.gn_loss()
        loss_hist = [loss_now]
        if print_hist:
            print('iter = 0', 'Loss =', loss_now)
        for iter_step in range(1, max_iter + 1):
            loss_now = eng.gn_step(step_size)
            loss_hist.append(loss_now)
            if print_hist:
                print('iter = ', iter_step, 'Gauss-Newton step size =', step_size, ' Loss = ', loss_now)
        self.timings['gn_ms'] = eng.timer_stop()
        self.max_iter, self.step_size, self.loss_hist = max_iter, step_size, loss_hist
        sol = eng.gn_get_z()
        self.sol = sol
        self.sol_vec_a = onp.append(sol[N:3 * N], sol[:N])      # [w1; w2; w0]   (:176-177)
        self.sol_vec_u = eng.gn_residual(0)                     # [v1; v2; v3; v0; g] (:179-186)
        self.sol_sampled_pts = sol[3 * N:4 * N]
        self._state = 'solved'

    def extend_sol(self, X_test):
        """src/InverseProblems.py:188-196."""
        eng = self._engine()
        X_test = onp.ascontiguousarray(X_test, dtype=onp.float64)
        self.X_test, self.N_test = X_test, X_test.shape[0]
        self.extended_sol_a = eng.predict(1, X_test, eng.solve_vec(1, self.sol_vec_a))
        self.extended_sol_u = eng.predict(0, X_test, eng.solve_vec(0, self.sol_vec_u))

    def extend_sol_var(self, X_test):
        """Posterior variances at the test points of the two fields extend_sol predicts (see _GPProblem.extend_sol_var):
        extended_var_u from Theta_u (slot 0), extended_var_a from Theta_a (slot 1, the field of extended_sol_a)."""
        self._check_factored()
        eng = self._engine()
        X_test = onp.ascontiguousarray(X_test, dtype=onp.float64)
        self.extended_var_u = eng.predict_var(0, X_test)
        self.extended_var_a = eng.predict_var(1, X_test)
