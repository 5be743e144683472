"""``solver_GP``: the facade users of the reference drive (interface of src/solver.py:41-206).

Same constructor, method names, keyword arguments, attributes and console messages as upstream; the body is
table-driven here.  Deliberate differences: matplotlib is imported lazily by the plotting methods only; the
upstream bug of ``get_sample`` / ``get_sample_IP`` (``self`` passed twice, src/solver.py:86,110) is not
reproduced; error metrics are plain numpy."""
import numpy as onp

from .InverseProblems import Darcy_flow2d
from .PDEs import Burgers, Eikonal, Nonlinear_elliptic2d


def _box(domain):
    return f'[Equation domain] [{domain[0,0]},{domain[0,1]}]*[{domain[1,0]},{domain[1,1]}]'


_DATA_LINE = '[Equation data] Right hand side and boundary values set by the user'

# PDE_type -> (factory(cfg, bdy, rhs, domain), banner(cfg, domain) -> list of console lines)
_EQUATIONS = {
    "Nonlinear_elliptic": (
        lambda cfg, bdy, rhs, dom: Nonlinear_elliptic2d(alpha=cfg.alpha, m=cfg.m, bdy=bdy, rhs=rhs, domain=dom),
        lambda cfg, dom: ['[Equation type] Nonlinear elliptic equation', '[Equation form] - \\Delta u + alpha*u^m = f', _box(dom),
                          f'[Equation parameter] alpha = {cfg.alpha}, m = {cfg.m}', _DATA_LINE]),
    "Burgers": (
        lambda cfg, bdy, rhs, dom: Burgers(alpha=cfg.alpha, nu=cfg.nu, bdy=bdy, rhs=rhs, domain=dom),
        lambda cfg, dom: ['[Equation type] Burgers equation', '[Equation form] u_t+ alpha u u_x- nu u_xx=0', _box(dom),
                          f'[Equation parameter] alpha = {cfg.alpha}, m = {cfg.nu}', _DATA_LINE]),   # "m =" as printed upstream
    "Eikonal": (
        lambda cfg, bdy, rhs, dom: Eikonal(eps=cfg.eps, bdy=bdy, rhs=rhs, domain=dom),
        lambda cfg, dom: ['[Equation type] Eikonal equation', '[Equation form] |grad u|^2 = f + eps*Delta u', _box(dom),
                          f'[Equation parameter] eps = {cfg.eps}', _DATA_LINE]),
    "Darcy_flow2d": (
        lambda cfg, bdy, rhs, dom: Darcy_flow2d(bdy=bdy, rhs=rhs, domain=dom),
        lambda cfg, dom: ['[Inverse problem type] Darcy flow 2d',
                          '[Inverse problem form] -div(a grad u) = f, infer a from f and some observed u', _box(dom), _DATA_LINE]),
}


def _say(enabled, *lines):
    if enabled:
        for line in lines:
            print(line)


def _pyplot():
    try:
        import matplotlib.pyplot as plt
    except Exception as exc:  # pragma: no cover
        raise RuntimeError("plotting needs matplotlib, which is not installed in this environment") from exc
    return plt


class solver_GP(object):
    def __init__(self, cfg=None, PDE_type="Nonlinear_elliptic"):
        self.config = cfg
        self.PDE_type = PDE_type

    # ------------------------------------------------------------------ problem definition
    def set_equation(self, bdy=None, rhs=None, domain=onp.array([[0, 1], [0, 1]]), print_option=True):
        if self.PDE_type not in _EQUATIONS:
            raise ValueError(f"unknown PDE_type {self.PDE_type!r}")
        make, banner = _EQUATIONS[self.PDE_type]
        self.eqn = make(self.config, bdy, rhs, domain)
        _say(print_option, '\n Solver started', *banner(self.config, domain))

    def _report_sample(self, enabled, how, with_data):
        e = self.eqn
        counts = f'[Sample points] N_domain = {e.N_domain}, N_boundary = {e.N_boundary}'
        if with_data:
            counts += f', N_data = {e.N_data}'
        _say(enabled, f'[Sample points] Collocation points sampled, {how}', counts)

    def get_sample(self, X_domain, X_boundary, print_option=True):
        self.eqn.get_sampled_points(X_domain, X_boundary)
        self._report_sample(print_option, 'specified by the user', False)

    def auto_sample(self, N_domain, N_boundary, sampled_type='random', print_option=True):
        self.eqn.sampled_pts(N_domain, N_boundary, sampled_type=sampled_type)
        self._report_sample(print_option, f'type {sampled_type}', False)

    def get_sample_IP(self, X_domain, X_boundary, X_data, print_option=True):
        self.eqn.get_sampled_points(X_domain, X_boundary, X_data)
        self._report_sample(print_option, 'specified by the user', True)

    def auto_sample_IP(self, N_domain, N_boundary, N_data, sampled_type='random', print_option=True):
        self.eqn.sampled_pts(N_domain, N_boundary, N_data, sampled_type=sampled_type)
        self._report_sample(print_option, f'type {sampled_type}', True)

    def get_observed_data(self, data_u, noise_level, print_option=True):
        self.eqn.get_observation(data_u, noise_level)
        _say(print_option, '[Observed Data] Get observed data from solving the PDE using FD and interpolation',
             f'[Observed Data] Noise level {noise_level}')

    # ------------------------------------------------------------------ the hot path
    def solve(self, method='elimination', pen_lambda=1e-10, print_option=True):
        """Gram assembly -> Cholesky -> Gauss-Newton (src/solver.py:139-160), all on the GPU."""
        cfg, eqn = self.config, self.eqn
        _say(print_option, '[Kernel] ' + cfg.kernel, f'[Kernel parameter]: {cfg.kernel_parameter}')
        eqn.Gram_matrix(kernel=cfg.kernel, kernel_parameter=cfg.kernel_parameter, nugget=cfg.nugget, nugget_type=cfg.nugget_type)
        _say(print_option, f'[Gram matrix] Finish assembly of the Gram matrix, nugget {cfg.nugget}, type {cfg.nugget_type}')
        eqn.Gram_Cholesky()
        _say(print_option, '[Gram matrix] Finish Cholesky factorization of the Gram matrix',
             '[Gauss Newton] Start Gauss Newton iteration', f'[Gauss Newton] {method} approaches')
        loop = dict(max_iter=cfg.GNsteps, step_size=cfg.step_size, initial_sol=cfg.initial_sol, print_hist=cfg.print_hist)
        if method == 'elimination':
            eqn.GN_method(**loop)
        elif method == 'relaxation':
            eqn.GN_relaxed_method(pen_lambda=pen_lambda, **loop)
        _say(print_option, '[Gauss Newton] Gauss Newton iteration finished')

    # ------------------------------------------------------------------ errors
    @staticmethod
    def _abs_max_rms(truth, approx, count):
        err = abs(truth - approx)
        return err, onp.max(err), onp.sqrt(onp.sum(err ** 2) / count)

    def collocation_pts_err(self, truth, print_option=True):
        _say(print_option, '[Calculating collocation errors...]')
        self.pts_err_all, self.pts_max_err, self.pts_L2_err = self._abs_max_rms(truth, self.eqn.sol_sampled_pts, self.eqn.N_domain)
        _say(print_option, f'[Collocation point error] Max error {self.pts_max_err}', f'[Collocation point error] L2 error {self.pts_L2_err}')

    def test(self, X_test, print_option=True):
        _say(print_option, f'[Testing...] Number of test points: {X_test.shape[0]}')
        self.eqn.extend_sol(X_test)

    @staticmethod
    def _max_std(var):
        return onp.sqrt(onp.max(onp.maximum(var, 0.0)))

    def test_var(self, X_test, print_option=True):
        """Posterior variance at the test points (extend_sol_var): test_var_all, and for Darcy_flow2d test_var_all = the
        variance of u and test_var_all_a = that of a."""
        self.eqn.extend_sol_var(X_test)
        if hasattr(self.eqn, 'extended_var_u'):
            self.test_var_all, self.test_var_all_a = self.eqn.extended_var_u, self.eqn.extended_var_a
            _say(print_option, f'[Test variance] Max posterior standard deviation of u {self._max_std(self.test_var_all)}',
                 f'[Test variance] Max posterior standard deviation of a {self._max_std(self.test_var_all_a)}')
        else:
            self.test_var_all = self.eqn.extended_var
            _say(print_option, f'[Test variance] Max posterior standard deviation {self._max_std(self.test_var_all)}')

    def get_test_error(self, truth, print_option=True):
        self.truth = truth
        self.test_err_all, self.test_max_err, self.test_L2_err = self._abs_max_rms(truth, self.eqn.extended_sol, self.eqn.N_test)
        _say(print_option, f'[Test error] Max error {self.test_max_err}', f'[Test error] L2 error {self.test_L2_err}')

    # ------------------------------------------------------------------ optional plots (need matplotlib)
    def _scatter(self, title, groups, marker=None):
        plt = _pyplot()
        ax = plt.figure().add_subplot(111)
        for pts, label in groups:
            ax.scatter(pts[:, 0], pts[:, 1], marker=marker, label=label).set_clip_on(False)
        ax.legend(loc="upper right")
        plt.title(title)

    def show_sample(self):
        self._scatter('Collocation points', [(self.eqn.X_domain, 'Interior nodes'), (self.eqn.X_boundary, 'Boundary nodes')], marker="x")

    def show_sample_IP(self):
        e = self.eqn
        self._scatter('Collocation and data points',
                      [(e.X_domain, 'Interior nodes'), (e.X_boundary, 'Boundary nodes'), (e.X_domain[:e.N_data], 'Data nodes')])

    def show_loss_hist(self):
        plt = _pyplot()
        plt.figure()
        plt.plot(onp.arange(self.eqn.max_iter + 1), self.eqn.loss_hist)
        plt.yscale("log")
        plt.title('Loss function history')
        plt.xlabel('Gauss-Newton step')

    def contour_of_test_err(self, XX, YY):
        plt = _pyplot()
        fig = plt.figure()
        filled = fig.add_subplot(111).contourf(XX, YY, self.test_err_all.reshape(XX.shape), 50, cmap=plt.cm.coolwarm)
        self.XX, self.YY = XX, YY
        plt.xlabel('$x_1$')
        plt.ylabel('$x_2$')
        plt.title('Contour of errors')
        fig.colorbar(filled)
        plt.show()
