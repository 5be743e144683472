"""ctypes binding of libgpp_b200.so (C ABI: include/gpp.h).  Plumbing only: argument checking, numpy
buffers in / out.  There is deliberately no fallback: if the library is missing, or there is no
sm_100 GPU, the first call raises."""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libgpp_b200.so")

LAYOUT = {"Nonlinear_elliptic": 0, "Burgers": 1, "Eikonal": 2, "Darcy_flow2d": 2, "Darcy_flow2d_a": 3}
KERNEL = {"Gaussian": 0, "anisotropic_Gaussian": 1}
PDE = {"Nonlinear_elliptic": 0, "Burgers": 1, "Eikonal": 2, "Darcy_flow2d": 3, "Nonlinear_elliptic_relaxed": 4}

_lib = None
_dp = C.POINTER(C.c_double)
_ip = C.POINTER(C.c_int)


class GppError(RuntimeError):
    pass


def _sig(lib):
    H = C.c_void_p
    sigs = {
        "gpp_create": [C.c_int, C.POINTER(H)],
        "gpp_destroy": [H],
        "gpp_set_option": [H, C.c_char_p, C.c_double],
        "gpp_sync": [H],
        "gpp_timer_start": [H],
        "gpp_timer_stop": [H, C.POINTER(C.c_float)],
        "gpp_timer2_start": [H],
        "gpp_timer2_stop": [H, C.POINTER(C.c_float)],
        "gpp_set_points": [H, _dp, C.c_int, _dp, C.c_int],
        "gpp_gram_assemble": [H, C.c_int, C.c_int, C.c_int, _dp],
        "gpp_gram_size": [H, C.c_int, _ip, _ip],
        "gpp_gram_get_diag": [H, C.c_int, _dp],
        "gpp_gram_add_diag": [H, C.c_int, _dp],
        "gpp_gram_download": [H, C.c_int, C.c_int, _dp],
        "gpp_gram_upload": [H, C.c_int, _dp],
        "gpp_potrf": [H, C.c_int, _ip],
        "gpp_inverse": [H, C.c_int],
        "gpp_solve_vec": [H, C.c_int, _dp, _dp],
        "gpp_gn_setup": [H, C.c_int, _dp, _dp, _dp, _dp, C.c_int, C.c_double],
        "gpp_gn_set_z": [H, _dp],
        "gpp_gn_get_z": [H, _dp],
        "gpp_gn_loss": [H, _dp],
        "gpp_gn_step": [H, C.c_double, _dp],
        "gpp_gn_residual": [H, C.c_int, _dp],
        "gpp_gn_grad_hess": [H, _dp, _dp],
        "gpp_gn_coef": [H, C.c_int, C.c_int, C.c_int, _dp, _ip],
        "gpp_predict": [H, C.c_int, _dp, C.c_int, _dp, _dp],
        "gpp_theta_test": [H, C.c_int, _dp, C.c_int, _dp],
        "gpp_predict_var": [H, C.c_int, _dp, C.c_int, _dp],
        "gpp_kernel_eval": [H, C.c_int, _dp, C.c_int, C.c_int, _dp, _dp, _dp, _dp, C.c_long, _dp],
        "gpp_dist_unique_id": [C.POINTER(C.c_ubyte)],
        "gpp_dist_init": [H, C.c_int, C.c_int, C.POINTER(C.c_ubyte)],
        "gpp_dist_init_virtual": [H, C.c_int],
        "gpp_dist_set_grid": [H, C.c_int, C.c_int],
        "gpp_dist_info": [H, _ip, _ip, _ip, _ip],
        "gpp_dist_exchange_mode": [H],
        "gpp_dist_plan_check": [C.c_int] * 6,
        "gpp_dist_hess_plan_check": [C.c_int] * 6,
        "gpp_dist_finalize": [H],
        "gpp_dist_gram_assemble": [H, C.c_int, C.c_int, _dp],
        "gpp_dist_get_diag": [H, _dp],
        "gpp_dist_add_diag": [H, _dp],
        "gpp_dist_potrf": [H, _ip],
        "gpp_dist_inverse": [H],
        "gpp_dist_gn_step": [H, C.c_double, _dp],
        "gpp_dist_predict_var": [H, _dp, C.c_int, _dp],
    }
    for name, args in sigs.items():
        fn = getattr(lib, name)
        fn.argtypes = args
        fn.restype = C.c_int
    lib.gpp_last_error.argtypes = [H]
    lib.gpp_last_error.restype = C.c_char_p
    lib.gpp_launch_count.argtypes = [H]
    lib.gpp_launch_count.restype = C.c_long


def load():
    """Load the CUDA library.  Raises (never falls back) when it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise GppError(f"{LIB_PATH} not built: run `python __graft_entry__.py` (or nonlinpdes-gpsolver_b200/build.py)")
        lib = C.CDLL(LIB_PATH)
        _sig(lib)
        _lib = lib
    return _lib


def _f64(a, shape=None):
    a = np.ascontiguousarray(np.asarray(a, dtype=np.float64))
    if shape is not None and a.shape != tuple(shape):
        raise ValueError(f"expected shape {shape}, got {a.shape}")
    return a


def _test_points(X_test):
    Xt = _f64(X_test)
    if Xt.ndim != 2 or Xt.shape[1] != 2 or Xt.shape[0] == 0:
        raise ValueError(f"X_test must be (N_test, 2) with N_test >= 1, got {Xt.shape}")
    return Xt


def _ptr(a):
    return a.ctypes.data_as(_dp) if a is not None else None


def kernel_params(kernel, kernel_parameter):
    """{b1, b2, e1, e2} of include/gpp.h from the reference's (kernel, kernel_parameter) pair,
    evaluated with the same Python expressions as src/kernels.py:13 and :96-99."""
    if kernel == "Gaussian":
        s = float(kernel_parameter)
        a = 1.0 / (s * s)
        return np.array([a, a, -(1 / (2 * s ** 2)), 0.0])
    if kernel == "anisotropic_Gaussian":
        st, sx = float(kernel_parameter[0]), float(kernel_parameter[1])
        return np.array([2.0 / (st * st), 2.0 / (sx * sx), st, sx])
    raise ValueError(f"unknown kernel {kernel!r}")


class Engine:
    """One handle = one GPU.  Thin, typed wrapper over the C ABI."""

    def __init__(self, device=None):
        lib = load()
        if device is None:
            device = int(os.environ.get("LOCAL_RANK", "0"))
        h = C.c_void_p()
        rc = lib.gpp_create(int(device), C.byref(h))
        if rc != 0:
            raise GppError(f"gpp_create(device={device}) failed with code {rc}: no usable sm_100 GPU "
                           "(this package has no CPU fallback)")
        self._lib, self._h, self.device = lib, h, int(device)
        nb = os.environ.get("GPP_NB")
        if nb:
            self.set_option("NB", float(nb))
        gt = os.environ.get("GPP_GEMM_TILE")
        if gt:
            self.set_option("gemm_tile", float(gt))
        la = os.environ.get("GPP_LOOKAHEAD")
        if la is not None:
            self.set_option("lookahead", float(la))
        for env, opt in (("GPP_BLOCKSUM", "blocksum"), ("GPP_RL_POTRF", "rl_potrf"), ("GPP_TILED_POTRF", "tiled_potrf"),
                         ("GPP_PERSISTENT_GEMM", "persistent_gemm")):
            v = os.environ.get(env)
            if v is not None:
                self.set_option(opt, float(v))

    def close(self):
        if getattr(self, "_h", None):
            self._lib.gpp_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _ck(self, rc, what):
        if rc != 0:
            msg = self._lib.gpp_last_error(self._h)
            raise GppError(f"{what} failed (code {rc}): {msg.decode() if msg else ''}")

    # ---- misc
    def set_option(self, name, value):
        self._ck(self._lib.gpp_set_option(self._h, name.encode(), float(value)), "gpp_set_option")

    def sync(self):
        self._ck(self._lib.gpp_sync(self._h), "gpp_sync")

    def launch_count(self):
        return int(self._lib.gpp_launch_count(self._h))

    def timer_start(self):
        self._ck(self._lib.gpp_timer_start(self._h), "gpp_timer_start")

    def timer_stop(self):
        ms = C.c_float()
        self._ck(self._lib.gpp_timer_stop(self._h, C.byref(ms)), "gpp_timer_stop")
        return float(ms.value)

    def timer2_start(self):
        self._ck(self._lib.gpp_timer2_start(self._h), "gpp_timer2_start")

    def timer2_stop(self):
        ms = C.c_float()
        self._ck(self._lib.gpp_timer2_stop(self._h, C.byref(ms)), "gpp_timer2_stop")
        return float(ms.value)

    # ---- points / Gram
    def set_points(self, X_domain, X_boundary):
        Xd = _f64(X_domain)
        Xb = _f64(X_boundary).reshape(-1, 2)
        if Xd.ndim != 2 or Xd.shape[1] != 2:
            raise ValueError("X_domain must be (N, 2)")
        self.N, self.Nb = Xd.shape[0], Xb.shape[0]
        self._ck(self._lib.gpp_set_points(self._h, _ptr(Xd), self.N, _ptr(Xb) if self.Nb else None, self.Nb),
                 "gpp_set_points")

    def gram_assemble(self, slot, layout, kernel, kernel_parameter):
        kp = kernel_params(kernel, kernel_parameter)
        self._ck(self._lib.gpp_gram_assemble(self._h, slot, LAYOUT[layout], KERNEL[kernel], _ptr(kp)), "gpp_gram_assemble")

    def gram_size(self, slot):
        M, Mi = C.c_int(), C.c_int()
        self._ck(self._lib.gpp_gram_size(self._h, slot, C.byref(M), C.byref(Mi)), "gpp_gram_size")
        return M.value, Mi.value

    def gram_get_diag(self, slot):
        M, _ = self.gram_size(slot)
        out = np.empty(M)
        self._ck(self._lib.gpp_gram_get_diag(self._h, slot, _ptr(out)), "gpp_gram_get_diag")
        return out

    def gram_add_diag(self, slot, add):
        M, _ = self.gram_size(slot)
        add = _f64(add, (M,))
        self._ck(self._lib.gpp_gram_add_diag(self._h, slot, _ptr(add)), "gpp_gram_add_diag")

    def gram_download(self, slot, what):
        M, Mi = self.gram_size(slot)
        n = Mi if what == 2 else M
        out = np.empty((n, n))
        self._ck(self._lib.gpp_gram_download(self._h, slot, what, _ptr(out)), "gpp_gram_download")
        return out

    def gram_upload(self, slot, theta):
        M, _ = self.gram_size(slot)
        theta = _f64(theta, (M, M))
        self._ck(self._lib.gpp_gram_upload(self._h, slot, _ptr(theta)), "gpp_gram_upload")

    def potrf(self, slot):
        info = C.c_int()
        self._ck(self._lib.gpp_potrf(self._h, slot, C.byref(info)), "gpp_potrf")
        return info.value

    def inverse(self, slot):
        self._ck(self._lib.gpp_inverse(self._h, slot), "gpp_inverse")

    def solve_vec(self, slot, b):
        M, _ = self.gram_size(slot)
        b = _f64(b, (M,))
        x = np.empty(M)
        self._ck(self._lib.gpp_solve_vec(self._h, slot, _ptr(b), _ptr(x)), "gpp_solve_vec")
        return x

    # ---- Gauss-Newton
    def gn_setup(self, pde, params, rhs_f, bdy_g, data_u=None, noise=1.0):
        params = _f64(list(params) + [0.0] * (4 - len(params)))
        rhs_f = _f64(rhs_f, (self.N,))
        bdy_g = _f64(bdy_g, (self.Nb,))
        nd = 0
        if data_u is not None:
            data_u = _f64(data_u)
            nd = data_u.shape[0]
        self.nz = {0: 1, 1: 3, 2: 3, 3: 6, 4: 2}[PDE[pde]]
        self._ck(self._lib.gpp_gn_setup(self._h, PDE[pde], _ptr(params), _ptr(rhs_f), _ptr(bdy_g) if self.Nb else None,
                                        _ptr(data_u) if nd else None, nd, float(noise)), "gpp_gn_setup")

    def gn_set_z(self, z):
        z = _f64(z, (self.nz * self.N,))
        self._ck(self._lib.gpp_gn_set_z(self._h, _ptr(z)), "gpp_gn_set_z")

    def gn_get_z(self):
        z = np.empty(self.nz * self.N)
        self._ck(self._lib.gpp_gn_get_z(self._h, _ptr(z)), "gpp_gn_get_z")
        return z

    def gn_loss(self):
        v = C.c_double()
        self._ck(self._lib.gpp_gn_loss(self._h, C.byref(v)), "gpp_gn_loss")
        return float(v.value)

    def gn_step(self, step):
        v = C.c_double()
        self._ck(self._lib.gpp_gn_step(self._h, float(step), C.byref(v)), "gpp_gn_step")
        return float(v.value)

    def gn_grad_hess(self, want_grad=True, want_hess=True):
        n = self.nz * self.N
        g = np.empty(n) if want_grad else None
        H = np.empty((n, n)) if want_hess else None
        self._ck(self._lib.gpp_gn_grad_hess(self._h, _ptr(g), _ptr(H)), "gpp_gn_grad_hess")
        return g, H

    def gn_residual(self, slot):
        M, _ = self.gram_size(slot)
        out = np.empty(M)
        self._ck(self._lib.gpp_gn_residual(self._h, slot, _ptr(out)), "gpp_gn_residual")
        return out

    def gn_coef(self, slot, p, q):
        out = np.empty(self.N)
        present = C.c_int()
        self._ck(self._lib.gpp_gn_coef(self._h, slot, p, q, _ptr(out), C.byref(present)), "gpp_gn_coef")
        return out, bool(present.value)

    # ---- prediction
    def predict(self, slot, X_test, w):
        Xt = _f64(X_test)
        M, _ = self.gram_size(slot)
        w = _f64(w, (M,))
        out = np.empty(Xt.shape[0])
        self._ck(self._lib.gpp_predict(self._h, slot, _ptr(Xt), Xt.shape[0], _ptr(w), _ptr(out)), "gpp_predict")
        return out

    def theta_test(self, slot, X_test):
        Xt = _f64(X_test)
        M, _ = self.gram_size(slot)
        out = np.empty((Xt.shape[0], M))
        self._ck(self._lib.gpp_theta_test(self._h, slot, _ptr(Xt), Xt.shape[0], _ptr(out)), "gpp_theta_test")
        return out

    def predict_var(self, slot, X_test):
        """Posterior variance kappa(x, x) - theta(x)^T Theta^{-1} theta(x) at the test points (unclamped)."""
        Xt = _test_points(X_test)
        out = np.empty(Xt.shape[0])
        self._ck(self._lib.gpp_predict_var(self._h, slot, _ptr(Xt), Xt.shape[0], _ptr(out)), "gpp_predict_var")
        return out

    def kernel_eval(self, kernel, kernel_parameter, op_x, op_y, x1, x2, y1, y2):
        arrs = np.broadcast_arrays(*[np.asarray(a, dtype=np.float64) for a in (x1, x2, y1, y2)])
        shape = arrs[0].shape
        flat = [np.ascontiguousarray(a.ravel()) for a in arrs]
        out = np.empty(flat[0].shape[0])
        kp = kernel_params(kernel, kernel_parameter)
        self._ck(self._lib.gpp_kernel_eval(self._h, KERNEL[kernel], _ptr(kp), op_x, op_y, _ptr(flat[0]), _ptr(flat[1]),
                                           _ptr(flat[2]), _ptr(flat[3]), out.shape[0], _ptr(out)), "gpp_kernel_eval")
        return out.reshape(shape)


    # ---- multi-GPU: one problem sharded over the GPUs of a box (one process per GPU); see _dist.py for the plumbing
    def dist_init(self, rank, world, id_bytes):
        buf = (C.c_ubyte * 128).from_buffer_copy(bytes(id_bytes))
        self._ck(self._lib.gpp_dist_init(self._h, int(rank), int(world), buf), "gpp_dist_init")
        self.rank, self.world = int(rank), int(world)

    def dist_init_virtual(self, nranks):
        """Tests: run the task plans of `nranks` ranks one after the other on this GPU (no NCCL)."""
        self._ck(self._lib.gpp_dist_init_virtual(self._h, int(nranks)), "gpp_dist_init_virtual")
        self.rank, self.world = 0, int(nranks)

    def dist_set_grid(self, P, Q):
        self._ck(self._lib.gpp_dist_set_grid(self._h, int(P), int(Q)), "gpp_dist_set_grid")

    def dist_info(self):
        v = [C.c_int() for _ in range(4)]
        self._ck(self._lib.gpp_dist_info(self._h, *[C.byref(x) for x in v]), "gpp_dist_info")
        return dict(zip(("rank", "world", "P", "Q"), (x.value for x in v)))

    def dist_exchange_mode(self):
        """'p2p' (fused peer stores over NVLink + flags) or 'nccl' (all-gather / broadcast)."""
        return "p2p" if self._lib.gpp_dist_exchange_mode(self._h) == 1 else "nccl"

    def dist_finalize(self):
        self._ck(self._lib.gpp_dist_finalize(self._h), "gpp_dist_finalize")

    def dist_gram_assemble(self, layout, kernel, kernel_parameter):
        kp = kernel_params(kernel, kernel_parameter)
        self._ck(self._lib.gpp_dist_gram_assemble(self._h, LAYOUT[layout], KERNEL[kernel], _ptr(kp)), "gpp_dist_gram_assemble")

    def dist_get_diag(self):
        M, _ = self.gram_size(0)
        out = np.empty(M)
        self._ck(self._lib.gpp_dist_get_diag(self._h, _ptr(out)), "gpp_dist_get_diag")
        return out

    def dist_add_diag(self, add):
        M, _ = self.gram_size(0)
        add = _f64(add, (M,))
        self._ck(self._lib.gpp_dist_add_diag(self._h, _ptr(add)), "gpp_dist_add_diag")

    def dist_potrf(self):
        info = C.c_int()
        self._ck(self._lib.gpp_dist_potrf(self._h, C.byref(info)), "gpp_dist_potrf")
        return info.value

    def dist_inverse(self):
        self._ck(self._lib.gpp_dist_inverse(self._h), "gpp_dist_inverse")

    def dist_gn_step(self, step):
        v = C.c_double()
        self._ck(self._lib.gpp_dist_gn_step(self._h, float(step), C.byref(v)), "gpp_dist_gn_step")
        return float(v.value)

    def dist_predict_var(self, X_test):
        """predict_var of slot 0 with the test points split over the ranks; the same vector on every rank."""
        Xt = _test_points(X_test)
        out = np.empty(Xt.shape[0])
        self._ck(self._lib.gpp_dist_predict_var(self._h, _ptr(Xt), Xt.shape[0], _ptr(out)), "gpp_dist_predict_var")
        return out


def dist_plan_check(n, NB, P, Q=1, phase=0, nb_extra=0):
    """Host-only consistency check of the sharded task plans (works without a GPU); 0 = consistent."""
    return int(load().gpp_dist_plan_check(int(n), int(NB), int(P), int(Q), int(phase), int(nb_extra)))


def dist_hess_plan_check(N, NB, P, Q=1, pde="Burgers", nb_extra=0):
    """Host-only check of the Theta^-1 sub-block plans of a PDE's sharded Hessian (works without a GPU); 0 = consistent."""
    return int(load().gpp_dist_hess_plan_check(int(N), int(NB), int(P), int(Q), PDE[pde], int(nb_extra)))


def nccl_unique_id():
    lib = load()
    buf = (C.c_ubyte * 128)()
    if lib.gpp_dist_unique_id(buf) != 0:
        raise GppError("gpp_dist_unique_id failed")
    return bytes(buf)


_default_engine = None


def default_engine():
    """Process-wide engine used by the free functions (Gram_matrix_assembly, kernel classes)."""
    global _default_engine
    if _default_engine is None:
        _default_engine = Engine()
    return _default_engine
