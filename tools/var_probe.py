"""Posterior-variance timing on one GPU (developer tool; bench.py is the contract).

Solves the bench.py workload (nonlinear elliptic, N_domain = 40 000, N_boundary = 4 (ceil(sqrt(N)) + 1), Gaussian
sigma = 0.2, adaptive nugget 1e-12, numpy seed 0, 4 GN steps), then times extend_sol_var on a 100 x 100 grid and on
18 944 random points (one warm-up call per shape, then one timed call, host clock around a call that ends in a device
synchronise).  Prints one JSON line: GPU name and power limit read in the same run, M, and per shape N_test, ms,
N_test M^2 / t in TFLOP/s (the flops of the triangular solve W L^T = Theta_test), kernel launches of the call and the
min / max of the variance.  --trace DIR: a torch.profiler trace of one more call on the random points, written there."""
import argparse, json, math, os, subprocess, sys, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np

ap = argparse.ArgumentParser()
ap.add_argument("--N", type=int, default=40000)
ap.add_argument("--nugget", type=float, default=1e-12)
ap.add_argument("--gn_steps", type=int, default=4)
ap.add_argument("--random_points", type=int, default=18944)
ap.add_argument("--trace", default=None, metavar="DIR")
a = ap.parse_args()
if a.trace:
    import torch                                        # before the library: torch must resolve its own NCCL symbols first
    from torch.profiler import ProfilerActivity, profile

from nonlinpdes_gpsolver_b200 import PDEs


def u_true(x1, x2):
    return np.sin(np.pi * x1) * np.sin(np.pi * x2) + 2 * np.sin(4 * np.pi * x1) * np.sin(4 * np.pi * x2)


def f_rhs(x1, x2):
    s1 = np.sin(np.pi * x1) * np.sin(np.pi * x2)
    s4 = np.sin(4 * np.pi * x1) * np.sin(4 * np.pi * x2)
    w = s1 + 2 * s4
    return 2 * np.pi ** 2 * s1 + 64 * np.pi ** 2 * s4 + 1.0 * (w * w * w)


def gpu_info():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                         capture_output=True, text=True, check=True).stdout.strip().split(", ")
    return out[0], out[1]


N = a.N
np.random.seed(0)
p = PDEs.Nonlinear_elliptic2d(alpha=1.0, m=3, bdy=u_true, rhs=f_rhs, domain=np.array([[0.0, 1.0], [0.0, 1.0]]))
p.sampled_pts(N, 4 * (math.ceil(math.sqrt(N)) + 1))
init = np.random.normal(0.0, 1.0, N)
p.Gram_matrix("Gaussian", 0.2, a.nugget, "adaptive")
p.Gram_Cholesky()
p.GN_method(a.gn_steps, 1, init, print_hist=False)
eng = p._engine()
M = eng.gram_size(0)[0]
g = np.linspace(0.0, 1.0, 100)
grid = np.stack(np.meshgrid(g, g), axis=-1).reshape(-1, 2)
rand = np.random.RandomState(7).uniform(0.0, 1.0, (a.random_points, 2))
runs = []
for name, X in (("grid_100x100", grid), ("random", rand)):
    p.extend_sol_var(X)                                 # warm-up of this shape
    eng.sync()
    l0 = eng.launch_count()
    t0 = time.perf_counter()
    p.extend_sol_var(X)                                 # returns after the device-to-host copy of the result
    ms = (time.perf_counter() - t0) * 1e3
    var = p.extended_var
    runs.append(dict(points=name, N_test=X.shape[0], ms=round(ms, 1), TFLOPs=round(X.shape[0] * M * M / ms / 1e9, 2),
                     launches=eng.launch_count() - l0, var_min=float(var.min()), var_max=float(var.max())))
name, power = gpu_info()
print(json.dumps(dict(gpu=name, power_limit=power, N_domain=N, M=M, NB=512, nugget=a.nugget, chol_info=p.chol_info,
                      runs=runs)), flush=True)
if a.trace:
    os.makedirs(a.trace, exist_ok=True)
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        p.extend_sol_var(rand)
        torch.cuda.synchronize()
    prof.export_chrome_trace(os.path.join(a.trace, "var_probe.pt.trace.json"))
    with open(os.path.join(a.trace, "var_probe_kernels.txt"), "w") as f:
        f.write(prof.key_averages().table(sort_by="cuda_time_total", row_limit=20))
