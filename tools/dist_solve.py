"""One elliptic solve sharded over N GPUs (torchrun --nproc-per-node N tools/dist_solve.py --N 40000), or over `--virtual n`
emulated ranks on one GPU.  Prints one JSON line per repetition with the per-phase times (max over ranks).
--check: backward error of the sharded factor, and the sharded solve against the single-GPU solve on the same inputs
(small sizes).
--pde burgers: the Burgers problem of main_Burgers1d.py instead (u(0, x) = -sin(pi x), zero lateral boundary, f = 0,
alpha = 1, nu = 0.02, anisotropic kernel (0.3, 0.05), (t, x) in [0, 1] x [-1, 1]; M = 4 N + N_boundary); its JSON line also
carries the flops of the Theta^-1 sub-block phase (max over ranks and total), counted with the rule of the plan builder.
--single: the unsharded class path on the same inputs, with the same per-phase times (the one-GPU baseline at sizes too
large for --check).  --dump-outputs DIR: loss history, solution and predictions of the last repetition as .npy files."""
import argparse, json, math, os, sys, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np

ap = argparse.ArgumentParser()
ap.add_argument("--N", type=int, default=10000)
ap.add_argument("--Nb", type=int, default=0, help="boundary points (default: 4 (ceil(sqrt(N)) + 1))")
ap.add_argument("--pde", choices=("elliptic", "burgers"), default="elliptic")
ap.add_argument("--nugget", type=float, default=None, help="default 1e-10 (elliptic), 1e-5 (burgers)")
ap.add_argument("--gn_steps", type=int, default=4)
ap.add_argument("--reps", type=int, default=2)
ap.add_argument("--NB", type=int, default=512)
ap.add_argument("--Q", type=int, default=1)
ap.add_argument("--virtual", type=int, default=0)
ap.add_argument("--check", action="store_true")
ap.add_argument("--single", action="store_true", help="unsharded class path on one GPU")
ap.add_argument("--dump-outputs", default=None, metavar="DIR")
a = ap.parse_args()
if a.nugget is None:
    a.nugget = 1e-5 if a.pde == "burgers" else 1e-10
if a.single and (a.virtual or a.check):
    ap.error("--single runs the unsharded path alone")

rank, world, local = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1)), int(os.environ.get("LOCAL_RANK", 0))
dist = None
if not a.virtual and not a.single:
    import torch
    import torch.distributed as dist
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
from nonlinpdes_gpsolver_b200 import PDEs, _lib


def u_true(x1, x2):
    return np.sin(np.pi * x1) * np.sin(np.pi * x2) + 2 * np.sin(4 * np.pi * x1) * np.sin(4 * np.pi * x2)


def f_rhs(x1, x2):
    s1 = np.sin(np.pi * x1) * np.sin(np.pi * x2)
    s4 = np.sin(4 * np.pi * x1) * np.sin(4 * np.pi * x2)
    w = s1 + 2 * s4
    return 2 * np.pi ** 2 * s1 + 64 * np.pi ** 2 * s4 + 1.0 * (w * w * w)


def burgers_bdy(x1, x2):                            # main_Burgers1d.py: u(0, x) = -sin(pi x), zero at x = -1, 1
    return -np.sin(np.pi * x2) * (x1 == 0) + 0 * (x2 == 0)


def make_problem():
    if a.pde == "burgers":
        return PDEs.Burgers(alpha=1.0, nu=0.02, bdy=burgers_bdy, rhs=lambda x1, x2: 0, domain=dom)
    return PDEs.Nonlinear_elliptic2d(alpha=1.0, m=3, bdy=u_true, rhs=f_rhs, domain=dom)


def gram(p):
    if a.pde == "burgers":
        p.Gram_matrix("anisotropic_Gaussian", [0.3, 0.05], a.nugget, "adaptive")
    else:
        p.Gram_matrix("Gaussian", 0.2, a.nugget, "adaptive")


# Hessian terms (p, p') of each unknown-field pair (q, q'): p runs over the operator blocks whose Jacobian coefficient
# c_pq is nonzero (csrc/gn.cu, set_kind)
ROWS_OF_FIELD = {"elliptic": [[0, 1]], "burgers": [[0, 3], [0, 1], [0, 2]]}[a.pde]


def ablock_flops(N, M, NB, P, Q):
    """flops of the Theta^-1 sub-block phase per rank, by the rule of build_ablock_plan (csrc/dist.cu): every own block of
    the nz N x nz N Hessian is cut into one-field segments, and every term of a segment pair is a GEMM over
    K = [floor16(max(a_row, b_row)), round_up(M, 16))."""
    nz = len(ROWS_OF_FIELD)
    n, k1 = nz * N, -(-M // 16) * 16
    nblk = -(-n // NB)

    def segs(b):
        out, r, g1 = [], b * NB, min((b + 1) * NB, n)
        while r < g1:
            q = r // N
            e = min(g1, (q + 1) * N)
            out.append((q, r - q * N, e - r))
            r = e
        return out
    per = [0] * (P * Q)
    for bi in range(nblk):
        for bc in range(bi + 1):
            owner = (bi % P) * Q + bc % Q
            for q, i0, li in segs(bi):
                for qq, j0, lj in segs(bc):
                    for p in ROWS_OF_FIELD[q]:
                        for pp in ROWS_OF_FIELD[qq]:
                            per[owner] += 2 * li * lj * (k1 - max(p * N + i0, pp * N + j0) // 16 * 16)
    return per


N = a.N
Nb = a.Nb or 4 * (math.ceil(math.sqrt(N)) + 1)
np.random.seed(0)                                   # same points / initial guess on every rank
dom = np.array([[0.0, 1.0], [-1.0, 1.0]]) if a.pde == "burgers" else np.array([[0.0, 1.0], [0.0, 1.0]])
prob = make_problem()
if a.single:
    prob._eng = _lib.Engine(local)
prob._engine().set_option("NB", a.NB)
prob.sampled_pts(N, Nb)
nz = len(ROWS_OF_FIELD)
init = np.random.normal(0.0, 1.0, nz * N)
if a.single:
    pass
elif a.virtual:
    prob.shard(virtual_ranks=a.virtual, Q=a.Q)
else:
    prob.shard(dist, Q=a.Q)
eng = prob._engine()
M = (4 if a.pde == "burgers" else 2) * N + prob.N_boundary


def maxred(vals):
    if dist is None:
        return list(vals)
    import torch
    t = torch.tensor(list(vals), dtype=torch.float64, device="cuda")
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return t.tolist()


for rep in range(a.reps):
    if dist is not None:
        dist.barrier()
    eng.sync()
    eng.timer2_start()
    gram(prob)
    prob.Gram_Cholesky()
    prob.GN_method(a.gn_steps, 1, init, print_hist=False)
    total = eng.timer2_stop()
    t = prob.timings
    asm, potrf, inv, gn, tot = maxred([t["assembly_ms"], t["potrf_ms"], t["inverse_ms"], t["gn_ms"], total])
    if rank == 0:
        rec = dict(world=1 if a.single else (a.virtual or world), virtual=bool(a.virtual),
                   grid=None if a.single else eng.dist_info(), exchange=None if a.single else eng.dist_exchange_mode(),
                   N=N, M=M, NB=a.NB, rep=rep, info=prob.chol_info,
                   asm_ms=round(asm, 3), potrf_ms=round(potrf, 2), potrf_TF=round(M ** 3 / 3 / potrf / 1e9, 2),
                   inverse_ms=round(inv, 2), inverse_TF=round(2 * M ** 3 / 3 / inv / 1e9, 2), gn_ms=round(gn, 2),
                   gn_step_ms=round(gn / a.gn_steps, 2), solve_ms=round(tot, 2), final_loss=prob.loss_hist[-1])
        if a.pde == "elliptic":
            err = np.abs(u_true(prob.X_domain[:, 0], prob.X_domain[:, 1]) - prob.sol_sampled_pts)
            rec["pts_L2_err"] = float(np.sqrt(np.mean(err ** 2)))
        if a.pde != "elliptic" or a.single:
            rec.update(pde=a.pde, single=a.single, N_boundary=prob.N_boundary, nugget=a.nugget, gn_steps=a.gn_steps)
        if a.pde != "elliptic" and not a.single:
            info = eng.dist_info()
            fl = ablock_flops(N, M, a.NB, info["P"], info["Q"])
            rec.update(ablock_flop_max_rank=float(max(fl)), ablock_flop_total=float(sum(fl)))
        print(json.dumps(rec), flush=True)

Xt = np.random.RandomState(1).uniform(dom[:, 0], dom[:, 1], (64, 2))
if a.dump_outputs and rank == 0:
    prob.extend_sol(Xt)
    os.makedirs(a.dump_outputs, exist_ok=True)
    for name, v in (("loss_hist", prob.loss_hist), ("sol", prob.sol), ("pred", prob.extended_sol)):
        np.save(os.path.join(a.dump_outputs, name + ".npy"), np.asarray(v, dtype=np.float64))

if a.check:
    L = eng.gram_download(0, 1)                        # every rank holds the whole factor
    ref = make_problem()
    ref._eng = _lib.Engine(local)
    ref._eng.set_option("NB", a.NB)
    ref.get_sampled_points(prob.X_domain, prob.X_boundary)
    gram(ref)
    theta = ref.Theta
    ref.Gram_Cholesky()
    ref.GN_method(a.gn_steps, 1, init, print_hist=False)
    Lsingle = ref.L
    e_res = float(np.max(np.abs(L @ L.T - theta)) / (np.max(np.abs(theta)) * np.sqrt(M)))     # backward error of the sharded factor
    e_lap = float(np.max(np.abs(L - Lsingle)) / np.max(np.abs(Lsingle)))                      # vs the single-GPU factor
    e_loss = float(np.max(np.abs(np.array(prob.loss_hist) - np.array(ref.loss_hist)) / np.abs(ref.loss_hist)))
    e_sol = float(np.max(np.abs(prob.sol_sampled_pts - ref.sol_sampled_pts)) / np.max(np.abs(ref.sol_sampled_pts)))
    prob.extend_sol(Xt); ref.extend_sol(Xt)
    e_pred = float(np.max(np.abs(prob.extended_sol - ref.extended_sol)))
    ok = e_res < 1e-13 and e_lap < 1e-5 and e_loss < 1e-6 and e_sol < 1e-6 and e_pred < 1e-5
    vals = maxred([e_res, e_lap, e_loss, e_sol, e_pred, 0.0 if ok else 1.0])
    if rank == 0:
        print(json.dumps(dict(check="sharded factor: backward error and vs single-GPU factor; sharded solve vs single-GPU solve",
                              LLt_minus_Theta_rel=vals[0], L_vs_single_gpu=vals[1], loss_hist_rel=vals[2], sol_rel=vals[3], pred_abs=vals[4],
                              ok=bool(vals[5] == 0.0))), flush=True)
    assert ok, (e_res, e_lap, e_loss, e_sol, e_pred)
if dist is not None:
    eng.dist_finalize()
    dist.destroy_process_group()
