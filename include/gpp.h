/* libgpp_b200 -- C ABI of the B200-native GP-PDE Gauss-Newton hot path.
 *
 * The reference (yifanc96/NonLinPDEs-GPsolver) has no FFI: its boundary is the Python
 * object API (src/solver.py, src/PDEs.py, src/InverseProblems.py, src/Gram_matrice.py).
 * Each entry point below names the reference call it replaces; the Python package
 * nonlinpdes_gpsolver_b200 binds them with ctypes (see INTEGRATION.md).
 *
 * Conventions
 *   - return 0 = OK; < 0 = bad argument / state; >= 1000 = CUDA error;
 *     numerical failure is reported through *info (LAPACK style, first failed pivot).
 *   - all host arrays are float64, C-contiguous (numpy row-major); the caller owns them.
 *   - device memory, the stream and all intermediate matrices belong to the handle.
 *   - one handle = one device, NOT thread-safe (one host thread per handle).
 *   - calls enqueue work on the handle's stream; calls that return data synchronise it.
 */
#ifndef GPP_B200_H
#define GPP_B200_H

#ifdef __cplusplus
extern "C" {
#endif

typedef struct gpp_handle gpp_handle;

/* Block layouts of Theta: Gram_matrix_assembly(eqn=...)  src/Gram_matrice.py:41-187 */
#define GPP_LAYOUT_ELLIPTIC 0 /* [Delta(d); delta(db)]             :41-56   */
#define GPP_LAYOUT_BURGERS  1 /* [d1(d); d2(d); d22(d); delta(db)]  :58-99   */
#define GPP_LAYOUT_EIKONAL  2 /* [d1; d2; Delta; delta(db)]  (= Darcy Theta_u) :100-179 */
#define GPP_LAYOUT_DARCY_A  3 /* [d1; d2; delta(d)]  (Darcy Theta_a) :183-186 */
/* kernels: src/kernels.py:8 (Gaussian_kernel), :91 (Anisotropic_Gaussian_kernel) */
#define GPP_KERNEL_GAUSSIAN 0
#define GPP_KERNEL_ANISOTROPIC 1
/* PDE ids for the GN step: src/PDEs.py:18,211,352 ; src/InverseProblems.py:16 */
#define GPP_PDE_ELLIPTIC 0
#define GPP_PDE_BURGERS 1
#define GPP_PDE_EIKONAL 2
#define GPP_PDE_DARCY 3
#define GPP_PDE_ELLIPTIC_RELAXED 4 /* GN_relaxed_method, src/PDEs.py:137-201: z = [v; w], params {alpha, m, pen_lambda} */

int gpp_create(int device, gpp_handle** out);
int gpp_destroy(gpp_handle* h);
const char* gpp_last_error(gpp_handle* h);
/* options: "NB" (block-column width of the blocked factorisations, multiple of 128) */
int gpp_set_option(gpp_handle* h, const char* name, double value);
int gpp_sync(gpp_handle* h);
/* number of kernels this library launched on the handle so far */
long gpp_launch_count(gpp_handle* h);
/* CUDA-event timer on the handle's stream */
int gpp_timer_start(gpp_handle* h);
int gpp_timer_stop(gpp_handle* h, float* ms);
/* a second, independent event pair (outer timed region of bench.py around whole solves) */
int gpp_timer2_start(gpp_handle* h);
int gpp_timer2_stop(gpp_handle* h, float* ms);

/* collocation points: X.sampled_pts / X.get_sampled_points  src/PDEs.py:34-54 */
int gpp_set_points(gpp_handle* h, const double* X_domain, int N_domain, const double* X_boundary, int N_boundary);

/* Gram_matrix_assembly  src/Gram_matrice.py:11-187.  Theta stays device-resident in `slot`
 * (lower triangle).  kparams = {b1, b2, e1, e2}: kappa = exp(-(b1 d1^2 + b2 d2^2)/2); the exponent is
 * evaluated as e1*(d1^2+d2^2) (Gaussian, e1 = -(1/(2 sigma^2))) or -((d1/e1)^2 + (d2/e2)^2) (anisotropic). */
int gpp_gram_assemble(gpp_handle* h, int slot, int layout, int kernel, const double* kparams);
int gpp_gram_size(gpp_handle* h, int slot, int* M, int* M_interior);
/* diagonal access for the trace-ratio nugget  src/PDEs.py:56-73 (host computes the ratios like numpy) */
int gpp_gram_get_diag(gpp_handle* h, int slot, double* diag_out);
int gpp_gram_add_diag(gpp_handle* h, int slot, const double* add);
/* what: 0 = Theta (symmetric, from the lower triangle), 1 = L (zeros above the diagonal),
 *       2 = interior block of Theta^{-1} (M_interior x M_interior).  out is dense row-major. */
int gpp_gram_download(gpp_handle* h, int slot, int what, double* out);
int gpp_gram_upload(gpp_handle* h, int slot, const double* theta); /* tests: replace Theta by a host matrix */

/* X.Gram_Cholesky  src/PDEs.py:75-80 (jnp.linalg.cholesky).  *info = 0 or the 1-based index of the
 * first non-positive pivot (the factor then holds NaNs from there on, like JAX's NaN output). */
int gpp_potrf(gpp_handle* h, int slot, int* info);
/* interior block of Theta^{-1} (all rows J touches), computed once per solve and reused by every GN step */
int gpp_inverse(gpp_handle* h, int slot);
/* x = Theta^{-1} b by two triangular solves  (extend_sol  src/PDEs.py:205) */
int gpp_solve_vec(gpp_handle* h, int slot, const double* b, double* x);

/* GN problem data.  params: elliptic {alpha, m}; Burgers {alpha, nu}; Eikonal {eps}; Darcy {}.
 * rhs_f[N], bdy_g[Nb]; Darcy: data_u[N_data], noise_level  (src/InverseProblems.py:62-64). */
int gpp_gn_setup(gpp_handle* h, int pde, const double* params, const double* rhs_f, const double* bdy_g,
                 const double* data_u, int N_data, double noise_level);
int gpp_gn_set_z(gpp_handle* h, const double* z);
int gpp_gn_get_z(gpp_handle* h, double* z);
/* X.loss(z) at the current z  src/PDEs.py:83-87 */
int gpp_gn_loss(gpp_handle* h, double* loss);
/* one iteration of X.GN_method's loop body  src/PDEs.py:117-120: z <- z - step * H^{-1} g, returns loss(z) */
int gpp_gn_step(gpp_handle* h, double step_size, double* loss);
/* X.grad_loss(z) and X.Hessian_GN(z, z)  src/PDEs.py:90-91,101-102 at the current z (either pointer may be NULL);
 * grad_out[n], hess_out[n x n] row-major with n = (#unknown blocks) * N.  Needs gpp_inverse. */
int gpp_gn_grad_hess(gpp_handle* h, double* grad_out, double* hess_out);
/* F(z) of slot (the reference's sol_vec, src/PDEs.py:132-133) at the current z */
int gpp_gn_residual(gpp_handle* h, int slot, double* F_out);
/* Jacobian coefficient vector c_pq (length N) of slot at the current z; returns 1 in *present if nonzero */
int gpp_gn_coef(gpp_handle* h, int slot, int p, int q, double* c_out, int* present);

/* X.extend_sol  src/PDEs.py:203-208: out = Theta_test(X_test) @ w, Theta_test never materialised */
int gpp_predict(gpp_handle* h, int slot, const double* X_test, int N_test, const double* w, double* out);
/* construct_Theta_test  src/Gram_matrice.py:190-289: out is N_test x M row-major */
int gpp_theta_test(gpp_handle* h, int slot, const double* X_test, int N_test, double* out);

/* Gaussian_kernel / Anisotropic_Gaussian_kernel methods  src/kernels.py:8-179, vectorised over n pairs:
 * out = L_x(op_x) L_y(op_y) kappa(x, y).  Operator ids: 0 identity, 1 d/dx1, 2 d/dx2, 3 d^2/dx2^2, 4 Laplacian
 * (e.g. Delta_x_D_y1_kappa = (4, 1)). */
int gpp_kernel_eval(gpp_handle* h, int kernel, const double* kparams, int op_x, int op_y, const double* x1,
                    const double* x2, const double* y1, const double* y2, long n, double* out);

/* ---- multi-GPU: ONE problem sharded over the GPUs of a box (new functionality: the reference is single-process,
 * SURVEY section 2).  One process per GPU; NCCL over NVLink.  Storage is replicated, work is owner-computes on a
 * P x Q block-cyclic grid of NB x NB blocks (default P = world, Q = 1); finished panels are gathered with NCCL.
 * Rank 0 creates the 128-byte NCCL id and distributes it out of band (torch.distributed / MPI / a file); every rank
 * then calls gpp_dist_init.  All ranks must set the same points and make the same calls in the same order. */
int gpp_dist_unique_id(unsigned char* id128);
int gpp_dist_init(gpp_handle* h, int rank, int world, const unsigned char* id128);
/* tests: run the plans of `nranks` ranks one after the other on this one GPU (no NCCL, shared storage) */
int gpp_dist_init_virtual(gpp_handle* h, int nranks);
/* process grid, P * Q = number of ranks; block (bi, bc) belongs to rank (bi mod P) * Q + (bc mod Q) */
int gpp_dist_set_grid(gpp_handle* h, int P, int Q);
int gpp_dist_info(gpp_handle* h, int* rank, int* world, int* P, int* Q);
/* host-only self-check of the owner-computes task plans for an n x n matrix on a P x Q grid (no GPU needed): every block
 * that a step must solve / update is handled by exactly one rank, its owner.  phase 0 Cholesky, 1 U = L^-T, 2 Theta^-1
 * sub-blocks (n = N_domain, nb_extra = boundary rows).  0 = consistent. */
int gpp_dist_plan_check(int n, int NB, int P, int Q, int phase, int nb_extra);
/* host-only self-check of the Theta^-1 sub-block plans of a PDE's sharded Hessian (pde GPP_PDE_ELLIPTIC, _BURGERS or
 * _EIKONAL; N = N_domain, nb_extra = boundary rows): every lower block of the nz N x nz N Hessian has exactly one owner, and
 * every element of it receives each term of its unknown-block pair exactly once, from the right operand rows and K range.
 * Blocks that straddle the boundary between two unknown fields (N % NB != 0) are split into one-field segments.
 * 0 = consistent, -1 = bad argument or a PDE that does not shard.  Phase 2 of gpp_dist_plan_check is the elliptic case. */
int gpp_dist_hess_plan_check(int N, int NB, int P, int Q, int pde, int nb_extra);
/* how finished panels travel: 1 = peer-to-peer (the solve kernels store every finished tile straight into the peers'
 * replicated buffers over NVLink through CUDA IPC mappings and announce it by flags), 0 = NCCL all-gather / broadcast
 * (GPP_DIST_P2P=0, or CUDA IPC unavailable) */
int gpp_dist_exchange_mode(gpp_handle* h);
int gpp_dist_finalize(gpp_handle* h);
/* sharded Gram_matrix_assembly into slot 0: this rank's block rows (bi mod P == p), no exchange */
int gpp_dist_gram_assemble(gpp_handle* h, int layout, int kernel, const double* kparams);
/* nugget support: full diagonal on every rank (all-reduce) / add a full-length vector to the held diagonal entries */
int gpp_dist_get_diag(gpp_handle* h, double* diag_out);
int gpp_dist_add_diag(gpp_handle* h, const double* add);
/* distributed X.Gram_Cholesky of slot 0 (right-looking, look-ahead, one panel gather per block column).  Afterwards every
 * rank holds the whole factor: gpp_gn_loss, gpp_solve_vec, gpp_predict, gpp_gram_download(h, 0, 1, .) work on any rank. */
int gpp_dist_potrf(gpp_handle* h, int* info);
/* distributed counterpart of gpp_inverse (elliptic, Burgers and Eikonal layouts; the Darcy layouts are refused): U = L^{-T}
 * sharded then replicated, and the sub-blocks of the interior block of Theta^{-1} that this rank's Hessian blocks need for
 * the PDE of the layout in slot 0 */
int gpp_dist_inverse(gpp_handle* h);
/* gpp_gn_step with the Hessian assembled block-wise by the owners and factorised by the distributed Cholesky; z and the
 * returned loss are identical on every rank.  PDE ids GPP_PDE_ELLIPTIC, GPP_PDE_BURGERS and GPP_PDE_EIKONAL (the relaxed
 * method and Darcy are refused); the PDE of gpp_gn_setup must be the one of the layout gpp_dist_inverse planned for,
 * otherwise -5 */
int gpp_dist_gn_step(gpp_handle* h, double step_size, double* loss);

#ifdef __cplusplus
}
#endif
#endif
