// Internal declarations shared by the translation units of libgpp_b200.so.
// Everything here is device-side plumbing for the GP-PDE Gauss-Newton hot path
// (Gram assembly -> Cholesky -> GN steps); the public C ABI is include/gpp.h.
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <map>
#include <string>
#include <vector>

// TMA descriptors of one buffer for both GEMM tile sizes (box 16 x 128 and 16 x 64 doubles, 128B swizzle)
struct TMap2 {
  CUtensorMap m128, m64;
};

#define GPP_MAX_SLOTS 2      // Darcy needs Theta_u and Theta_a
#define GPP_MAX_BLOCKS 4     // row-operator blocks per Gram matrix
#define GPP_MAX_ZBLOCKS 6    // unknown blocks (Darcy: w0 w1 w2 v0 v1 v2)

// row operators (src/Gram_matrice.py block layouts)
enum { OP_ID = 0, OP_D1 = 1, OP_D2 = 2, OP_D22 = 3, OP_LAP = 4 };
// layouts
enum { LAY_ELLIPTIC = 0, LAY_BURGERS = 1, LAY_EIKONAL = 2, LAY_DARCY_A = 3 };
// PDE ids for the GN step
enum { PDE_ELLIPTIC = 0, PDE_BURGERS = 1, PDE_EIKONAL = 2, PDE_DARCY = 3, PDE_ELLIPTIC_RELAXED = 4 };

struct Layout {
  int nblk;
  int op[GPP_MAX_BLOCKS];
  int with_bdy[GPP_MAX_BLOCKS];
};

inline Layout make_layout(int id) {
  Layout l{};
  switch (id) {
    case LAY_ELLIPTIC: l.nblk = 2; l.op[0] = OP_LAP; l.op[1] = OP_ID; l.with_bdy[1] = 1; break;
    case LAY_BURGERS:  l.nblk = 4; l.op[0] = OP_D1; l.op[1] = OP_D2; l.op[2] = OP_D22; l.op[3] = OP_ID; l.with_bdy[3] = 1; break;
    case LAY_EIKONAL:  l.nblk = 4; l.op[0] = OP_D1; l.op[1] = OP_D2; l.op[2] = OP_LAP; l.op[3] = OP_ID; l.with_bdy[3] = 1; break;
    case LAY_DARCY_A:  l.nblk = 3; l.op[0] = OP_D1; l.op[1] = OP_D2; l.op[2] = OP_ID; break;
    default: l.nblk = 0;
  }
  return l;
}

// One Gram system: Theta -> L (lower triangle, in place), U = L^{-T} (strict upper
// triangle of the same buffer + clean diagonal blocks in udiag), Ainv = interior
// block of Theta^{-1} (full symmetric, separate buffer).
struct GramSlot {
  int layout_id = -1;
  Layout lay{};
  int N = 0, Nb = 0, M = 0, Mint = 0;   // Mint = rows that J touches (all but boundary rows)
  int off[GPP_MAX_BLOCKS + 1] = {0};
  long ld = 0;                           // leading dimension (doubles), multiple of 16
  double* T = nullptr;                   // M x ld
  double* udiag = nullptr;               // (nblk*NB) x NB clean diagonal blocks of U
  double* Ainv = nullptr;                // Mint x ldA
  long ldA = 0;
  bool factored = false, inverted = false;
  TMap2 mapT, mapUdiag;            // TMA descriptors (box 16 x 128 doubles, 128B swizzle)
  double kp_b1 = 0, kp_b2 = 0;           // kernel scales b1, b2
  double kp_e1 = 0, kp_e2 = 0;           // exponent coefficients (see gram.cu)
  int kernel_id = 0;
};

struct GnState {
  int pde = -1;
  int nz = 0;                 // number of unknown blocks
  int n = 0;                  // nz * N
  double params[4] = {0};
  int m_int = 0;              // elliptic: integer exponent m (0 if non-integer)
  double* rhs_f = nullptr;    // N
  double* bdy_g = nullptr;    // Nb
  double* data_u = nullptr;   // N_data
  int N_data = 0;
  double noise = 1.0;
  double* z = nullptr;        // n
  double* F[GPP_MAX_SLOTS] = {nullptr, nullptr};     // M_s
  double* s[GPP_MAX_SLOTS] = {nullptr, nullptr};     // L^{-1} F
  double* t[GPP_MAX_SLOTS] = {nullptr, nullptr};     // L^{-T} L^{-1} F
  double* coef = nullptr;     // [slot][p][q][N] Jacobian coefficient vectors
  unsigned char coef_kind[GPP_MAX_SLOTS][GPP_MAX_BLOCKS][GPP_MAX_ZBLOCKS]; // 0 zero, 1 vector
  double* H = nullptr;        // n x ldH
  long ldH = 0;
  double* g = nullptr;        // n
  double* scal = nullptr;     // small device scratch for reductions
  TMap2 mapH;
  bool ready = false;
  bool current = false;       // F, s = L^{-1} F and the coefficient vectors belong to the present z
};

struct gpp_handle {
  int device = 0;
  cudaStream_t stream = nullptr;      // main stream (all public calls are ordered on it)
  cudaStream_t cur = nullptr;         // stream the launch helpers use right now (= stream unless look-ahead is active)
  cudaStream_t sG[2] = {nullptr, nullptr};  // look-ahead: alternating streams of the long-K updates
  cudaStream_t sP = nullptr;          // look-ahead: high-priority stream of the panel chain
  std::vector<cudaEvent_t> evpool;    // events of the look-ahead dependency graph
  int lookahead = 1;
  int force_tile = 0;                 // 0 = heuristic, 64 / 128 = force that GEMM tile size (tests, tuning)
  std::string err;
  int N = 0, Nb = 0;
  double* Xd = nullptr;       // N x 2
  double* Xb = nullptr;       // Nb x 2
  double* Xall = nullptr;     // (N+Nb) x 2 : interior then boundary
  GramSlot slot[GPP_MAX_SLOTS];
  GnState gn;
  int* d_info = nullptr;      // device flag: first failed pivot (1-based) or 0
  int* d_trsv_flag = nullptr; // progress counters of the persistent triangular solves (ring of 16)
  unsigned trsv_calls = 0;
  unsigned* d_bar = nullptr;  // global-barrier counters of the persistent tiled Cholesky (ring of 64)
  unsigned bar_calls = 0;
  int tiled_potrf = 1;        // use the persistent tiled kernel for diagonal blocks and small matrices
  int tiled_max_n = 4608;     // largest matrix factored whole by the tiled kernel
  int tiled_grid_limit = 0;   // tests / tuning: cap on its grid size (0 = resident capacity)
  int blocksum = 1;           // task-list updates (right-looking schedules): 1 = sum the K = NB products of a launch from zero and
                              // subtract once (block summation, what LAPACK's GEMM-based updates do); 0 = entry-by-entry
                              // progressive subtraction.  Measured (profiles/r02_nugget_*.jsonl): at N_domain = 20 000, nugget 1e-13
                              // every progressive schedule breaks down near pivot 35 000, block summation (NB 128 / 256 / 512) does not
  int rl_potrf = 0;           // Cholesky of a Gram slot larger than tiled_max_n: 1 = right-looking task-list schedule (block summation,
                              // factors N_domain = 20 000 at nugget 1e-13 where the progressive schedules break down) instead of the
                              // left-looking long-K schedule (15 % faster on one GPU: 5.15 s against 5.94 s at N_domain = 40 000).
                              // The Python classes retry with it automatically when the fast schedule reports a failed pivot.
  void* dist_local = nullptr; // one-rank instance of the sharded scheduler used by the single-GPU right-looking factorisation
  int persistent_gemm = 0;    // task-list GEMM: 1 = CTAs stay resident and walk the tile list, 0 = one CTA per tile (default).
                              // Measured (profiles/r02_summary.md): resident CTAs never hand an SM to the high-priority panel chain
                              // that runs beside the trailing update, so the look-ahead stalls: 3.57 s instead of 2.99 s per
                              // N_domain = 40 000 solve on 8 GPUs (single GPU, right-looking: no gain either, 28.8 vs 28.9 TFLOP/s)
  int fused_trsm_rows = 65536; // sharded path: panels with at most this many own rows use the one-launch panel solve
  double* work = nullptr;     // scratch (panel copies)
  size_t work_bytes = 0;
  int NB = 512;               // block-column width of the blocked factorisations
  // timing
  cudaEvent_t ev[10];               // [0,1] phase timer, [2..7] GN trace, [8,9] outer (bench) timer
  float t_asm = 0, t_potrf = 0, t_inv = 0, t_step = 0;
  long launches = 0;
  // distributed (dist.cu)
  void* dist = nullptr;
  bool dist_gn = false;               // GN steps use the sharded Hessian assembly + distributed Cholesky of H
  // capacity (doubles) of every device buffer obtained through dev_reserve, keyed by the address of its pointer:
  // buffers are grown, never shrunk, so repeated solves on one handle do not touch the allocator
  std::map<double**, size_t> caps;
};

#define GPP_OK 0
#define GPP_CUDA_ERR 1000

#define CUDA_TRY(h, expr)                                                         \
  do {                                                                            \
    cudaError_t _e = (expr);                                                      \
    if (_e != cudaSuccess) {                                                      \
      (h)->err = std::string(#expr) + ": " + cudaGetErrorString(_e);              \
      return GPP_CUDA_ERR;                                                        \
    }                                                                             \
  } while (0)

static inline long round_up(long x, long m) { return (x + m - 1) / m * m; }

// *p holds at least n doubles afterwards; reallocates (contents lost) only when the present buffer is too small
static inline int dev_reserve(gpp_handle* h, double** p, size_t n) {
  if (n == 0) n = 1;
  auto it = h->caps.find(p);
  if (*p && it != h->caps.end() && it->second >= n) return GPP_OK;
  if (*p) { cudaFree(*p); *p = nullptr; }
  h->caps.erase(p);
  CUDA_TRY(h, cudaMalloc(p, n * sizeof(double)));
  h->caps[p] = n;
  return GPP_OK;
}
static inline void dev_release(gpp_handle* h, double** p) {
  if (*p) { cudaFree(*p); *p = nullptr; }
  h->caps.erase(p);
}

// ---- gemm_dmma.cu -----------------------------------------------------------
struct GemmDesc {
  const TMap2* mapA;      // operand A rows (K-contiguous)
  const TMap2* mapB;      // operand B rows (K-contiguous)
  const TMap2* mapAdiag;  // optional clean diagonal blocks for A (U operand), else null
  const TMap2* mapBdiag;  // optional clean diagonal blocks for B
  int a_row0, b_row0;           // first row of A / B operand (map coordinates)
  double* C; long ldc;          // output origin pointer (row-major), already offset
  const double* Cin; long ldcin;// optional addend (may alias C), already offset
  int m, n;                     // output extents
  int k0, k1;                   // K range in A-map column coordinates
  int kb_off;                   // B-map column = k + kb_off
  int ktri;                     // 1: A rows are upper-triangular: k starts at diag block of the row tile
  int diag_nb;                  // block size of the clean diagonal blocks (NB)
  double alpha;
  int lower_only;               // skip tiles strictly above the diagonal (uses global row/col = a_row0+i, b_row0+j)
  // block-diagonal batch (multi-GPU Cholesky): bd_count diagonal blocks of the row-sharded matrix, one per owned block
  // row starting at local block bd_lblk0: C_blk -= A_blk[:, k0:k1] A_blk[:, k0:k1]^T (lower tiles).  0 = off.
  int bd_count, bd_world, bd_rank, bd_lblk0, bd_nb, bd_M;
};
int gemm_nt_launch(gpp_handle* h, const GemmDesc& d);

// Task-list mode of the same kernel (multi-GPU path): one task = one output block of up to bs x bs elements, processed
// by (bs / TILE)^2 CTAs.  C[c_row + i, c_col + j] (+)= alpha * sum_{k in [k0, k1)} A[a_row + i, k] * B[b_row + j, k + kb_off]
// for i < m, j < n; tri != 0: the block lies on the diagonal of a symmetric matrix, tiles strictly above it are skipped.
struct GemmTask {
  int a_row, b_row;
  int c_row, c_col;
  int m, n;
  int k0, k1;
  int kb_off, tri;
  int pad0, pad1;
};
static_assert(sizeof(GemmTask) == 48, "GemmTask is read as three 16-byte words");
struct GemmTaskDesc {
  const TMap2* mapA; const TMap2* mapB;
  double* C; long ldc;              // matrix origin (tasks carry the block position)
  const double* Cin; long ldcin;    // optional addend origin (may alias C)
  double alpha;
  const GemmTask* tasks;            // device pointer
  int ntasks, bs;                   // bs: task block size, a multiple of 128
  int blocksum;                     // 1: accumulate the products from zero, add Cin in the epilogue
};
int gemm_tasks_launch(gpp_handle* h, const GemmTaskDesc& d);
int make_tensor_map(gpp_handle* h, TMap2* map, const double* base, long rows, long cols, long ld);

// ---- chol.cu ---------------------------------------------------------------
struct Mat {
  double* base;
  long ld;
  const TMap2* map;
};
// rows of a panel solve: contiguous (stride_blk == 0) or block-cyclic: logical row block b of `nb` rows sits at
// physical rows (first_blk + b * stride_blk) * nb
struct TrsmRows {
  int rows;
  int first_blk, stride_blk, nb;
};
// Peer push (multi-GPU, replicated storage): results are stored not only locally but at the same position of every
// peer's buffer through NVLink (CUDA IPC mappings), and when the whole launch is done each peer's flag slot of this
// rank is set to `seq` (release at system scope).  npeers == 0: local only.
#define GPP_MAX_PEERS 7
struct PeerPush {
  int npeers;
  double* base[GPP_MAX_PEERS];                // peer copy of the pointer the kernel receives as its output origin
  unsigned long long* flag[GPP_MAX_PEERS];    // peer's flag slot for this rank
  unsigned long long seq;
  unsigned* counter;                          // local CTA counter (self-resetting)
};
// 64-wide base case of the panel solve X L^T = P (in place), L = nbl x nbl lower block; P points at column 0 of the panel
int trsm_base_launch(gpp_handle* h, double* P, long ldp, const TrsmRows& rm, const double* L, long ldl, int nbl);
// the same solve for the whole nbw-wide panel (nbw <= NB) in one launch: one CTA per 64 rows, no recursion
int trsm_panel_launch(gpp_handle* h, double* P, long ldp, const TrsmRows& rm, const double* L, long ldl, int nbw, const PeerPush* push = nullptr);
int fill_identity_launch(gpp_handle* h, double* A, long ld, int rows, int cols);
// X * L^T = P in place; P = rows x nb block of P at (pr0, pc0); L = nb x nb lower block of L at (lr0, lc0)
int trsm_right_lt(gpp_handle* h, const Mat& P, int pr0, int pc0, int rows, const Mat& L, int lr0, int lc0, int nb);
// Cholesky of the nb x nb block at (r0, c0) of A (recursive, 64-wide base), gidx0 = global pivot offset
int potrf_diag(gpp_handle* h, const Mat& A, int r0, int c0, int nb, int gidx0);
// ---- gram.cu: rows [i_begin, i_begin + nrows) of row-operator block `prow`, all column blocks q <= prow
int gram_assemble_rows(gpp_handle* h, GramSlot& s, int prow, int i_begin, int nrows, double* dst, long ld);
// Blocked lower Cholesky of the n x n matrix at A (row-major, ld), in place, using map for TMA.
int potrf_lower(gpp_handle* h, double* A, long ld, int n, const TMap2* map);
// U = L^{-T} into the strict upper triangle + udiag, then Ainv = (L L^T)^{-1}[0:mint,0:mint]
int inverse_interior(gpp_handle* h, GramSlot& s);
// y = L^{-1} b (forward) / y = L^{-T} b (backward), vectors, in place in x
int trsv_lower(gpp_handle* h, const double* L, long ld, int n, double* x, bool transposed);

// ---- capi.cu: size / layout bookkeeping, buffer and tensor map of a Gram slot (no assembly)
int gram_slot_prepare(gpp_handle* h, int slot, int layout, int kernel, const double* kparams);
// ---- gram.cu ---------------------------------------------------------------
int gram_assemble(gpp_handle* h, GramSlot& s);
int gram_predict(gpp_handle* h, GramSlot& s, const double* d_xtest, int ntest, const double* d_w, double* d_out);
int gram_theta_test(gpp_handle* h, GramSlot& s, const double* d_xtest, int ntest, double* d_out, long ldo);

// ---- gn.cu -----------------------------------------------------------------
int gn_eval_F(gpp_handle* h, const double* d_z, bool with_coef);
int gn_loss(gpp_handle* h, const double* d_z, double* loss_host);
int gn_step(gpp_handle* h, double step, double* loss_host);
int gn_grad_hess(gpp_handle* h);
int gn_grad(gpp_handle* h);           // t = L^{-T} s and the gradient
// Hessian terms: H[(q, i), (q', j)] = 2 sum_t c_{s p q}[i] A_s[(p, i), (p', j)] c_{s p' q'}[j] over the terms t = (s, p, p')
// of the unknown-block pair (q, q') (index q * nz + q'), in the order the Hessian kernels sum them
struct TermTable {
  int nz, nslots;
  int nterms[GPP_MAX_ZBLOCKS * GPP_MAX_ZBLOCKS];
  unsigned char ts[GPP_MAX_ZBLOCKS * GPP_MAX_ZBLOCKS][8];
  unsigned char tp[GPP_MAX_ZBLOCKS * GPP_MAX_ZBLOCKS][8];
  unsigned char tpp[GPP_MAX_ZBLOCKS * GPP_MAX_ZBLOCKS][8];
};
int pde_nz(int pde);                                   // number of unknown blocks of a PDE id
int make_term_table(int pde, TermTable* tt);           // host only; -1 on an unknown PDE id
// multi-GPU: H blocks listed in d_blocks (int4: bi, bc, index e of the block's group of four sub-blocks, unused) from the
// compact sub-block store Asub (nbh x nbh sub-blocks, leading dimension nbh): element (r, c) of block e takes term t of
// its unknown-block pair from row (4 e + t) * nbh + r, column c.  Elliptic, Burgers and Eikonal (at most four terms a pair).
int dist_gn_hess_potrf(gpp_handle* h);   // dist.cu
// single GPU: the right-looking schedule of the sharded path with one rank (task-list updates, look-ahead streams)
int potrf_right_looking(gpp_handle* h, double* A, long ld, int n, const TMap2* map);
void dist_local_release(gpp_handle* h);
int gn_hess_blocks(gpp_handle* h, const int4* d_blocks, int nblocks, const double* Asub, int nbh);
int gram_kernel_eval(gpp_handle* h, int kernel, const double* kparams, int opx, int opy, const double* d_in, long n,
                     double* d_out);
