// Multi-GPU path: ONE problem sharded over the GPUs of a box.  One process per GPU, NCCL over NVLink / NVSwitch.
// The reference has no multi-device code at all (SURVEY section 2): this is new.
//
// Storage is REPLICATED, work is OWNER-COMPUTES.  Every rank holds the full M x ld buffer of Theta -> L (and of
// U = L^{-T}, and of the GN Hessian H); block (bi, bc) of NB x NB is owned by rank (bi mod P) * Q + (bc mod Q) of a
// P x Q process grid (2-D block-cyclic; Q = 1, the default, is block-row cyclic).  Only the owner updates a block;
// a block column that has become final is made consistent on every rank by one gather.  With NVSwitch every rank
// receives a panel at full link bandwidth whatever the grid shape, and 180 GB of HBM hold the replicated buffers at
// N_domain = 40 000 (52 GB each), so the classic reason for 2-D grids (panel volume per rank) does not apply; what
// does matter is the per-column critical path, and the right-looking schedule below keeps it short:
//
//   assembly : every Gram entry depends on two points only -> each rank fills the block rows it holds, no exchange.
//   Cholesky : right-looking by block column j.  owner(j, j) factorises the diagonal block and broadcasts it; the
//              owners of the panel blocks (bi, j) solve them against it (block-cyclic rows: all P process rows work);
//              the solved panel is gathered on every rank; every rank applies C(bi, bc) -= L(bi, j) L(bc, j)^T to the
//              trailing blocks it owns in ONE task-list launch of the DMMA kernel (K = NB, thousands of tiles, so wave
//              quantisation is negligible).  Look-ahead: column j+1 is updated first and its panel chain (diagonal
//              factorisation, broadcast, solve, gather) runs on a high-priority stream under the bulk of step j.
//              Each entry receives its updates in column order, each rounded relative to the remainder: the same
//              progressive accumulation as the single-GPU factorisation (DESIGN.md section 2.5).
//   U = L^-T : same skeleton on a second, clean buffer (zeros below the diagonal): at step i the owners solve
//              column i (U(b, i) L_ii^T = acc(b, i)), then update acc(b, c) -= U(b, i) L(c, i)^T for c > i.  L is
//              replicated, so for Q = 1 this needs no exchange on the critical path; the finished columns are
//              gathered on a third stream because every rank needs all of U next.
//   A blocks : the GN Hessian block (bi, bc) needs the four sub-blocks A_pp'(bi, bc) of the interior inverse
//              A = (U U^T)[interior]; their owner computes exactly those (one task-list launch, K from the diagonal to M).
//   GN step  : z, F, the triangular solves with L and the gradient are replicated (identical on every rank); the
//              Hessian blocks are assembled by their owners and H is factorised by the same distributed Cholesky.
//
// "Virtual" mode (gpp_dist_init_virtual) runs the same plans for all P*Q ranks one after the other on a single GPU,
// without NCCL: it lets the single-GPU test suite check ownership, task lists and kernels of the sharded path.
#include "../../include/gpp.h"
#include "gpp_internal.cuh"

#include <nccl.h>

#include <algorithm>
#include <cstring>
#include <map>
#include <vector>

namespace {

struct Grid { int P, Q, p, q; };
inline int owner_of(const Grid& g, int bi, int bc) { return (bi % g.P) * g.Q + (bc % g.Q); }
inline bool mine(const Grid& g, int bi, int bc) { return bi % g.P == g.p && bc % g.Q == g.q; }

struct Launch { size_t off = 0; int count = 0; };

// Task lists of one phase for one (virtual) rank; built once per (size, NB, grid) and kept on the device.
constexpr int kKeyLen = 9;
struct Plan {
  long key[kKeyLen] = {0};
  bool valid = false;
  std::vector<GemmTask> host;
  GemmTask* dev = nullptr;
  size_t dev_cap = 0;
  std::vector<Launch> la, bulkA, bulkB;           // per step
  std::vector<std::vector<Launch>> trsm;          // per step: GEMMs of the panel-solve recursion, in execution order
  std::vector<TrsmRows> rows;                     // per step: (block-cyclic) rows of the panel solve
  std::vector<int4> hblocks;                      // A phase: own Hessian blocks {bi, bc, e, 0}
  int4* dev_hblocks = nullptr;
  size_t dev_hblocks_cap = 0;
  Launch all;                                     // A phase: the single launch
};

struct DistState {
  ncclComm_t comm = nullptr;
  int rank = 0, world = 1;       // NCCL rank / size (world == 1 in virtual mode)
  int nv = 0;                    // > 0: virtual mode, nv ranks emulated on this GPU
  int P = 1, Q = 1;
  double* U = nullptr;           // M x ld, U = L^{-T} (clean: zeros below the diagonal)
  TMap2 mapU;
  double* Asub = nullptr;        // own sub-blocks of the interior inverse, NBH x NBH each
  int nbh = 0;
  double* gbuf = nullptr;        // panel gather staging
  double* dbuf = nullptr;        // diagonal-block staging
  double* dvec = nullptr;        // M doubles
  cudaStream_t sC = nullptr;     // communication stream of the U phase
  std::map<int, Plan> plans;     // key: phase * 4096 + virtual rank
  bool inverse_ready = false;
  int inv_pde = -1;              // PDE whose Hessian the sub-block plan of the last gpp_dist_inverse serves
  // peer-to-peer path (GPP_DIST_P2P=1): the replicated buffers of all ranks are mapped into every process (CUDA IPC);
  // finished blocks are stored straight into the peers' copies over NVLink by the solve kernel and announced by flags.
  // Measured on 8 B200 (profiles/r02b_dist8_*.log): 3.79 s per N=40k solve against 2.98 s with the NCCL all-gather --
  // every tile is written 7 times by the SMs of the kernel on the critical path, where NCCL's all-gather is not -- so
  // NCCL is the default and this path is an option.
  bool p2p = false;
  struct PeerMap { size_t cap = 0; double* peer[8] = {nullptr}; } pm[3];   // 0: Theta / L, 1: U, 2: H
  unsigned long long* flags = nullptr;          // [2][8] on this device: [kind][source rank], kind 0 panel, 1 diagonal block
  unsigned long long* peer_flags[8] = {nullptr};
  unsigned* push_counter = nullptr;             // [4]
  unsigned char* ipc_dev = nullptr;             // staging of the handle exchange
  unsigned long long seq = 0;                   // push sequence number, identical on all ranks
};

DistState* ds(gpp_handle* h) { return static_cast<DistState*>(h->dist); }

#define NCCL_TRY(h, expr)                                                      \
  do {                                                                         \
    ncclResult_t _r = (expr);                                                  \
    if (_r != ncclSuccess) {                                                   \
      (h)->err = std::string(#expr) + ": " + ncclGetErrorString(_r);           \
      return GPP_CUDA_ERR + 2;                                                 \
    }                                                                          \
  } while (0)

inline int nblocks_of(int n, int NB) { return (n + NB - 1) / NB; }
inline int rows_of(int n, int NB, int b) { return (n - b * NB < NB) ? (n - b * NB) : NB; }

std::vector<Grid> grids_of(const DistState* d) {
  std::vector<Grid> v;
  if (d->nv > 0) {
    for (int r = 0; r < d->nv; ++r) v.push_back(Grid{d->P, d->Q, r / d->Q, r % d->Q});
  } else {
    v.push_back(Grid{d->P, d->Q, d->rank / d->Q, d->rank % d->Q});
  }
  return v;
}

struct EventPool {
  gpp_handle* h;
  size_t used = 0;
  explicit EventPool(gpp_handle* hh) : h(hh) {}
  cudaEvent_t get() {
    if (used == h->evpool.size()) {
      cudaEvent_t e;
      cudaEventCreateWithFlags(&e, cudaEventDisableTiming);
      h->evpool.push_back(e);
    }
    return h->evpool[used++];
  }
};

// ---------------------------------------------------------------------------------------------------------
// small kernels
// ---------------------------------------------------------------------------------------------------------
__global__ void dist_get_diag_kernel(const double* __restrict__ T, long ld, int g0, int nrows, double* __restrict__ out) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < nrows) out[g0 + i] = T[(long)(g0 + i) * ld + g0 + i];
}
__global__ void dist_add_diag_kernel(double* __restrict__ T, long ld, int g0, int nrows, const double* __restrict__ add) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < nrows) T[(long)(g0 + i) * ld + g0 + i] += add[g0 + i];
}

// Panel staging.  Blocks (b, col), b in [b_lo, b_hi), of a replicated matrix X; the blocks of process row pr
// (b mod P == pr, ascending) occupy slots pr * cnt_max + t of the staging buffer, NB * NB doubles each, rows of w doubles.
struct PanelGeom {
  int NB, n, col0, w;        // block size, matrix size, first column of the panel, panel width
  int b_lo, b_hi, P, cnt_max;
};
__device__ __forceinline__ int panel_slot(const PanelGeom& g, int b) {
  const int pr = b % g.P;
  int first = g.b_lo + ((pr - g.b_lo % g.P) + g.P) % g.P;       // smallest b' >= b_lo with b' mod P == pr
  return pr * g.cnt_max + (b - first) / g.P;
}
// grid: (blocks to copy, NB / 8); 256 threads.  mode 0: pack blocks of process row `pr_sel`; mode 1: unpack all blocks
// except those of (pr_skip) when skip >= 0
__global__ void __launch_bounds__(256)
panel_copy_kernel(double* __restrict__ X, long ld, double* __restrict__ buf, const PanelGeom g, int mode, int pr_sel) {
  int b;
  if (mode == 0) {
    int first = g.b_lo + ((pr_sel - g.b_lo % g.P) + g.P) % g.P;
    b = first + blockIdx.x * g.P;
  } else {
    b = g.b_lo + blockIdx.x;
    if (pr_sel >= 0 && b % g.P == pr_sel) return;
  }
  if (b >= g.b_hi) return;
  const int rows = (g.n - b * g.NB < g.NB) ? (g.n - b * g.NB) : g.NB;
  double* sb = buf + (long)panel_slot(g, b) * g.NB * g.NB;
  for (int r = blockIdx.y * 8 + (threadIdx.x >> 5); r < rows; r += gridDim.y * 8) {
    double* xr = X + (long)(b * g.NB + r) * ld + g.col0;
    double* br = sb + (long)r * g.w;
    for (int c = threadIdx.x & 31; c < g.w; c += 32) {
      if (mode == 0) br[c] = xr[c];
      else xr[c] = br[c];
    }
  }
}

// ---- peer-to-peer push: copy a w-wide column strip of own rows (contiguous or block-cyclic) to the same place of every
// peer's buffer, then announce it.  grid.x CTAs, each warp a row at a time.
__global__ void __launch_bounds__(256)
push_rows_kernel(const double* __restrict__ X, long ld, const TrsmRows rm, int w, const __grid_constant__ PeerPush pp) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int r = blockIdx.x * 8 + warp; r < rm.rows; r += gridDim.x * 8) {
    const long pr = rm.stride_blk == 0 ? r : (long)(rm.first_blk + (r / rm.nb) * rm.stride_blk) * rm.nb + r % rm.nb;
    const double* src = X + pr * ld;
    for (int c = lane; c < w; c += 32) {
      const double v = src[c];
      for (int q = 0; q < pp.npeers; ++q) pp.base[q][pr * ld + c] = v;
    }
  }
  __threadfence_system();
  __syncthreads();
  if (threadIdx.x == 0) {
    const unsigned prev = atomicAdd(pp.counter, 1u);
    if (prev == gridDim.x - 1) {
      atomicExch(pp.counter, 0u);
      __threadfence_system();
      for (int q = 0; q < pp.npeers; ++q)
        asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(pp.flag[q]), "l"(pp.seq) : "memory");
    }
  }
}
// nothing to push at this step: only the announcement
__global__ void signal_kernel(const __grid_constant__ PeerPush pp) {
  if (threadIdx.x < pp.npeers) {
    __threadfence_system();
    asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(pp.flag[threadIdx.x]), "l"(pp.seq) : "memory");
  }
}
// wait until the flags of the sources in `mask` have reached seq (written by the peers' push kernels)
__global__ void wait_flags_kernel(const unsigned long long* __restrict__ flags, unsigned mask, unsigned long long seq) {
  const int r = threadIdx.x;
  if (r < 8 && ((mask >> r) & 1u)) {
    unsigned long long v;
    do {
      asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(flags + r) : "memory");
    } while (v < seq);
  }
  __syncthreads();
  __threadfence_system();
}

// ---------------------------------------------------------------------------------------------------------
// plans
// ---------------------------------------------------------------------------------------------------------
Plan& plan_slot(DistState* d, int phase, int vr) { return d->plans[phase * 4096 + vr]; }

bool plan_matches(Plan& pl, const long* key) {
  if (!pl.valid) return false;
  for (int k = 0; k < kKeyLen; ++k) if (pl.key[k] != key[k]) return false;
  return true;
}

void plan_reset(Plan& pl, const long* key) {
  for (int k = 0; k < kKeyLen; ++k) pl.key[k] = key[k];
  pl.host.clear(); pl.la.clear(); pl.bulkA.clear(); pl.bulkB.clear(); pl.trsm.clear(); pl.rows.clear(); pl.hblocks.clear();
  pl.all = Launch{};
  pl.valid = false;
}

int plan_upload(gpp_handle* h, Plan& pl) {
  if (pl.host.size() > pl.dev_cap) {
    if (pl.dev) cudaFree(pl.dev);
    pl.dev = nullptr;
    pl.dev_cap = pl.host.size() + pl.host.size() / 8 + 16;
    CUDA_TRY(h, cudaMalloc(&pl.dev, pl.dev_cap * sizeof(GemmTask)));
  }
  if (!pl.host.empty())
    CUDA_TRY(h, cudaMemcpyAsync(pl.dev, pl.host.data(), pl.host.size() * sizeof(GemmTask), cudaMemcpyHostToDevice, h->stream));
  if (pl.hblocks.size() > pl.dev_hblocks_cap) {
    if (pl.dev_hblocks) cudaFree(pl.dev_hblocks);
    pl.dev_hblocks = nullptr;
    pl.dev_hblocks_cap = pl.hblocks.size() + 16;
    CUDA_TRY(h, cudaMalloc(&pl.dev_hblocks, pl.dev_hblocks_cap * sizeof(int4)));
  }
  if (!pl.hblocks.empty())
    CUDA_TRY(h, cudaMemcpyAsync(pl.dev_hblocks, pl.hblocks.data(), pl.hblocks.size() * sizeof(int4), cudaMemcpyHostToDevice, h->stream));
  CUDA_TRY(h, cudaStreamSynchronize(h->stream));     // the host vectors may be rebuilt later
  pl.valid = true;
  return GPP_OK;
}

GemmTask make_task(int a_row, int b_row, int c_row, int c_col, int m, int n, int k0, int k1, int kb_off, int tri) {
  GemmTask t{};
  t.a_row = a_row; t.b_row = b_row; t.c_row = c_row; t.c_col = c_col;
  t.m = m; t.n = n; t.k0 = k0; t.k1 = k1; t.kb_off = kb_off; t.tri = tri;
  return t;
}

// GEMMs of the recursive panel solve X L^T = P (mirrors trsm_right_lt in chol.cu) over the row blocks `blks`
// (physical block indices, `brows` rows each); panel columns [pc0, pc0 + nb), L block at (lr0, lc0) of the L operand.
void plan_trsm(Plan& pl, std::vector<Launch>& out, const std::vector<int>& blks, const std::vector<int>& brows, int NB,
               int pc0, int lr0, int lc0, int nb) {
  if (nb <= 64 || blks.empty()) return;
  const int hh = (int)round_up((nb + 1) / 2, 64);
  plan_trsm(pl, out, blks, brows, NB, pc0, lr0, lc0, hh);
  Launch l;
  l.off = pl.host.size(); l.count = (int)blks.size();
  for (size_t t = 0; t < blks.size(); ++t)
    pl.host.push_back(make_task(blks[t] * NB, lr0 + hh, blks[t] * NB, pc0 + hh, brows[t], nb - hh, pc0, pc0 + hh, lc0 - pc0, 0));
  out.push_back(l);
  plan_trsm(pl, out, blks, brows, NB, pc0 + hh, lr0 + hh, lc0 + hh, nb - hh);
}

TrsmRows rows_of_blocks(const std::vector<int>& blks, const std::vector<int>& brows, int NB, int stride) {
  TrsmRows r{0, 0, 0, NB};
  if (blks.empty()) return r;
  r.first_blk = blks[0];
  r.stride_blk = stride;
  r.rows = (int)(blks.size() - 1) * NB + brows.back();
  return r;
}

// right-looking Cholesky of an n x n matrix, block size NB, for the rank at g
void build_potrf_plan(Plan& pl, const Grid& g, int n, int NB) {
  const int nblk = nblocks_of(n, NB);
  pl.la.assign(nblk, Launch{}); pl.bulkA.assign(nblk, Launch{}); pl.bulkB.assign(nblk, Launch{});
  pl.trsm.assign(nblk, {}); pl.rows.assign(nblk, TrsmRows{0, 0, 0, NB});
  for (int j = 0; j < nblk; ++j) {
    const int j0 = j * NB, nbj = rows_of(n, NB, j);
    std::vector<int> blks, brows;
    if (j % g.Q == g.q)
      for (int bi = j + 1; bi < nblk; ++bi)
        if (bi % g.P == g.p) { blks.push_back(bi); brows.push_back(rows_of(n, NB, bi)); }
    pl.rows[j] = rows_of_blocks(blks, brows, NB, g.P);
    plan_trsm(pl, pl.trsm[j], blks, brows, NB, j0, j0, j0, nbj);
    auto emit = [&](Launch& l, int c_lo, int c_hi) {       // own blocks (bi, bc), c_lo <= bc < c_hi, bc <= bi
      l.off = pl.host.size();
      for (int bc = c_lo; bc < c_hi && bc < nblk; ++bc)
        for (int bi = bc; bi < nblk; ++bi)
          if (mine(g, bi, bc))
            pl.host.push_back(make_task(bi * NB, bc * NB, bi * NB, bc * NB, rows_of(n, NB, bi), rows_of(n, NB, bc), j0, j0 + nbj, 0, bi == bc));
      l.count = (int)(pl.host.size() - l.off);
    };
    emit(pl.la[j], j + 1, j + 2);
    emit(pl.bulkA[j], j + 2, j + 3);
    emit(pl.bulkB[j], j + 3, nblk);
  }
}

// U = L^{-T}: at step i the blocks (b, i), b <= i, are solved; then (b, c), b <= i < c, receive -U(b, i) L(c, i)^T
void build_uinv_plan(Plan& pl, const Grid& g, int n, int NB) {
  const int nblk = nblocks_of(n, NB);
  pl.la.assign(nblk, Launch{}); pl.bulkA.assign(nblk, Launch{}); pl.bulkB.assign(nblk, Launch{});
  pl.trsm.assign(nblk, {}); pl.rows.assign(nblk, TrsmRows{0, 0, 0, NB});
  for (int i = 0; i < nblk; ++i) {
    const int i0 = i * NB, nbi = rows_of(n, NB, i);
    std::vector<int> blks, brows;
    if (i % g.Q == g.q)
      for (int b = 0; b <= i; ++b)
        if (b % g.P == g.p) { blks.push_back(b); brows.push_back(rows_of(n, NB, b)); }
    pl.rows[i] = rows_of_blocks(blks, brows, NB, g.P);
    plan_trsm(pl, pl.trsm[i], blks, brows, NB, i0, i0, i0, nbi);
    auto emit = [&](Launch& l, int c_lo, int c_hi) {
      l.off = pl.host.size();
      for (int c = c_lo; c < c_hi && c < nblk; ++c)
        for (int b = 0; b <= i; ++b)
          if (mine(g, b, c))
            pl.host.push_back(make_task(b * NB, c * NB, b * NB, c * NB, rows_of(n, NB, b), rows_of(n, NB, c), i0, i0 + nbi, 0, 0));
      l.count = (int)(pl.host.size() - l.off);
    };
    emit(pl.la[i], i + 1, i + 2);
    emit(pl.bulkA[i], i + 2, i + 3);
    emit(pl.bulkB[i], i + 3, nblk);
  }
}

// PDEs whose Hessian the sharded GN step assembles, by the layout of their (single) Gram system; -1: not sharded
int sharded_pde_of_layout(int layout) {
  switch (layout) {
    case LAY_ELLIPTIC: return PDE_ELLIPTIC;
    case LAY_BURGERS: return PDE_BURGERS;
    case LAY_EIKONAL: return PDE_EIKONAL;
    default: return -1;
  }
}

// Rows [b NB, b NB + NB) of the nz N x nz N Hessian cut where the unknown field changes: field q, first index i0 within
// the field, first row r0 within the block, length len.  A block straddles a field boundary when N % NB != 0.
struct Seg { int q, i0, r0, len; };
std::vector<Seg> field_segments(int b, int NB, int n, int N) {
  std::vector<Seg> v;
  const int g0 = b * NB, g1 = std::min(g0 + NB, n);
  for (int r = g0; r < g1;) {
    const int q = r / N, e = std::min(g1, (q + 1) * N);
    v.push_back(Seg{q, r - q * N, r - g0, e - r});
    r = e;
  }
  return v;
}

// sub-blocks of the interior inverse needed by the own Hessian blocks: for every pair of field segments of an own block
// and every term t = (p, p') of their pair (q, q'), A_pp'(i, j) = sum_k U[off[p] + i, k] U[off[p'] + j, k] lands in slot t
// (of four) of the block's group in the compact store.  Every pair of elliptic, Burgers and Eikonal has at most four terms.
// Elliptic (one field, four terms everywhere) gives exactly one task per (block, p, p').
void build_ablock_plan(Plan& pl, const Grid& g, const TermTable& tt, int N, int M, const int* off, int nbh) {
  const int n = tt.nz * N, nblk = nblocks_of(n, nbh);
  for (int bi = 0; bi < nblk; ++bi)
    for (int bc = 0; bc <= bi; ++bc)
      if (mine(g, bi, bc)) pl.hblocks.push_back(make_int4(bi, bc, (int)pl.hblocks.size(), 0));
  pl.all.off = 0;
  const int k1 = (int)round_up(M, 16);
  for (const int4& hb : pl.hblocks) {
    const std::vector<Seg> rs = field_segments(hb.x, nbh, n, N), cs = field_segments(hb.y, nbh, n, N);
    for (const Seg& a : rs)
      for (const Seg& b : cs) {
        const int pr = a.q * tt.nz + b.q;
        for (int t = 0; t < tt.nterms[pr]; ++t) {
          const int a_row = off[tt.tp[pr][t]] + a.i0, b_row = off[tt.tpp[pr][t]] + b.i0;
          const int k0 = (std::max(a_row, b_row) / 16) * 16;      // U is upper triangular
          pl.host.push_back(make_task(a_row, b_row, (hb.z * 4 + t) * nbh + a.r0, b.r0, a.len, b.len, k0, k1, 0, 0));
        }
      }
  }
  // longest K first: the hardware scheduler then balances the variable-length tiles
  std::stable_sort(pl.host.begin(), pl.host.end(), [](const GemmTask& a, const GemmTask& b) { return (a.k1 - a.k0) > (b.k1 - b.k0); });
  pl.all.count = (int)pl.host.size();
}

// phase 2: n = N_domain, extraM = M, off = the layout's row offsets, pde = the sharded PDE of that layout (else -1)
int ensure_plan(gpp_handle* h, DistState* d, int phase, int vr, const Grid& g, int n, int NB, int extraM, const int* off, int pde,
                Plan** out) {
  Plan& pl = plan_slot(d, phase, vr);
  const long key[kKeyLen] = {phase, n, NB, g.P, g.Q, g.p * 65536L + g.q, extraM, off ? off[1] : 0, pde};
  if (!plan_matches(pl, key)) {
    plan_reset(pl, key);
    if (phase == 0 || phase == 3) {
      build_potrf_plan(pl, g, n, NB);
    } else if (phase == 1) {
      build_uinv_plan(pl, g, n, NB);
    } else {
      TermTable tt;
      if (make_term_table(pde, &tt) || tt.nslots != 1) { h->err = "sub-block plan: PDE not sharded"; return -1; }
      build_ablock_plan(pl, g, tt, n, extraM, off, NB);
    }
    int rc = plan_upload(h, pl);
    if (rc) return rc;
  }
  *out = &pl;
  return GPP_OK;
}

// ---------------------------------------------------------------------------------------------------------
// execution helpers (all on h->cur)
// ---------------------------------------------------------------------------------------------------------
struct MatRef { double* base; long ld; const TMap2* map; };

int run_tasks(gpp_handle* h, const Plan& pl, const Launch& l, const MatRef& A, const MatRef& B, const MatRef& C, int bs, double alpha, bool accumulate) {
  if (l.count <= 0) return GPP_OK;
  GemmTaskDesc d{};
  d.mapA = A.map; d.mapB = B.map;
  d.C = C.base; d.ldc = C.ld;
  d.Cin = accumulate ? C.base : nullptr; d.ldcin = C.ld;
  d.alpha = alpha;
  d.tasks = pl.dev + l.off; d.ntasks = l.count; d.bs = bs;
  d.blocksum = (accumulate && h->blocksum) ? 1 : 0;
  return gemm_tasks_launch(h, d);
}

// recursive panel solve over block-cyclic rows (mirrors trsm_right_lt); consumes the planned GEMMs in order
int exec_trsm(gpp_handle* h, const Plan& pl, const std::vector<Launch>& gemms, size_t& next, const TrsmRows& rm, const MatRef& Pm, int pc0,
              const MatRef& Lm, int lr0, int lc0, int nb, int NB) {
  if (rm.rows <= 0 || nb <= 0) return GPP_OK;
  if (nb <= 64) return trsm_base_launch(h, Pm.base + pc0, Pm.ld, rm, Lm.base + (long)lr0 * Lm.ld + lc0, Lm.ld, nb);
  const int hh = (int)round_up((nb + 1) / 2, 64);
  int rc = exec_trsm(h, pl, gemms, next, rm, Pm, pc0, Lm, lr0, lc0, hh, NB);
  if (rc) return rc;
  if (next >= gemms.size()) { h->err = "panel-solve plan exhausted"; return -1; }
  rc = run_tasks(h, pl, gemms[next++], Pm, Lm, Pm, NB, -1.0, true);
  if (rc) return rc;
  return exec_trsm(h, pl, gemms, next, rm, Pm, pc0 + hh, Lm, lr0 + hh, lc0 + hh, nb - hh, NB);
}

PanelGeom panel_geom(const DistState* d, int n, int NB, int col, int b_lo, int b_hi) {
  PanelGeom g;
  g.NB = NB; g.n = n; g.col0 = col * NB; g.w = rows_of(n, NB, col);
  g.b_lo = b_lo; g.b_hi = b_hi; g.P = d->P;
  g.cnt_max = (b_hi - b_lo + d->P - 1) / d->P;
  return g;
}

// blocks (b, col), b in [b_lo, b_hi), are final on their owners: make them so on every rank (on stream st)
int gather_panel(gpp_handle* h, DistState* d, double* X, long ld, int n, int NB, int col, int b_lo, int b_hi, cudaStream_t st) {
  if (d->world <= 1 || b_hi <= b_lo) return GPP_OK;
  const PanelGeom g = panel_geom(d, n, NB, col, b_lo, b_hi);
  const int myp = d->rank / d->Q, myq = d->rank % d->Q, cq = col % d->Q;
  const size_t slot = (size_t)NB * NB;
  dim3 blk(256);
  if (myq == cq) {
    const int first = b_lo + ((myp - b_lo % d->P) + d->P) % d->P;
    const int cnt = first < b_hi ? (b_hi - first + d->P - 1) / d->P : 0;
    if (cnt > 0) {
      panel_copy_kernel<<<dim3(cnt, NB / 64), blk, 0, st>>>(X, ld, d->gbuf, g, 0, myp);
      h->launches++;
    }
  }
  if (d->Q == 1) {
    NCCL_TRY(h, ncclAllGather(d->gbuf + (size_t)d->rank * g.cnt_max * slot, d->gbuf, (size_t)g.cnt_max * slot, ncclDouble, d->comm, st));
  } else {
    NCCL_TRY(h, ncclGroupStart());
    for (int pr = 0; pr < d->P; ++pr) {
      const int first = b_lo + ((pr - b_lo % d->P) + d->P) % d->P;
      const int cnt = first < b_hi ? (b_hi - first + d->P - 1) / d->P : 0;
      if (cnt <= 0) continue;
      double* reg = d->gbuf + (size_t)pr * g.cnt_max * slot;
      NCCL_TRY(h, ncclBroadcast(reg, reg, (size_t)cnt * slot, ncclDouble, pr * d->Q + cq, d->comm, st));
    }
    NCCL_TRY(h, ncclGroupEnd());
  }
  panel_copy_kernel<<<dim3(b_hi - b_lo, NB / 64), blk, 0, st>>>(X, ld, d->gbuf, g, 1, myq == cq ? myp : -1);
  h->launches++;
  CUDA_TRY(h, cudaGetLastError());
  return GPP_OK;
}

// diagonal block (j, j) is final on its owner: broadcast it (on stream st)
int bcast_diag(gpp_handle* h, DistState* d, double* X, long ld, int n, int NB, int j, cudaStream_t st) {
  if (d->world <= 1) return GPP_OK;
  const Grid g{d->P, d->Q, d->rank / d->Q, d->rank % d->Q};
  const int j0 = j * NB, w = rows_of(n, NB, j), root = owner_of(g, j, j);
  double* blk = X + (long)j0 * ld + j0;
  if (d->rank == root)
    CUDA_TRY(h, cudaMemcpy2DAsync(d->dbuf, (size_t)w * 8, blk, ld * 8, (size_t)w * 8, w, cudaMemcpyDeviceToDevice, st));
  NCCL_TRY(h, ncclBroadcast(d->dbuf, d->dbuf, (size_t)w * w, ncclDouble, root, d->comm, st));
  if (d->rank != root)
    CUDA_TRY(h, cudaMemcpy2DAsync(blk, ld * 8, d->dbuf, (size_t)w * 8, (size_t)w * 8, w, cudaMemcpyDeviceToDevice, st));
  return GPP_OK;
}

int ensure_staging(gpp_handle* h, DistState* d, int n, int NB) {
  if (d->world <= 1) return GPP_OK;       // nothing travels
  const int nblk = nblocks_of(n, NB);
  int rc = dev_reserve(h, &d->gbuf, (size_t)(nblk + d->P) * NB * NB);
  if (rc) return rc;
  return dev_reserve(h, &d->dbuf, (size_t)NB * NB);
}

// ---------------------------------------------------------------------------------------------------------
// peer-to-peer plumbing
// ---------------------------------------------------------------------------------------------------------
// exchange the CUDA IPC handle of `base` (an allocation start) with all ranks and map the peers' allocations
int ipc_exchange(gpp_handle* h, DistState* d, void* base, void** peer_out) {
  cudaIpcMemHandle_t mine;
  CUDA_TRY(h, cudaIpcGetMemHandle(&mine, base));
  static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle is 64 bytes");
  if (!d->ipc_dev) CUDA_TRY(h, cudaMalloc(&d->ipc_dev, 8 * 64));
  cudaStream_t S = h->stream;
  CUDA_TRY(h, cudaMemcpyAsync(d->ipc_dev + 64 * d->rank, &mine, 64, cudaMemcpyHostToDevice, S));
  NCCL_TRY(h, ncclAllGather(d->ipc_dev + 64 * d->rank, d->ipc_dev, 64, ncclChar, d->comm, S));
  cudaIpcMemHandle_t all[8];
  CUDA_TRY(h, cudaMemcpyAsync(all, d->ipc_dev, 64 * d->world, cudaMemcpyDeviceToHost, S));
  CUDA_TRY(h, cudaStreamSynchronize(S));
  for (int r = 0; r < d->world; ++r) {
    if (r == d->rank) { peer_out[r] = base; continue; }
    CUDA_TRY(h, cudaIpcOpenMemHandle(&peer_out[r], all[r], cudaIpcMemLazyEnablePeerAccess));
  }
  return GPP_OK;
}

bool use_p2p(const DistState* d) { return d->p2p && d->world > 1 && d->world <= 8 && d->nv == 0; }

// (re)map replicated buffer `which` after it was (re)allocated; `cap` is its capacity, which changes on every rank at
// the same call (identical sizes), so the exchange stays collective
int share_buffer(gpp_handle* h, DistState* d, int which, double* base, size_t cap) {
  if (!use_p2p(d)) return GPP_OK;
  DistState::PeerMap& pm = d->pm[which];
  if (pm.cap == cap && pm.peer[d->rank] == base) return GPP_OK;
  for (int r = 0; r < d->world; ++r) {
    if (r != d->rank && pm.peer[r]) cudaIpcCloseMemHandle(pm.peer[r]);
    pm.peer[r] = nullptr;
  }
  void* peers[8] = {nullptr};
  int rc = ipc_exchange(h, d, base, peers);
  if (rc) return rc;
  for (int r = 0; r < d->world; ++r) pm.peer[r] = static_cast<double*>(peers[r]);
  pm.cap = cap;
  return GPP_OK;
}

int init_p2p(gpp_handle* h, DistState* d) {
  if (!use_p2p(d)) return GPP_OK;
  CUDA_TRY(h, cudaMalloc(&d->flags, 16 * sizeof(unsigned long long)));
  CUDA_TRY(h, cudaMemset(d->flags, 0, 16 * sizeof(unsigned long long)));
  CUDA_TRY(h, cudaMalloc(&d->push_counter, 4 * sizeof(unsigned)));
  CUDA_TRY(h, cudaMemset(d->push_counter, 0, 4 * sizeof(unsigned)));
  void* peers[8] = {nullptr};
  int rc = ipc_exchange(h, d, d->flags, peers);
  if (rc) return rc;
  for (int r = 0; r < d->world; ++r) d->peer_flags[r] = static_cast<unsigned long long*>(peers[r]);
  return GPP_OK;
}

// push descriptor for a kernel whose output origin is `local_ptr` inside replicated buffer `which`
PeerPush make_push(DistState* d, int which, const double* local_ptr, int kind, unsigned long long seq) {
  PeerPush pp{};
  const DistState::PeerMap& pm = d->pm[which];
  const long off = local_ptr - pm.peer[d->rank];
  for (int r = 0; r < d->world; ++r) {
    if (r == d->rank) continue;
    pp.base[pp.npeers] = pm.peer[r] + off;
    pp.flag[pp.npeers] = d->peer_flags[r] + kind * 8 + d->rank;
    ++pp.npeers;
  }
  pp.seq = seq;
  pp.counter = d->push_counter + kind;
  return pp;
}

int push_rows(gpp_handle* h, const double* X, long ld, const TrsmRows& rm, int w, const PeerPush& pp, cudaStream_t st) {
  if (rm.rows <= 0 || w <= 0) {
    signal_kernel<<<1, 32, 0, st>>>(pp);
  } else {
    int grid = (rm.rows + 7) / 8;
    if (grid > 296) grid = 296;
    push_rows_kernel<<<grid, 256, 0, st>>>(X, ld, rm, w, pp);
  }
  h->launches++;
  CUDA_TRY(h, cudaGetLastError());
  return GPP_OK;
}

int wait_flags(gpp_handle* h, DistState* d, int kind, int root, unsigned long long seq, cudaStream_t st) {
  unsigned mask = 0;
  for (int r = 0; r < d->world; ++r)
    if (r != d->rank && (root < 0 || r == root)) mask |= 1u << r;
  if (!mask) return GPP_OK;
  wait_flags_kernel<<<1, 32, 0, st>>>(d->flags + kind * 8, mask, seq);
  h->launches++;
  CUDA_TRY(h, cudaGetLastError());
  return GPP_OK;
}

// ---------------------------------------------------------------------------------------------------------
// distributed right-looking Cholesky of the replicated n x n matrix A (Theta in slot 0, or the GN Hessian)
// ---------------------------------------------------------------------------------------------------------
// all ranks have finished whatever they enqueued before: one-sided pushes into their buffers may start
int phase_barrier(gpp_handle* h, DistState* d) {
  if (!use_p2p(d)) return GPP_OK;
  NCCL_TRY(h, ncclAllReduce(d->push_counter + 3, d->push_counter + 3, 1, ncclUint32, ncclSum, d->comm, h->stream));
  return GPP_OK;
}

int dist_potrf_matrix(gpp_handle* h, DistState* d, double* A, long ld, int n, const TMap2* map, int phase, bool want_info, int* info,
                      size_t cap) {
  const int NB = h->NB;
  const int which = (phase == 3) ? 2 : 0;
  const bool p2p = use_p2p(d);
  if (p2p) {
    int rcs = share_buffer(h, d, which, A, cap);
    if (!rcs) rcs = phase_barrier(h, d);
    if (rcs) return rcs;
  }
  const int nblk = nblocks_of(n, NB);
  const MatRef Am{A, ld, map};
  const std::vector<Grid> grids = grids_of(d);
  std::vector<Plan*> plans(grids.size());
  for (size_t v = 0; v < grids.size(); ++v) {
    int rc = ensure_plan(h, d, phase, d->nv > 0 ? (int)v : 0, grids[v], n, NB, 0, nullptr, -1, &plans[v]);
    if (rc) return rc;
  }
  int rc = ensure_staging(h, d, n, NB);
  if (rc) return rc;
  cudaStream_t S = h->stream;
  CUDA_TRY(h, cudaMemsetAsync(h->d_info, 0, sizeof(int), S));
  const Mat Amat{A, ld, map};

  auto panel_factor = [&](const Grid& g, int j) -> int {       // diagonal factorisation on its owner
    if (owner_of(g, j, j) != g.p * g.Q + g.q) return GPP_OK;
    return potrf_diag(h, Amat, j * NB, j * NB, rows_of(n, NB, j), j * NB);
  };
  auto panel_solve = [&](const Plan& pl, int j) -> int {
    if (pl.rows[j].rows <= h->fused_trsm_rows)      // one launch; the recursion pays ~15 launches under SM contention
      return trsm_panel_launch(h, A + (long)j * NB, ld, pl.rows[j], A + (long)j * NB * ld + (long)j * NB, ld, rows_of(n, NB, j));
    size_t next = 0;
    return exec_trsm(h, pl, pl.trsm[j], next, pl.rows[j], Am, j * NB, Am, j * NB, j * NB, rows_of(n, NB, j), NB);
  };

  if (d->nv > 0) {
    // virtual ranks, one stream: per step every rank's share in turn (storage is shared, so no exchange)
    h->cur = S;
    for (int j = 0; j < nblk && !rc; ++j) {
      for (size_t v = 0; v < grids.size() && !rc; ++v) rc = panel_factor(grids[v], j);
      for (size_t v = 0; v < grids.size() && !rc; ++v) rc = panel_solve(*plans[v], j);
      for (size_t v = 0; v < grids.size() && !rc; ++v) {
        const Plan& pl = *plans[v];
        rc = run_tasks(h, pl, pl.la[j], Am, Am, Am, NB, -1.0, true);
        if (!rc) rc = run_tasks(h, pl, pl.bulkA[j], Am, Am, Am, NB, -1.0, true);
        if (!rc) rc = run_tasks(h, pl, pl.bulkB[j], Am, Am, Am, NB, -1.0, true);
      }
    }
    if (rc) return rc;
  } else {
    const Grid& g = grids[0];
    const Plan& pl = *plans[0];
    cudaStream_t Sp = h->sP, Sb = h->sG[0];
    EventPool ev(h);
    cudaEvent_t ev0 = ev.get();
    CUDA_TRY(h, cudaEventRecord(ev0, S));
    CUDA_TRY(h, cudaStreamWaitEvent(Sp, ev0, 0));
    CUDA_TRY(h, cudaStreamWaitEvent(Sb, ev0, 0));
    std::vector<cudaEvent_t> ev_panel(nblk), ev_a(nblk);
    // GPP_TRACE: timed events around the pieces of the panel chain of every 16th column (Sp is the critical path once
    // the bulk of a step is shorter than the chain)
    static const bool trace = getenv("GPP_TRACE") != nullptr;
    struct ChainEv { int j; cudaEvent_t e[6]; };
    std::vector<ChainEv> chain;
    auto tmark = [&](ChainEv* c, int k) { if (c) { cudaEventCreate(&c->e[k]); cudaEventRecord(c->e[k], Sp); } };
    ChainEv* cur_chain = nullptr;
    auto panel = [&](int j) -> int {          // on Sp: factorise, broadcast, solve, gather column j
      h->cur = Sp;
      tmark(cur_chain, 1);
      int r = panel_factor(g, j);
      tmark(cur_chain, 2);
      const int j0 = j * NB, w = rows_of(n, NB, j);
      double* diag = A + (long)j0 * ld + j0;
      if (!p2p) {
        if (!r) r = bcast_diag(h, d, A, ld, n, NB, j, Sp);
        tmark(cur_chain, 3);
        if (!r) r = panel_solve(pl, j);
        tmark(cur_chain, 4);
        if (!r) r = gather_panel(h, d, A, ld, n, NB, j, j + 1, nblk, Sp);
        tmark(cur_chain, 5);
        return r;
      }
      // peer-to-peer: the owner stores the factored diagonal block into every peer's copy; the panel solve stores each
      // solved tile into every peer's copy as it goes (the gather is part of the kernel); flags announce completion
      const int root = owner_of(g, j, j);
      const unsigned long long sd = ++d->seq;
      if (!r) {
        if (d->rank == root) {
          const TrsmRows dr{w, 0, 0, 0};
          r = push_rows(h, diag, ld, dr, w, make_push(d, which, diag, 1, sd), Sp);
        } else {
          r = wait_flags(h, d, 1, root, sd, Sp);
        }
      }
      tmark(cur_chain, 3);
      if (j + 1 < nblk && !r) {
        const unsigned long long sp = ++d->seq;
        const TrsmRows& rm = pl.rows[j];
        double* Pcol = A + j0;
        const PeerPush pp = make_push(d, which, Pcol, 0, sp);
        if (rm.rows > 0 && rm.rows <= h->fused_trsm_rows) {
          r = trsm_panel_launch(h, Pcol, ld, rm, diag, ld, w, &pp);
        } else {
          if (rm.rows > 0) r = panel_solve(pl, j);
          if (!r) r = push_rows(h, Pcol, ld, rm, w, pp, Sp);
        }
        tmark(cur_chain, 4);
        if (!r) r = wait_flags(h, d, 0, -1, sp, Sp);
      } else {
        tmark(cur_chain, 4);
      }
      tmark(cur_chain, 5);
      return r;
    };
    rc = panel(0);
    for (int j = 0; j < nblk && !rc; ++j) {
      ev_panel[j] = ev.get();
      CUDA_TRY(h, cudaEventRecord(ev_panel[j], Sp));
      if (j + 1 < nblk) {
        // look-ahead: column j+1 first (it has all updates of the panels < j once bulkA(j-1) is done), then its panel chain
        if (j >= 1) CUDA_TRY(h, cudaStreamWaitEvent(Sp, ev_a[j - 1], 0));
        h->cur = Sp;
        cur_chain = nullptr;
        if (trace && d->rank == 0 && (j + 1) % 16 == 0) { chain.push_back(ChainEv{j + 1, {}}); cur_chain = &chain.back(); }
        tmark(cur_chain, 0);
        rc = run_tasks(h, pl, pl.la[j], Am, Am, Am, NB, -1.0, true);
        if (!rc) rc = panel(j + 1);
        cur_chain = nullptr;
        if (rc) break;
      }
      CUDA_TRY(h, cudaStreamWaitEvent(Sb, ev_panel[j], 0));
      h->cur = Sb;
      rc = run_tasks(h, pl, pl.bulkA[j], Am, Am, Am, NB, -1.0, true);
      ev_a[j] = ev.get();
      CUDA_TRY(h, cudaEventRecord(ev_a[j], Sb));
      if (!rc) rc = run_tasks(h, pl, pl.bulkB[j], Am, Am, Am, NB, -1.0, true);
    }
    h->cur = S;
    if (rc) return rc;
    cudaEvent_t e1 = ev.get(), e2 = ev.get();
    CUDA_TRY(h, cudaEventRecord(e1, Sp));
    CUDA_TRY(h, cudaEventRecord(e2, Sb));
    CUDA_TRY(h, cudaStreamWaitEvent(S, e1, 0));
    CUDA_TRY(h, cudaStreamWaitEvent(S, e2, 0));
    if (!chain.empty()) {
      cudaStreamSynchronize(S);
      for (ChainEv& c : chain) {
        float t[5];
        for (int k = 0; k < 5; ++k) cudaEventElapsedTime(&t[k], c.e[k], c.e[k + 1]);
        fprintf(stderr, "[gpp trace] panel chain n=%d column %d/%d: look-ahead update %.3f ms | diag potrf %.3f | diag bcast %.3f | panel solve %.3f | gather %.3f\n",
                n, c.j, nblk, t[0], t[1], t[2], t[3], t[4]);
        for (int k = 0; k < 6; ++k) cudaEventDestroy(c.e[k]);
      }
    }
  }
  h->cur = S;
  if (want_info) {
    if (d->world > 1) NCCL_TRY(h, ncclAllReduce(h->d_info, h->d_info, 1, ncclInt, ncclMax, d->comm, S));
    int hinfo = 0;
    CUDA_TRY(h, cudaMemcpyAsync(&hinfo, h->d_info, sizeof(int), cudaMemcpyDeviceToHost, S));
    CUDA_TRY(h, cudaStreamSynchronize(S));
    if (info) *info = hinfo;
  }
  return GPP_OK;
}

// ---------------------------------------------------------------------------------------------------------
// U = L^{-T} into the clean replicated buffer d->U
// ---------------------------------------------------------------------------------------------------------
int dist_uinv(gpp_handle* h, DistState* d, GramSlot& s) {
  const int NB = h->NB, n = s.M;
  const int nblk = nblocks_of(n, NB);
  const MatRef Um{d->U, s.ld, &d->mapU}, Tm{s.T, s.ld, &s.mapT};
  const std::vector<Grid> grids = grids_of(d);
  std::vector<Plan*> plans(grids.size());
  for (size_t v = 0; v < grids.size(); ++v) {
    int rc = ensure_plan(h, d, 1, d->nv > 0 ? (int)v : 0, grids[v], n, NB, 0, nullptr, -1, &plans[v]);
    if (rc) return rc;
  }
  int rc = ensure_staging(h, d, n, NB);
  if (rc) return rc;
  cudaStream_t S = h->stream;
  const bool p2p = use_p2p(d);
  if (p2p) {
    rc = share_buffer(h, d, 1, d->U, h->caps.count(&d->U) ? h->caps[&d->U] : 0);
    if (!rc) rc = phase_barrier(h, d);
    if (rc) return rc;
  }
  CUDA_TRY(h, cudaMemsetAsync(d->U, 0, sizeof(double) * (size_t)n * s.ld, S));
  if (p2p) {
    // nobody may push into this rank's U before its memset has run: second barrier, after the memset
    rc = phase_barrier(h, d);
    if (rc) return rc;
  }
  unsigned long long last_seq = 0;

  auto panel_solve = [&](const Grid& g, const Plan& pl, int i) -> int {     // on h->cur
    const int i0 = i * NB, nbi = rows_of(n, NB, i);
    int r = GPP_OK;
    if (owner_of(g, i, i) == g.p * g.Q + g.q) r = fill_identity_launch(h, d->U + (long)i0 * s.ld + i0, s.ld, nbi, nbi);
    if (r) return r;
    const TrsmRows& rm = pl.rows[i];
    if (p2p) {
      // every finished column of U goes straight into the peers' copies (all of U is needed by every rank afterwards)
      last_seq = ++d->seq;
      const PeerPush pp = make_push(d, 1, d->U + i0, 0, last_seq);
      if (rm.rows > 0 && rm.rows <= h->fused_trsm_rows)
        return trsm_panel_launch(h, d->U + i0, s.ld, rm, s.T + (long)i0 * s.ld + i0, s.ld, nbi, &pp);
      if (rm.rows > 0) {
        size_t next = 0;
        r = exec_trsm(h, pl, pl.trsm[i], next, rm, Um, i0, Tm, i0, i0, nbi, NB);
        if (r) return r;
      }
      return push_rows(h, d->U + i0, s.ld, rm, nbi, pp, h->cur);
    }
    if (rm.rows <= h->fused_trsm_rows)
      return trsm_panel_launch(h, d->U + i0, s.ld, rm, s.T + (long)i0 * s.ld + i0, s.ld, nbi);
    size_t next = 0;
    return exec_trsm(h, pl, pl.trsm[i], next, rm, Um, i0, Tm, i0, i0, nbi, NB);
  };

  if (d->nv > 0) {
    h->cur = S;
    for (int i = 0; i < nblk && !rc; ++i) {
      for (size_t v = 0; v < grids.size() && !rc; ++v) rc = panel_solve(grids[v], *plans[v], i);
      for (size_t v = 0; v < grids.size() && !rc; ++v) {
        const Plan& pl = *plans[v];
        rc = run_tasks(h, pl, pl.la[i], Um, Tm, Um, NB, -1.0, true);
        if (!rc) rc = run_tasks(h, pl, pl.bulkA[i], Um, Tm, Um, NB, -1.0, true);
        if (!rc) rc = run_tasks(h, pl, pl.bulkB[i], Um, Tm, Um, NB, -1.0, true);
      }
    }
    return rc;
  }
  const Grid& g = grids[0];
  const Plan& pl = *plans[0];
  cudaStream_t Sp = h->sP, Sb = h->sG[0], Sc = d->sC;
  EventPool ev(h);
  cudaEvent_t ev0 = ev.get();
  CUDA_TRY(h, cudaEventRecord(ev0, S));
  CUDA_TRY(h, cudaStreamWaitEvent(Sp, ev0, 0));
  CUDA_TRY(h, cudaStreamWaitEvent(Sb, ev0, 0));
  CUDA_TRY(h, cudaStreamWaitEvent(Sc, ev0, 0));
  std::vector<cudaEvent_t> ev_panel(nblk), ev_a(nblk);
  auto panel = [&](int i) -> int {
    h->cur = Sp;
    int r = panel_solve(g, pl, i);
    if (r) return r;
    if (p2p) {
      // Q > 1: the other process columns need U(b, i) for their updates, wait for the pushes; Q = 1: own rows only
      if (d->Q > 1) r = wait_flags(h, d, 0, -1, last_seq, Sp);
      ev_panel[i] = ev.get();
      CUDA_TRY(h, cudaEventRecord(ev_panel[i], Sp));
    } else if (d->Q > 1) {
      // the other process columns need U(b, i) for their updates: gather on the critical path
      r = gather_panel(h, d, d->U, s.ld, n, NB, i, 0, i + 1, Sp);
      ev_panel[i] = ev.get();
      CUDA_TRY(h, cudaEventRecord(ev_panel[i], Sp));
    } else {
      // block-row cyclic: a rank only reads its own rows of U; the gather (every rank needs all of U for the next
      // phase) runs on the communication stream
      ev_panel[i] = ev.get();
      CUDA_TRY(h, cudaEventRecord(ev_panel[i], Sp));
      CUDA_TRY(h, cudaStreamWaitEvent(Sc, ev_panel[i], 0));
      r = gather_panel(h, d, d->U, s.ld, n, NB, i, 0, i + 1, Sc);
    }
    return r;
  };
  rc = panel(0);
  for (int i = 0; i < nblk && !rc; ++i) {
    if (i + 1 < nblk) {
      if (i >= 1) CUDA_TRY(h, cudaStreamWaitEvent(Sp, ev_a[i - 1], 0));
      h->cur = Sp;
      rc = run_tasks(h, pl, pl.la[i], Um, Tm, Um, NB, -1.0, true);
      if (rc) break;
    }
    // bulk of step i may start as soon as panel i is available (its event was recorded inside panel(i))
    CUDA_TRY(h, cudaStreamWaitEvent(Sb, ev_panel[i], 0));
    if (i + 1 < nblk) {
      rc = panel(i + 1);
      if (rc) break;
    }
    h->cur = Sb;
    rc = run_tasks(h, pl, pl.bulkA[i], Um, Tm, Um, NB, -1.0, true);
    ev_a[i] = ev.get();
    CUDA_TRY(h, cudaEventRecord(ev_a[i], Sb));
    if (!rc) rc = run_tasks(h, pl, pl.bulkB[i], Um, Tm, Um, NB, -1.0, true);
  }
  h->cur = S;
  if (rc) return rc;
  cudaEvent_t e1 = ev.get(), e2 = ev.get(), e3 = ev.get();
  CUDA_TRY(h, cudaEventRecord(e1, Sp));
  CUDA_TRY(h, cudaEventRecord(e2, Sb));
  CUDA_TRY(h, cudaEventRecord(e3, Sc));
  CUDA_TRY(h, cudaStreamWaitEvent(S, e1, 0));
  CUDA_TRY(h, cudaStreamWaitEvent(S, e2, 0));
  CUDA_TRY(h, cudaStreamWaitEvent(S, e3, 0));
  if (p2p && last_seq) return wait_flags(h, d, 0, -1, last_seq, S);      // every peer's last column has landed: U is complete here
  return GPP_OK;
}

// own sub-blocks of the interior inverse (one launch per virtual rank), on the main stream
int dist_ablocks(gpp_handle* h, DistState* d, GramSlot& s) {
  const int NB = h->NB;
  const std::vector<Grid> grids = grids_of(d);
  const MatRef Um{d->U, s.ld, &d->mapU};
  h->cur = h->stream;
  // virtual ranks share one store: rank v's blocks follow those of ranks < v
  size_t total_blocks = 0;
  std::vector<Plan*> plans(grids.size());
  for (size_t v = 0; v < grids.size(); ++v) {
    int rc = ensure_plan(h, d, 2, d->nv > 0 ? (int)v : 0, grids[v], s.N, NB, s.M, s.off, d->inv_pde, &plans[v]);
    if (rc) return rc;
    total_blocks += plans[v]->hblocks.size();
  }
  int rc = dev_reserve(h, &d->Asub, std::max<size_t>(1, total_blocks) * 4 * NB * NB);
  if (rc) return rc;
  d->nbh = NB;
  size_t base_blocks = 0;
  for (size_t v = 0; v < grids.size(); ++v) {
    const Plan& pl = *plans[v];
    const MatRef Cm{d->Asub + base_blocks * 4 * NB * NB, (long)NB, nullptr};
    rc = run_tasks(h, pl, pl.all, Um, Um, Cm, NB, 1.0, false);
    if (rc) return rc;
    base_blocks += pl.hblocks.size();
  }
  return GPP_OK;
}

}  // namespace

int potrf_right_looking(gpp_handle* h, double* A, long ld, int n, const TMap2* map) {
  if (!h->dist_local) {
    DistState* d = new DistState();
    d->rank = 0; d->world = 1; d->nv = 0; d->P = 1; d->Q = 1;
    int lo = 0, hi = 0;
    cudaDeviceGetStreamPriorityRange(&lo, &hi);
    CUDA_TRY(h, cudaStreamCreateWithPriority(&d->sC, cudaStreamNonBlocking, hi));
    h->dist_local = d;
  }
  return dist_potrf_matrix(h, static_cast<DistState*>(h->dist_local), A, ld, n, map, 0, false, nullptr, 0);
}

void dist_local_release(gpp_handle* h) {
  if (!h->dist_local) return;
  DistState* d = static_cast<DistState*>(h->dist_local);
  for (auto& kv : d->plans) {
    if (kv.second.dev) cudaFree(kv.second.dev);
    if (kv.second.dev_hblocks) cudaFree(kv.second.dev_hblocks);
  }
  if (d->sC) cudaStreamDestroy(d->sC);
  delete d;
  h->dist_local = nullptr;
}

// Hessian blocks of the own (bi, bc) pairs + distributed Cholesky of H; called from gn_step when h->dist_gn
int dist_gn_hess_potrf(gpp_handle* h) {
  DistState* d = ds(h);
  if (!d || !d->inverse_ready) { h->err = "gpp_dist_inverse first"; return -1; }
  GnState& g = h->gn;
  const std::vector<Grid> grids = grids_of(d);
  h->cur = h->stream;
  size_t base_blocks = 0;
  for (size_t v = 0; v < grids.size(); ++v) {
    Plan& pl = plan_slot(d, 2, d->nv > 0 ? (int)v : 0);
    if (!pl.valid) { h->err = "inverse plan missing"; return -1; }
    int rc = gn_hess_blocks(h, pl.dev_hblocks, (int)pl.hblocks.size(), d->Asub + base_blocks * 4 * (size_t)d->nbh * d->nbh, d->nbh);
    if (rc) return rc;
    base_blocks += pl.hblocks.size();
  }
  return dist_potrf_matrix(h, d, g.H, g.ldH, g.n, &g.mapH, 3, false, nullptr, h->caps.count(&g.H) ? h->caps[&g.H] : 0);
}

extern "C" {

int gpp_dist_unique_id(unsigned char* id128) {
  if (!id128) return -1;
  static_assert(sizeof(ncclUniqueId) == 128, "ncclUniqueId is 128 bytes");
  ncclUniqueId id;
  if (ncclGetUniqueId(&id) != ncclSuccess) return GPP_CUDA_ERR + 2;
  memcpy(id128, &id, 128);
  return GPP_OK;
}

static int dist_common_init(gpp_handle* h, DistState* d) {
  int lo = 0, hi = 0;
  cudaDeviceGetStreamPriorityRange(&lo, &hi);
  CUDA_TRY(h, cudaStreamCreateWithPriority(&d->sC, cudaStreamNonBlocking, hi));
  h->dist = d;
  h->dist_gn = false;
  return GPP_OK;
}

int gpp_dist_init(gpp_handle* h, int rank, int world, const unsigned char* id128) {
  if (h) cudaSetDevice(h->device);
  if (!h || !id128) return -1;
  if (world < 1 || rank < 0 || rank >= world) { h->err = "bad rank/world"; return -2; }
  if (h->dist) { h->err = "already initialised"; return -3; }
  CUDA_TRY(h, cudaSetDevice(h->device));
  DistState* d = new DistState();
  d->rank = rank; d->world = world; d->P = world; d->Q = 1;
  ncclUniqueId id;
  memcpy(&id, id128, 128);
  ncclResult_t r = ncclCommInitRank(&d->comm, world, id, rank);
  if (r != ncclSuccess) { h->err = std::string("ncclCommInitRank: ") + ncclGetErrorString(r); delete d; return GPP_CUDA_ERR + 2; }
  const char* env = getenv("GPP_DIST_P2P");
  if (env) d->p2p = env[0] == '1';
  int rc = dist_common_init(h, d);
  if (rc) return rc;
  if (use_p2p(d)) {
    // CUDA IPC may be unavailable (container restrictions): agree among all ranks, otherwise use the NCCL gathers
    int ok = init_p2p(h, d) == GPP_OK ? 1 : 0;
    int* d_ok = nullptr;
    CUDA_TRY(h, cudaMalloc(&d_ok, sizeof(int)));
    CUDA_TRY(h, cudaMemcpy(d_ok, &ok, sizeof(int), cudaMemcpyHostToDevice));
    NCCL_TRY(h, ncclAllReduce(d_ok, d_ok, 1, ncclInt, ncclMin, d->comm, h->stream));
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    CUDA_TRY(h, cudaMemcpy(&ok, d_ok, sizeof(int), cudaMemcpyDeviceToHost));
    cudaFree(d_ok);
    if (!ok) {
      if (getenv("GPP_TRACE")) fprintf(stderr, "[gpp trace] rank %d: CUDA IPC not available (%s): NCCL gathers\n", rank, h->err.c_str());
      d->p2p = false;
      cudaGetLastError();
      h->err.clear();
    }
  }
  return GPP_OK;
}

int gpp_dist_init_virtual(gpp_handle* h, int nranks) {
  if (h) cudaSetDevice(h->device);
  if (!h) return -1;
  if (nranks < 1 || nranks > 64) { h->err = "bad number of virtual ranks"; return -2; }
  if (h->dist) { h->err = "already initialised"; return -3; }
  DistState* d = new DistState();
  d->rank = 0; d->world = 1; d->nv = nranks; d->P = nranks; d->Q = 1;
  return dist_common_init(h, d);
}

int gpp_dist_set_grid(gpp_handle* h, int P, int Q) {
  if (!h || !h->dist) return -1;
  DistState* d = ds(h);
  const int n = d->nv > 0 ? d->nv : d->world;
  if (P < 1 || Q < 1 || P * Q != n) { h->err = "P * Q must equal the number of ranks"; return -2; }
  d->P = P; d->Q = Q;
  d->inverse_ready = false;
  return GPP_OK;
}

int gpp_dist_info(gpp_handle* h, int* rank, int* world, int* P, int* Q) {
  if (!h || !h->dist) return -1;
  DistState* d = ds(h);
  if (rank) *rank = d->rank;
  if (world) *world = d->nv > 0 ? d->nv : d->world;
  if (P) *P = d->P;
  if (Q) *Q = d->Q;
  return GPP_OK;
}

// Host-only check of the Theta^{-1} sub-block plans of a PDE's sharded Hessian (no GPU, no handle): builds the plans of all
// P * Q ranks for N = N_domain, block size NB and M = (operator blocks) N + nb_extra, and verifies for the nz N x nz N
// Hessian that every lower block has exactly one owner and that every element of an own block receives each term of its
// unknown-block pair exactly once, from the right operand rows and K range.  Returns 0, -1 on bad arguments or a PDE that
// does not shard, or a positive code identifying the first violated property.
int gpp_dist_hess_plan_check(int N, int NB, int P, int Q, int pde, int nb_extra) {
  if (N <= 0 || NB <= 0 || NB % 64 || P < 1 || Q < 1 || P * Q > 64 || nb_extra < 0) return -1;
  const int layout = pde == PDE_ELLIPTIC ? LAY_ELLIPTIC : pde == PDE_BURGERS ? LAY_BURGERS : pde == PDE_EIKONAL ? LAY_EIKONAL : -1;
  TermTable tt;
  if (layout < 0 || make_term_table(pde, &tt) || tt.nslots != 1) return -1;
  const Layout lay = make_layout(layout);
  int off[GPP_MAX_BLOCKS + 1] = {0};
  for (int p = 0; p <= lay.nblk; ++p) off[p] = p * N;
  const int M = lay.nblk * N + nb_extra, k1 = (int)round_up(M, 16);
  const int n = tt.nz * N, nblk = nblocks_of(n, NB);
  std::vector<Plan> plans(P * Q);
  std::vector<Grid> grids;
  for (int r = 0; r < P * Q; ++r) grids.push_back(Grid{P, Q, r / Q, r % Q});
  for (int r = 0; r < P * Q; ++r) build_ablock_plan(plans[r], grids[r], tt, N, M, off, NB);
  std::vector<int> cnt((size_t)nblk * nblk, 0);
  std::vector<unsigned char> w((size_t)4 * NB * NB);
  for (int r = 0; r < P * Q; ++r) {
    const Plan& pl = plans[r];
    std::vector<std::vector<const GemmTask*>> of_block(pl.hblocks.size());
    size_t want_tasks = 0;
    for (const int4& hb : pl.hblocks) {
      if (owner_of(grids[r], hb.x, hb.y) != r || hb.y > hb.x) return 21;
      cnt[(size_t)hb.x * nblk + hb.y]++;
      for (const Seg& a : field_segments(hb.x, NB, n, N))
        for (const Seg& b : field_segments(hb.y, NB, n, N)) want_tasks += tt.nterms[a.q * tt.nz + b.q];
    }
    if (pl.host.size() != want_tasks) return 20;        // elliptic: four tasks per Hessian block
    for (const GemmTask& t : pl.host) {
      const size_t e = (size_t)(t.c_row / (4 * NB));
      if (t.c_row < 0 || e >= of_block.size()) return 23;
      of_block[e].push_back(&t);
    }
    for (size_t e = 0; e < pl.hblocks.size(); ++e) {
      const int4 hb = pl.hblocks[e];
      const int rows = rows_of(n, NB, hb.x), cols = rows_of(n, NB, hb.y);
      std::fill(w.begin(), w.end(), 0);
      for (const GemmTask* t : of_block[e]) {
        const int slot = (t->c_row / NB) % 4, r0 = t->c_row % NB, c0 = t->c_col;
        if (t->m <= 0 || t->n <= 0 || c0 < 0 || r0 + t->m > rows || c0 + t->n > cols) return 23;
        if (t->k0 != (std::max(t->a_row, t->b_row) / 16) * 16 || t->k1 != k1 || t->kb_off != 0 || t->tri != 0) return 24;
        for (int x = 0; x < t->m; ++x) {
          const int gr = hb.x * NB + r0 + x, q = gr / N, i = gr - q * N;
          for (int y = 0; y < t->n; ++y) {
            const int gc = hb.y * NB + c0 + y, qq = gc / N, j = gc - qq * N;
            const int pr = q * tt.nz + qq;
            if (slot >= tt.nterms[pr]) return 23;
            if (t->a_row + x != off[tt.tp[pr][slot]] + i || t->b_row + y != off[tt.tpp[pr][slot]] + j) return 24;
            w[((size_t)slot * NB + r0 + x) * NB + c0 + y]++;
          }
        }
      }
      for (int x = 0; x < rows; ++x)
        for (int y = 0; y < cols; ++y) {
          const int pr = ((hb.x * NB + x) / N) * tt.nz + (hb.y * NB + y) / N;
          for (int slot = 0; slot < 4; ++slot)
            if (w[((size_t)slot * NB + x) * NB + y] != (slot < tt.nterms[pr] ? 1 : 0)) return 25;
        }
    }
  }
  for (int bi = 0; bi < nblk; ++bi)
    for (int bc = 0; bc <= bi; ++bc)
      if (cnt[(size_t)bi * nblk + bc] != 1) return 22;
  return 0;
}

// Host-only consistency check of the task plans (no GPU, no handle): builds the plans of all P * Q ranks for an n x n
// matrix with block size NB and verifies, for every step, that each block that must be touched is touched by exactly one
// rank (its owner) -- panel blocks solved once, trailing blocks updated once, Hessian blocks owned once.
// phase: 0 = right-looking Cholesky, 1 = U = L^{-T}, 2 = Theta^{-1} sub-blocks of the elliptic Hessian (n = N_domain,
// M = 2 n + nb_extra; gpp_dist_hess_plan_check).  Returns 0, or a positive code identifying the first violated property.
int gpp_dist_plan_check(int n, int NB, int P, int Q, int phase, int nb_extra) {
  if (n <= 0 || NB <= 0 || NB % 64 || P < 1 || Q < 1 || P * Q > 64 || phase < 0 || phase > 2) return -1;
  if (phase == 2) return gpp_dist_hess_plan_check(n, NB, P, Q, PDE_ELLIPTIC, nb_extra);
  const int nblk = nblocks_of(n, NB);
  std::vector<Plan> plans(P * Q);
  std::vector<Grid> grids;
  for (int r = 0; r < P * Q; ++r) grids.push_back(Grid{P, Q, r / Q, r % Q});
  for (int r = 0; r < P * Q; ++r) {
    if (phase == 0) build_potrf_plan(plans[r], grids[r], n, NB);
    else build_uinv_plan(plans[r], grids[r], n, NB);
  }
  for (int j = 0; j < nblk; ++j) {
    std::vector<int> upd((size_t)nblk * nblk, 0), solved(nblk, 0);
    for (int r = 0; r < P * Q; ++r) {
      const Plan& pl = plans[r];
      // panel rows of this rank: block-cyclic arithmetic map
      const TrsmRows& rm = pl.rows[j];
      for (int lr = 0; lr < rm.rows; lr += NB) {
        const int b = rm.first_blk + (lr / NB) * rm.stride_blk;
        if (b < 0 || b >= nblk) return 10;
        if (owner_of(grids[r], b, j) != r) return 11;
        solved[b]++;
      }
      for (const Launch* l : {&pl.la[j], &pl.bulkA[j], &pl.bulkB[j]})
        for (int t = 0; t < l->count; ++t) {
          const GemmTask& g = pl.host[l->off + t];
          const int bi = g.c_row / NB, bc = g.c_col / NB;
          if (owner_of(grids[r], bi, bc) != r) return 12;
          if (g.k0 != j * NB || g.k1 != j * NB + rows_of(n, NB, j)) return 13;
          if (g.m != rows_of(n, NB, bi) || g.n != rows_of(n, NB, bc)) return 14;
          upd[(size_t)bi * nblk + bc]++;
        }
    }
    for (int b = 0; b < nblk; ++b) {
      const bool want = phase == 0 ? (b > j) : (b <= j);       // Cholesky: blocks below the diagonal; U: rows up to the diagonal
      if (solved[b] != (want ? 1 : 0)) return 15;
    }
    for (int bi = 0; bi < nblk; ++bi)
      for (int bc = 0; bc < nblk; ++bc) {
        const bool want = phase == 0 ? (bc > j && bc <= bi) : (bi <= j && bc > j);
        if (upd[(size_t)bi * nblk + bc] != (want ? 1 : 0)) return 16;
      }
  }
  return 0;
}

int gpp_dist_exchange_mode(gpp_handle* h) {
  if (!h || !h->dist) return -1;
  return use_p2p(ds(h)) ? 1 : 0;
}

int gpp_dist_finalize(gpp_handle* h) {
  if (h) cudaSetDevice(h->device);
  if (!h || !h->dist) return -1;
  DistState* d = ds(h);
  cudaStreamSynchronize(h->stream);
  cudaDeviceSynchronize();
  for (auto& pm : d->pm)
    for (int r = 0; r < d->world; ++r)
      if (r != d->rank && pm.peer[r]) cudaIpcCloseMemHandle(pm.peer[r]);
  for (int r = 0; r < d->world; ++r)
    if (r != d->rank && d->peer_flags[r]) cudaIpcCloseMemHandle(d->peer_flags[r]);
  if (d->comm) {
    // the peers may still have this rank's buffers mapped: leave together
    if (d->world > 1 && d->push_counter) ncclAllReduce(d->push_counter + 3, d->push_counter + 3, 1, ncclUint32, ncclSum, d->comm, h->stream);
    cudaStreamSynchronize(h->stream);
    ncclCommDestroy(d->comm);
  }
  if (d->flags) cudaFree(d->flags);
  if (d->push_counter) cudaFree(d->push_counter);
  if (d->ipc_dev) cudaFree(d->ipc_dev);
  dev_release(h, &d->U); dev_release(h, &d->Asub); dev_release(h, &d->gbuf); dev_release(h, &d->dbuf); dev_release(h, &d->dvec);
  for (auto& kv : d->plans) {
    if (kv.second.dev) cudaFree(kv.second.dev);
    if (kv.second.dev_hblocks) cudaFree(kv.second.dev_hblocks);
  }
  if (d->sC) cudaStreamDestroy(d->sC);
  delete d;
  h->dist = nullptr;
  h->dist_gn = false;
  return GPP_OK;
}

// Sharded Gram_matrix_assembly (src/Gram_matrice.py:11-187): this rank fills the block rows bi with bi mod P == p of the
// replicated buffer of slot 0 (all column blocks up to the diagonal); no exchange.
int gpp_dist_gram_assemble(gpp_handle* h, int layout, int kernel, const double* kparams) {
  if (h) cudaSetDevice(h->device);
  if (!h || !h->dist) return -1;
  CUDA_TRY(h, cudaSetDevice(h->device));
  int rc = gram_slot_prepare(h, 0, layout, kernel, kparams);
  if (rc) return rc;
  DistState* d = ds(h);
  GramSlot& s = h->slot[0];
  d->inverse_ready = false;
  h->dist_gn = false;
  const int NB = h->NB, M = s.M;
  const int nblk = nblocks_of(M, NB);
  h->cur = h->stream;
  for (const Grid& g : grids_of(d)) {
    if (d->nv > 0 && g.q != 0) continue;           // virtual ranks of one process row hold the same rows
    for (int b = g.p; b < nblk; b += g.P) {
      const int g0 = b * NB, g1 = (g0 + NB < M) ? g0 + NB : M;
      for (int p = 0; p < s.lay.nblk; ++p) {        // split at the row-operator block boundaries
        const int lo = g0 > s.off[p] ? g0 : s.off[p];
        const int hi = g1 < s.off[p + 1] ? g1 : s.off[p + 1];
        if (hi <= lo) continue;
        rc = gram_assemble_rows(h, s, p, lo - s.off[p], hi - lo, s.T + (long)lo * s.ld, s.ld);
        if (rc) return rc;
      }
    }
  }
  return GPP_OK;
}

// diag_out[M]: the full diagonal on every rank (sum all-reduce of the parts held by the owners of the diagonal blocks)
int gpp_dist_get_diag(gpp_handle* h, double* diag_out) {
  if (h) cudaSetDevice(h->device);
  if (!h || !h->dist || !diag_out) return -1;
  DistState* d = ds(h);
  GramSlot& s = h->slot[0];
  if (!s.T) { h->err = "assemble first"; return -2; }
  const int NB = h->NB, M = s.M;
  int rc = dev_reserve(h, &d->dvec, M);
  if (rc) return rc;
  CUDA_TRY(h, cudaMemsetAsync(d->dvec, 0, sizeof(double) * M, h->stream));
  for (const Grid& g : grids_of(d))
    for (int b = 0; b * NB < M; ++b) {
      if (owner_of(g, b, b) != g.p * g.Q + g.q) continue;
      const int g0 = b * NB, nr = rows_of(M, NB, b);
      dist_get_diag_kernel<<<(nr + 255) / 256, 256, 0, h->stream>>>(s.T, s.ld, g0, nr, d->dvec);
      h->launches++;
    }
  if (d->world > 1) NCCL_TRY(h, ncclAllReduce(d->dvec, d->dvec, M, ncclDouble, ncclSum, d->comm, h->stream));
  CUDA_TRY(h, cudaMemcpyAsync(diag_out, d->dvec, sizeof(double) * M, cudaMemcpyDeviceToHost, h->stream));
  CUDA_TRY(h, cudaStreamSynchronize(h->stream));
  return GPP_OK;
}

// add a full-length vector to the diagonal entries of the block rows this rank holds
int gpp_dist_add_diag(gpp_handle* h, const double* add) {
  if (h) cudaSetDevice(h->device);
  if (!h || !h->dist || !add) return -1;
  DistState* d = ds(h);
  GramSlot& s = h->slot[0];
  if (!s.T) { h->err = "assemble first"; return -2; }
  const int NB = h->NB, M = s.M;
  int rc = dev_reserve(h, &d->dvec, M);
  if (rc) return rc;
  CUDA_TRY(h, cudaMemcpyAsync(d->dvec, add, sizeof(double) * M, cudaMemcpyHostToDevice, h->stream));
  for (const Grid& g : grids_of(d)) {
    if (d->nv > 0 && g.q != 0) continue;
    for (int b = g.p; b * NB < M; b += g.P) {
      const int g0 = b * NB, nr = rows_of(M, NB, b);
      dist_add_diag_kernel<<<(nr + 255) / 256, 256, 0, h->stream>>>(s.T, s.ld, g0, nr, d->dvec);
      h->launches++;
    }
  }
  CUDA_TRY(h, cudaStreamSynchronize(h->stream));
  return GPP_OK;
}

// Distributed X.Gram_Cholesky (src/PDEs.py:75-80).  *info as in gpp_potrf, identical on every rank.  Afterwards every
// rank holds the full factor: gpp_gn_loss, gpp_solve_vec, gpp_predict and gpp_gram_download(.., 1) work unchanged.
int gpp_dist_potrf(gpp_handle* h, int* info) {
  if (h) cudaSetDevice(h->device);
  if (!h || !h->dist) return -1;
  DistState* d = ds(h);
  GramSlot& s = h->slot[0];
  if (!s.T) { h->err = "assemble first"; return -2; }
  if (s.factored) { h->err = "already factored"; return -3; }
  CUDA_TRY(h, cudaSetDevice(h->device));
  int rc = dist_potrf_matrix(h, d, s.T, s.ld, s.M, &s.mapT, 0, true, info, h->caps.count(&s.T) ? h->caps[&s.T] : 0);
  if (rc) return rc;
  s.factored = true;
  s.inverted = false;
  return GPP_OK;
}

// Distributed counterpart of gpp_inverse for the elliptic, Burgers and Eikonal layouts: U = L^{-T} (sharded, then
// replicated) and the sub-blocks of the interior inverse that this rank's Hessian blocks need for the PDE of that layout.
// Enables gpp_dist_gn_step for that PDE.
int gpp_dist_inverse(gpp_handle* h) {
  if (h) cudaSetDevice(h->device);
  if (!h || !h->dist) return -1;
  DistState* d = ds(h);
  GramSlot& s = h->slot[0];
  if (!s.factored) { h->err = "gpp_dist_potrf first"; return -2; }
  const int pde = sharded_pde_of_layout(s.layout_id);
  if (pde < 0) { h->err = "the sharded GN path supports the elliptic, Burgers and Eikonal layouts only"; return -3; }
  CUDA_TRY(h, cudaSetDevice(h->device));
  d->inverse_ready = false;
  d->inv_pde = pde;
  int rc = dev_reserve(h, &d->U, (size_t)s.M * s.ld);
  if (rc) return rc;
  rc = make_tensor_map(h, &d->mapU, d->U, s.M, s.M, s.ld);
  if (rc) return rc;
  static const bool trace = getenv("GPP_TRACE") != nullptr;
  if (trace) cudaEventRecord(h->ev[2], h->stream);
  rc = dist_uinv(h, d, s);
  if (rc) return rc;
  if (trace) cudaEventRecord(h->ev[3], h->stream);
  rc = dist_ablocks(h, d, s);
  if (rc) return rc;
  if (trace) {
    cudaEventRecord(h->ev[4], h->stream);
    cudaEventSynchronize(h->ev[4]);
    float t1 = 0, t2 = 0;
    cudaEventElapsedTime(&t1, h->ev[2], h->ev[3]);
    cudaEventElapsedTime(&t2, h->ev[3], h->ev[4]);
    fprintf(stderr, "[gpp trace] dist inverse (rank %d): U = L^-T %.2f ms | A blocks %.2f ms\n", d->rank, t1, t2);
  }
  d->inverse_ready = true;
  h->dist_gn = true;
  return GPP_OK;
}

// one iteration of GN_method's loop body (src/PDEs.py:117-120) with the sharded Hessian assembly and the distributed
// Cholesky of H; every rank ends with the same z and returns the same loss.  The PDE set up by gpp_gn_setup must be the
// one of the layout gpp_dist_inverse planned for.
int gpp_dist_gn_step(gpp_handle* h, double step, double* loss) {
  if (h) cudaSetDevice(h->device);
  if (!h || !h->dist) return -1;
  if (!h->gn.ready) { h->err = "gpp_gn_setup first"; return -1; }
  const int pde = h->gn.pde;
  if (pde != PDE_ELLIPTIC && pde != PDE_BURGERS && pde != PDE_EIKONAL) {
    h->err = "the sharded GN path supports Nonlinear_elliptic, Burgers and Eikonal only";
    return -2;
  }
  if (!ds(h)->inverse_ready || !h->dist_gn) { h->err = "gpp_dist_inverse first"; return -3; }
  if (pde != ds(h)->inv_pde) { h->err = "gpp_dist_inverse was built for the Gram layout of another PDE"; return -5; }
  if (!loss) return -4;
  CUDA_TRY(h, cudaSetDevice(h->device));
  return gn_step(h, step, loss);
}

}  // extern "C"
