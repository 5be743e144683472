// Posterior variance of the GP solution at test points (no counterpart in the reference, which returns the posterior
// mean only):
//   var(x) = kappa(x, x) - theta(x)^T Theta^{-1} theta(x) = kappa(x, x) - |w(x)|^2,   w(x) = L^{-1} theta(x),
// theta(x) = the row of construct_Theta_test for x (identity functional on the test side, the slot's operators on the
// collocation side), L = the Cholesky factor the slot holds (nugget included).  For a chunk of test rows:
//   W = Theta_test (theta_test_kernel, one exp per pair), then W L^T = Theta_test is solved in place, left-looking over
//   the NB-wide block columns J of L:  W[:, J] -= W[:, <J] L[J, <J]^T  (long-K DMMA GEMM, K = [0, J NB)), then the
//   panel solve against L_JJ; finally var[t] = kappa(x_t, x_t) - sum_k W[t, k]^2.
// Only the lower triangle of T is read (after gpp_inverse its strict upper triangle holds U = L^{-T}).  Every step
// treats a row on its own with a fixed order of operations (the GEMM consumes K in the same order for either tile
// size, DESIGN section 4.1), so a row's result does not depend on the chunk it falls in, on the rank that computes it
// or on the GEMM tile size.
#include "gpp_internal.cuh"

namespace {

constexpr int kChunkRows = 18944;        // 4 full waves of 128 x 128 tiles on 148 SMs per block column at NB = 512
constexpr size_t kMemMargin = size_t(2) << 30;

// one warp per row: lanes stride over k < M, then a fixed-order butterfly; no atomics
__global__ void __launch_bounds__(256)
var_rows_kernel(const double* __restrict__ W, long ld, int rows, int M, const double* __restrict__ kappa0,
                double* __restrict__ var) {
  const int t = blockIdx.x * 8 + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (t >= rows) return;
  const double* w = W + (long)t * ld;
  double acc = 0.0;
  for (int k = lane; k < M; k += 32) acc = fma(w[k], w[k], acc);
#pragma unroll
  for (int o = 16; o >= 1; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  if (lane == 0) var[t] = *kappa0 - acc;
}

// rows of the chunk buffer that fit beside what the device already holds (the present buffer is given back first)
int chunk_rows(gpp_handle* h, long ld, int* rows) {
  size_t free_b = 0, total_b = 0;
  CUDA_TRY(h, cudaMemGetInfo(&free_b, &total_b));
  auto it = h->caps.find(&h->var_W);
  const size_t have = (h->var_W && it != h->caps.end()) ? it->second * sizeof(double) : 0;
  const size_t avail = free_b + have > kMemMargin ? free_b + have - kMemMargin : 0;
  const long fit = (long)(avail / ((size_t)ld * sizeof(double))) / 64 * 64;
  if (fit < 64) { h->err = "predict_var: not enough device memory for 64 test rows"; return -7; }
  *rows = fit < kChunkRows ? (int)fit : kChunkRows;
  return GPP_OK;
}

}  // namespace

int predict_var(gpp_handle* h, int slot, const double* d_xtest, int row0, int nrows, double* d_var) {
  if (nrows <= 0) return GPP_OK;
  GramSlot& s = h->slot[slot];
  const int NB = h->NB, M = s.M;
  const long ld = s.ld;
  h->cur = h->stream;
  // kappa(x, x) through the kernel-functional code at d = 0 (stationary kernels: the same for every x)
  int rc = dev_reserve(h, &h->var_aux, 8);
  if (rc) return rc;
  CUDA_TRY(h, cudaMemsetAsync(h->var_aux, 0, 4 * sizeof(double), h->stream));
  const double kp[4] = {s.kp_b1, s.kp_b2, s.kp_e1, s.kp_e2};
  rc = gram_kernel_eval(h, s.kernel_id, kp, OP_ID, OP_ID, h->var_aux, 1, h->var_aux + 4);
  if (rc) return rc;
  const double* d_kappa = h->var_aux + 4;
  int cap = 0;
  rc = chunk_rows(h, ld, &cap);
  if (rc) return rc;
  for (int c0 = 0; c0 < nrows; c0 += cap) {
    const int rows = (nrows - c0 < cap) ? nrows - c0 : cap;
    rc = dev_reserve(h, &h->var_W, (size_t)rows * ld);
    if (rc) return rc;
    double* W = h->var_W;
    if (h->var_map_base != W || h->var_map_rows != rows || h->var_map_cols != M || h->var_map_ld != ld) {
      rc = make_tensor_map(h, &h->var_map, W, rows, M, ld);
      if (rc) return rc;
      h->var_map_base = W; h->var_map_rows = rows; h->var_map_cols = M; h->var_map_ld = ld;
    }
    rc = gram_theta_test(h, s, d_xtest + 2 * (long)(row0 + c0), rows, W, ld);
    if (rc) return rc;
    for (int j0 = 0; j0 < M; j0 += NB) {
      const int nbw = (M - j0 < NB) ? M - j0 : NB;
      if (j0 > 0) {
        GemmDesc d{};
        d.mapA = &h->var_map; d.mapB = &s.mapT;
        d.a_row0 = 0; d.b_row0 = j0;
        d.C = W + j0; d.ldc = ld; d.Cin = d.C; d.ldcin = ld;
        d.m = rows; d.n = nbw; d.k0 = 0; d.k1 = j0; d.kb_off = 0;
        d.alpha = -1.0;
        rc = gemm_nt_launch(h, d);
        if (rc) return rc;
      }
      rc = trsm_panel_launch(h, W + j0, ld, TrsmRows{rows, 0, 0, 0}, s.T + (long)j0 * ld + j0, ld, nbw);
      if (rc) return rc;
    }
    var_rows_kernel<<<(rows + 7) / 8, 256, 0, h->stream>>>(W, ld, rows, M, d_kappa, d_var + row0 + c0);
    h->launches++;
    CUDA_TRY(h, cudaGetLastError());
  }
  return GPP_OK;
}
