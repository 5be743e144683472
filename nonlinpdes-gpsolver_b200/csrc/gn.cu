// Gauss-Newton step on the device.
//
// Replaces loss / grad_loss / GN_loss / Hessian_GN / GN_method of the reference
// (src/PDEs.py:83-135, :279-343, :419-498; src/InverseProblems.py:106-186).
// With F(z) the stacked functional values and J = dF/dz:
//   loss = |L^{-1} F|^2,  g = 2 J^T Theta^{-1} F,  H = 2 J^T Theta^{-1} J,  z <- z - step H^{-1} g.
// J only has diagonal blocks: J[(p, i), (q, i)] = c_pq[i].  Hence
//   H[(q,i),(q',j)] = 2 sum_{p,p'} c_pq[i] Ainv[(p,i),(p',j)] c_p'q'[j]
// with Ainv the interior block of Theta^{-1} computed once per solve (chol.cu), so a GN
// step costs O(n^2) assembly + one n x n Cholesky instead of the reference's dense
// M x n triangular solve and M n^2 product.
//
// The residual / linearisation kernels are bit-exact restatements of the reference's
// expression trees: this file is compiled with -fmad=false and every operation below is
// written in the order the Python expressions evaluate.
#include "gpp_internal.cuh"

#include <cmath>
#include <cstdlib>
#include <cstring>
#include <math_constants.h>

namespace {

// exp shared (same algorithm, same constants) with oracle/gpp_exp_ref.c so that Darcy's
// exp(-w0) (src/InverseProblems.py:114) is bit-identical on host and device.
__device__ __forceinline__ double gpp_exp(double x) {
  if (x != x) return x;
  if (x > 709.782712893384) return CUDART_INF;
  if (x < -745.1332191019412) return 0.0;
  const double L2E = 1.4426950408889634074;
  const double LN2HI = 6.93147180369123816490e-01, LN2LO = 1.90821492927058770002e-10;
  const double kf = rint(x * L2E);
  double r = __fma_rn(-kf, LN2HI, x);
  r = __fma_rn(-kf, LN2LO, r);
  double p = 1.0 / 6227020800.0;
  p = __fma_rn(p, r, 1.0 / 479001600.0);
  p = __fma_rn(p, r, 1.0 / 39916800.0);
  p = __fma_rn(p, r, 1.0 / 3628800.0);
  p = __fma_rn(p, r, 1.0 / 362880.0);
  p = __fma_rn(p, r, 1.0 / 40320.0);
  p = __fma_rn(p, r, 1.0 / 5040.0);
  p = __fma_rn(p, r, 1.0 / 720.0);
  p = __fma_rn(p, r, 1.0 / 120.0);
  p = __fma_rn(p, r, 1.0 / 24.0);
  p = __fma_rn(p, r, 1.0 / 6.0);
  p = __fma_rn(p, r, 0.5);
  p = __fma_rn(p, r, 1.0);
  p = __fma_rn(p, r, 1.0);
  return ldexp(p, (int)kf);
}

struct FParams {
  int pde, N, Nb, m_int;
  double p0, p1, p2, p3;      // elliptic: alpha, m, alpha*m ; burgers: alpha, nu, -alpha ; eikonal: eps
  const double* z;
  const double* rhs_f;
  const double* bdy_g;
  double* F0; double* F1;     // slot 0 / slot 1 residual vectors
  double* coef;               // [slot][p][q][N]
  int with_coef;
};

__device__ __forceinline__ double ipow(double z, int m) {
  double r = z;
  for (int k = 1; k < m; ++k) r = r * z;
  return r;
}

__device__ __forceinline__ double* cptr(double* coef, int N, int s, int p, int q) {
  return coef + ((long)((s * GPP_MAX_BLOCKS + p) * GPP_MAX_ZBLOCKS + q)) * N;
}

__global__ void fcoef_kernel(const FParams a) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  const int N = a.N;
  if (i < N) {
    if (a.pde == PDE_ELLIPTIC) {
      // F = [alpha*z^m - f ; z ; g]                         src/PDEs.py:84-85
      const double z = a.z[i];
      const double zm = (a.m_int >= 1) ? ipow(z, a.m_int) : ((a.m_int == 0 && a.p1 == 0.0) ? 1.0 : pow(z, a.p1));
      a.F0[i] = a.p0 * zm - a.rhs_f[i];
      a.F0[N + i] = z;
      if (a.with_coef) {
        // alpha*m*z^(m-1)                                   src/PDEs.py:95
        const double zm1 = (a.m_int >= 2) ? ipow(z, a.m_int - 1) : ((a.m_int == 1) ? 1.0 : pow(z, a.p1 - 1.0));
        cptr(a.coef, N, 0, 0, 0)[i] = a.p2 * zm1;
        cptr(a.coef, N, 0, 1, 0)[i] = 1.0;
      }
    } else if (a.pde == PDE_BURGERS) {
      // F = [nu*v3 + f - alpha*v0*v2 ; v2 ; v3 ; v0 ; g]   src/PDEs.py:280-287
      const double v0 = a.z[i], v2 = a.z[N + i], v3 = a.z[2 * N + i];
      a.F0[i] = (a.p1 * v3 + a.rhs_f[i]) - (a.p0 * v0) * v2;
      a.F0[N + i] = v2;
      a.F0[2 * N + i] = v3;
      a.F0[3 * N + i] = v0;
      if (a.with_coef) {
        // [-alpha diag(v2), -alpha diag(v0), nu I]          src/PDEs.py:301
        cptr(a.coef, N, 0, 0, 0)[i] = a.p2 * v2;
        cptr(a.coef, N, 0, 0, 1)[i] = a.p2 * v0;
        cptr(a.coef, N, 0, 0, 2)[i] = a.p1;
        cptr(a.coef, N, 0, 1, 1)[i] = 1.0;
        cptr(a.coef, N, 0, 2, 2)[i] = 1.0;
        cptr(a.coef, N, 0, 3, 0)[i] = 1.0;
      }
    } else if (a.pde == PDE_EIKONAL) {
      // v3 = -(f^2 - v1^2 - v2^2)/eps ; F = [v1; v2; v3; v0; g]   src/PDEs.py:420-428
      const double v0 = a.z[i], v1 = a.z[N + i], v2 = a.z[2 * N + i];
      const double f = a.rhs_f[i];
      a.F0[i] = v1;
      a.F0[N + i] = v2;
      a.F0[2 * N + i] = -((f * f - v1 * v1) - v2 * v2) / a.p0;
      a.F0[3 * N + i] = v0;
      if (a.with_coef) {
        // d v3 / d v1 = 2 v1 / eps                           src/PDEs.py:444
        cptr(a.coef, N, 0, 0, 1)[i] = 1.0;
        cptr(a.coef, N, 0, 1, 2)[i] = 1.0;
        cptr(a.coef, N, 0, 2, 1)[i] = (2.0 * v1) / a.p0;
        cptr(a.coef, N, 0, 2, 2)[i] = (2.0 * v2) / a.p0;
        cptr(a.coef, N, 0, 3, 0)[i] = 1.0;
      }
    } else if (a.pde == PDE_ELLIPTIC_RELAXED) {
      // relaxed formulation, z = [v; w]: F = [v; w; g], ss2 = -v + alpha*w^m - f      src/PDEs.py:137-148
      const double v = a.z[i], w = a.z[N + i];
      const double wm = (a.m_int >= 1) ? ipow(w, a.m_int) : pow(w, a.p1);
      a.F0[i] = v;
      a.F0[N + i] = w;
      cptr(a.coef, N, 1, 0, 0)[i] = ((-v) + a.p0 * wm) - a.rhs_f[i];                  // ss2
      if (a.with_coef) {
        const double wm1 = (a.m_int >= 2) ? ipow(w, a.m_int - 1) : ((a.m_int == 1) ? 1.0 : pow(w, a.p1 - 1.0));
        cptr(a.coef, N, 1, 0, 1)[i] = a.p2 * wm1;                                      // alpha*m*w^(m-1)   :164
        cptr(a.coef, N, 0, 0, 0)[i] = 1.0;
        cptr(a.coef, N, 0, 1, 1)[i] = 1.0;
      }
    } else {  // PDE_DARCY: z = [w0 w1 w2 v0 v1 v2]; slot 0 = Theta_u, slot 1 = Theta_a
      const double w0 = a.z[i], w1 = a.z[N + i], w2 = a.z[2 * N + i];
      const double v0 = a.z[3 * N + i], v1 = a.z[4 * N + i], v2 = a.z[5 * N + i];
      const double f = a.rhs_f[i];
      const double ew = gpp_exp(-w0);
      // v3 = -v1*w1 - v2*w2 + (-f)*exp(-w0)                  src/InverseProblems.py:114
      const double v3 = ((-v1) * w1 - v2 * w2) + (-f) * ew;
      a.F0[i] = v1; a.F0[N + i] = v2; a.F0[2 * N + i] = v3; a.F0[3 * N + i] = v0;
      a.F1[i] = w1; a.F1[N + i] = w2; a.F1[2 * N + i] = w0;
      if (a.with_coef) {
        // linearised v3 coefficients                          src/InverseProblems.py:140
        cptr(a.coef, N, 0, 0, 4)[i] = 1.0;
        cptr(a.coef, N, 0, 1, 5)[i] = 1.0;
        cptr(a.coef, N, 0, 2, 0)[i] = (-f) * (-ew);
        cptr(a.coef, N, 0, 2, 1)[i] = -v1;
        cptr(a.coef, N, 0, 2, 2)[i] = -v2;
        cptr(a.coef, N, 0, 2, 4)[i] = -w1;
        cptr(a.coef, N, 0, 2, 5)[i] = -w2;
        cptr(a.coef, N, 0, 3, 3)[i] = 1.0;
        cptr(a.coef, N, 1, 0, 1)[i] = 1.0;
        cptr(a.coef, N, 1, 1, 2)[i] = 1.0;
        cptr(a.coef, N, 1, 2, 0)[i] = 1.0;
      }
    }
  }
  if (i < a.Nb) {
    const int nb_rows = (a.pde == PDE_ELLIPTIC || a.pde == PDE_ELLIPTIC_RELAXED) ? 2 * N : 4 * N;
    a.F0[nb_rows + i] = a.bdy_g[i];
  }
}

// deterministic sum of squares (+ optional Darcy misfit), single CTA, fixed tree
__global__ void __launch_bounds__(1024)
sumsq_kernel(const double* __restrict__ a, int na, const double* __restrict__ b, int nb,
             const double* __restrict__ v0, const double* __restrict__ data, int ndata, double inv_noise2,
             double* __restrict__ out) {
  __shared__ double sh[1024];
  double acc = 0.0;
  for (int i = threadIdx.x; i < na; i += 1024) acc += a[i] * a[i];
  for (int i = threadIdx.x; i < nb; i += 1024) acc += b[i] * b[i];
  double mis = 0.0;
  for (int i = threadIdx.x; i < ndata; i += 1024) { double d = data ? v0[i] - data[i] : v0[i]; mis += d * d; }
  sh[threadIdx.x] = acc + inv_noise2 * mis;
  __syncthreads();
  for (int s = 512; s >= 1; s >>= 1) {
    if (threadIdx.x < s) sh[threadIdx.x] += sh[threadIdx.x + s];
    __syncthreads();
  }
  if (threadIdx.x == 0) out[0] = sh[0];
}

struct HParams {
  TermTable tt;
  int N;
  const double* coef;
  const double* A[GPP_MAX_SLOTS]; long ldA[GPP_MAX_SLOTS];
  double* H; long ldH;
  int data_block, ndata; double data_diag;   // Darcy: H[v0_i, v0_i] += 2/noise^2 for i < ndata
};

// H block (q, q') = blockIdx.z ; element (i, j)
__global__ void __launch_bounds__(256)
hess_kernel(const __grid_constant__ HParams a) {
  const int q = blockIdx.z / a.tt.nz, qq = blockIdx.z % a.tt.nz;
  const int j = blockIdx.x * 64 + (threadIdx.x & 63);
  const int ibase = blockIdx.y * 16 + (threadIdx.x >> 6) * 4;
  if (j >= a.N) return;
  const int nt = a.tt.nterms[blockIdx.z];
#pragma unroll
  for (int ii = 0; ii < 4; ++ii) {
    const int i = ibase + ii;
    if (i >= a.N) break;
    double acc = 0.0;
    for (int t = 0; t < nt; ++t) {
      const int s = a.tt.ts[blockIdx.z][t], p = a.tt.tp[blockIdx.z][t], pp = a.tt.tpp[blockIdx.z][t];
      const double ci = a.coef[((long)((s * GPP_MAX_BLOCKS + p) * GPP_MAX_ZBLOCKS + q)) * a.N + i];
      const double cj = a.coef[((long)((s * GPP_MAX_BLOCKS + pp) * GPP_MAX_ZBLOCKS + qq)) * a.N + j];
      const double av = a.A[s][(long)(p * a.N + i) * a.ldA[s] + pp * a.N + j];
      acc += (ci * av) * cj;
    }
    acc = 2.0 * acc;
    if (q == a.data_block && qq == a.data_block && i == j && i < a.ndata) acc += a.data_diag;
    a.H[(long)(q * a.N + i) * a.ldH + qq * a.N + j] = acc;
  }
}

// multi-GPU: one launch covers the Hessian blocks (bi, bc) this rank owns.  Row bi * nbh + r of H is (q, i), column
// bc * nbh + c is (q', j); term t of the pair (q, q') sits at row (4 e + t) * nbh + r of the compact sub-block store
// (leading dimension nbh).  Same terms in the same order as hess_kernel, e.g. elliptic:
// H_ij = 2 ((c_i A00) c_j + (c_i A01) 1 + (1 A10) c_j + (1 A11) 1)                       src/PDEs.py:94-102
__global__ void __launch_bounds__(256)
hess_blocks_kernel(const __grid_constant__ TermTable tt, const int4* __restrict__ blocks, const double* __restrict__ Asub,
                   int nbh, int N, const double* __restrict__ coef, double* __restrict__ H, long ldH) {
  const int4 b = blocks[blockIdx.z];
  const int n = tt.nz * N;
  const int c = blockIdx.x * 64 + (threadIdx.x & 63);
  const int rbase = blockIdx.y * 16 + (threadIdx.x >> 6) * 4;
  const int gc = b.y * nbh + c;
  if (c >= nbh || gc >= n) return;
  const int qq = gc / N, j = gc - qq * N;
  const long sub = (long)nbh * nbh;
#pragma unroll
  for (int ii = 0; ii < 4; ++ii) {
    const int r = rbase + ii;
    const int gr = b.x * nbh + r;
    if (r >= nbh || gr >= n) break;
    const int q = gr / N, i = gr - q * N;
    const int pr = q * tt.nz + qq;
    const int nt = tt.nterms[pr];
    const double* A = Asub + (long)b.z * 4 * sub + (long)r * nbh + c;
    double acc = 0.0;
    for (int t = 0; t < nt; ++t) {
      const int s = tt.ts[pr][t], p = tt.tp[pr][t], pp = tt.tpp[pr][t];
      const double ci = coef[((long)((s * GPP_MAX_BLOCKS + p) * GPP_MAX_ZBLOCKS + q)) * N + i];
      const double cj = coef[((long)((s * GPP_MAX_BLOCKS + pp) * GPP_MAX_ZBLOCKS + qq)) * N + j];
      acc += (ci * A[t * sub]) * cj;
    }
    H[(long)gr * ldH + gc] = 2.0 * acc;
  }
}

struct GParams {
  int N, nz, nslots;
  int nblk[GPP_MAX_SLOTS];
  unsigned char kind[GPP_MAX_SLOTS][GPP_MAX_BLOCKS][GPP_MAX_ZBLOCKS];
  const double* coef;
  const double* t[GPP_MAX_SLOTS];
  double* g;
  int data_block, ndata; double data_scale; const double* z; const double* data;
};

__global__ void grad_kernel(const __grid_constant__ GParams a) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= a.N) return;
  for (int q = 0; q < a.nz; ++q) {
    double acc = 0.0;
    for (int s = 0; s < a.nslots; ++s)
      for (int p = 0; p < a.nblk[s]; ++p)
        if (a.kind[s][p][q])
          acc += a.coef[((long)((s * GPP_MAX_BLOCKS + p) * GPP_MAX_ZBLOCKS + q)) * a.N + i] * a.t[s][p * a.N + i];
    acc = 2.0 * acc;
    if (q == a.data_block && i < a.ndata) acc += a.data_scale * (a.z[q * a.N + i] - a.data[i]);
    a.g[q * a.N + i] = acc;
  }
}

// relaxed elliptic: H += (2/lambda) B^T B, g += (2/lambda) B^T ss2 with B = [-I, diag(c)]   src/PDEs.py:166-169
__global__ void relax_penalty_kernel(int N, double two_over_lam, const double* __restrict__ ss2, const double* __restrict__ c,
                                     double* __restrict__ H, long ldH, double* __restrict__ g) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= N) return;
  const double ci = c[i], si = ss2[i];
  H[(long)i * ldH + i] += two_over_lam;
  H[(long)i * ldH + N + i] += -(two_over_lam * ci);
  H[(long)(N + i) * ldH + i] += -(two_over_lam * ci);
  H[(long)(N + i) * ldH + N + i] += two_over_lam * (ci * ci);
  g[i] += -(two_over_lam * si);
  g[N + i] += two_over_lam * (ci * si);
}

__global__ void axpy_kernel(double* __restrict__ z, const double* __restrict__ d, double step, int n) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) z[i] = z[i] - step * d[i];
}

void kind_table(int pde, unsigned char (&kind)[GPP_MAX_SLOTS][GPP_MAX_BLOCKS][GPP_MAX_ZBLOCKS]) {
  memset(kind, 0, sizeof(kind));
  auto K = [&](int s, int p, int q) { kind[s][p][q] = 1; };
  switch (pde) {
    case PDE_ELLIPTIC: K(0, 0, 0); K(0, 1, 0); break;
    case PDE_ELLIPTIC_RELAXED: K(0, 0, 0); K(0, 1, 1); break;
    case PDE_BURGERS: K(0, 0, 0); K(0, 0, 1); K(0, 0, 2); K(0, 1, 1); K(0, 2, 2); K(0, 3, 0); break;
    case PDE_EIKONAL: K(0, 0, 1); K(0, 1, 2); K(0, 2, 1); K(0, 2, 2); K(0, 3, 0); break;
    case PDE_DARCY:
      K(0, 0, 4); K(0, 1, 5); K(0, 2, 0); K(0, 2, 1); K(0, 2, 2); K(0, 2, 4); K(0, 2, 5); K(0, 3, 3);
      K(1, 0, 1); K(1, 1, 2); K(1, 2, 0);
      break;
  }
}

void set_kind(GnState& g) { kind_table(g.pde, g.coef_kind); }

int nslots_of(const GnState& g) { return g.pde == PDE_DARCY ? 2 : 1; }

}  // namespace

int pde_nz(int pde) { return (pde == PDE_ELLIPTIC) ? 1 : (pde == PDE_DARCY ? 6 : (pde == PDE_ELLIPTIC_RELAXED ? 2 : 3)); }

// every coefficient kind of a slot lies inside that slot's layout, so the term lists need no layout
int make_term_table(int pde, TermTable* tt) {
  if (pde < PDE_ELLIPTIC || pde > PDE_ELLIPTIC_RELAXED) return -1;
  unsigned char kind[GPP_MAX_SLOTS][GPP_MAX_BLOCKS][GPP_MAX_ZBLOCKS];
  kind_table(pde, kind);
  memset(tt, 0, sizeof(*tt));
  tt->nz = pde_nz(pde);
  tt->nslots = pde == PDE_DARCY ? 2 : 1;
  for (int q = 0; q < tt->nz; ++q)
    for (int qq = 0; qq < tt->nz; ++qq) {
      const int pr = q * tt->nz + qq;
      int nt = 0;
      for (int s = 0; s < tt->nslots; ++s)
        for (int p = 0; p < GPP_MAX_BLOCKS; ++p)
          for (int pp = 0; pp < GPP_MAX_BLOCKS; ++pp)
            if (kind[s][p][q] && kind[s][pp][qq]) {
              if (nt >= 8) return -1;
              tt->ts[pr][nt] = s; tt->tp[pr][nt] = p; tt->tpp[pr][nt] = pp;
              ++nt;
            }
      tt->nterms[pr] = nt;
    }
  return 0;
}

int gn_eval_F(gpp_handle* h, const double* d_z, bool with_coef) {
  GnState& g = h->gn;
  FParams a{};
  a.pde = g.pde; a.N = h->N; a.Nb = h->Nb; a.m_int = g.m_int;
  a.p0 = g.params[0]; a.p1 = g.params[1]; a.p2 = g.params[2]; a.p3 = g.params[3];
  a.z = d_z; a.rhs_f = g.rhs_f; a.bdy_g = g.bdy_g;
  a.F0 = g.F[0]; a.F1 = g.F[1]; a.coef = g.coef; a.with_coef = with_coef ? 1 : 0;
  const int nmax = h->N > h->Nb ? h->N : h->Nb;
  fcoef_kernel<<<(nmax + 255) / 256, 256, 0, h->stream>>>(a);
  h->launches++;
  CUDA_TRY(h, cudaGetLastError());
  return GPP_OK;
}

// F(z), s = L^{-1} F per slot, loss; leaves s in g.s[] and coefficients in g.coef
static int eval_loss_device(gpp_handle* h, const double* d_z, bool with_coef) {
  GnState& g = h->gn;
  int rc = gn_eval_F(h, d_z, with_coef);
  if (rc) return rc;
  const int ns = nslots_of(g);
  for (int s = 0; s < ns; ++s) {
    GramSlot& sl = h->slot[s];
    CUDA_TRY(h, cudaMemcpyAsync(g.s[s], g.F[s], sizeof(double) * sl.M, cudaMemcpyDeviceToDevice, h->stream));
    rc = trsv_lower(h, sl.T, sl.ld, sl.M, g.s[s], false);
    if (rc) return rc;
  }
  const bool darcy = g.pde == PDE_DARCY;
  if (g.pde == PDE_ELLIPTIC_RELAXED) {
    const double* ss2 = g.coef + ((long)((1 * GPP_MAX_BLOCKS + 0) * GPP_MAX_ZBLOCKS + 0)) * h->N;
    sumsq_kernel<<<1, 1024, 0, h->stream>>>(g.s[0], h->slot[0].M, nullptr, 0, ss2, nullptr, h->N, 1.0 / g.params[3], g.scal);
  } else {
    sumsq_kernel<<<1, 1024, 0, h->stream>>>(g.s[0], h->slot[0].M, darcy ? g.s[1] : nullptr, darcy ? h->slot[1].M : 0,
                                            darcy ? d_z + 3 * (long)h->N : nullptr, g.data_u, darcy ? g.N_data : 0,
                                            darcy ? 1.0 / (g.noise * g.noise) : 0.0, g.scal);
  }
  h->launches++;
  CUDA_TRY(h, cudaGetLastError());
  return GPP_OK;
}

int gn_loss(gpp_handle* h, const double* d_z, double* loss_host) {
  int rc = eval_loss_device(h, d_z, true);
  if (rc) return rc;
  CUDA_TRY(h, cudaMemcpyAsync(loss_host, h->gn.scal, sizeof(double), cudaMemcpyDeviceToHost, h->stream));
  CUDA_TRY(h, cudaStreamSynchronize(h->stream));
  if (d_z == h->gn.z) h->gn.current = true;
  return GPP_OK;
}

int gn_hess_blocks(gpp_handle* h, const int4* d_blocks, int nblocks, const double* Asub, int nbh) {
  GnState& g = h->gn;
  if (g.pde != PDE_ELLIPTIC && g.pde != PDE_BURGERS && g.pde != PDE_EIKONAL) {
    h->err = "sharded Hessian assembly: elliptic, Burgers and Eikonal only";
    return -1;
  }
  TermTable tt;
  if (make_term_table(g.pde, &tt)) { h->err = "term table"; return -1; }
  if (nblocks <= 0) return GPP_OK;
  for (int b0 = 0; b0 < nblocks; b0 += 32768) {
    const int nb = (nblocks - b0 < 32768) ? (nblocks - b0) : 32768;
    dim3 grid((nbh + 63) / 64, (nbh + 15) / 16, nb);
    hess_blocks_kernel<<<grid, 256, 0, h->cur>>>(tt, d_blocks + b0, Asub, nbh, h->N, g.coef, g.H, g.ldH);
    h->launches++;
  }
  CUDA_TRY(h, cudaGetLastError());
  return GPP_OK;
}

// t = L^{-T} s and g = grad loss(z); requires F, s and coef of g.z to be current.
int gn_grad(gpp_handle* h) {
  GnState& g = h->gn;
  const int ns = nslots_of(g);
  const int N = h->N;
  set_kind(g);
  int rc;
  for (int s = 0; s < ns; ++s) {
    GramSlot& sl = h->slot[s];
    CUDA_TRY(h, cudaMemcpyAsync(g.t[s], g.s[s], sizeof(double) * sl.M, cudaMemcpyDeviceToDevice, h->stream));
    rc = trsv_lower(h, sl.T, sl.ld, sl.M, g.t[s], true);
    if (rc) return rc;
  }
  GParams a{};
  a.N = N; a.nz = g.nz; a.nslots = ns;
  for (int s = 0; s < ns; ++s) { a.nblk[s] = h->slot[s].lay.nblk; a.t[s] = g.t[s]; }
  memcpy(a.kind, g.coef_kind, sizeof(a.kind));
  a.coef = g.coef; a.g = g.g;
  a.data_block = (g.pde == PDE_DARCY) ? 3 : -1; a.ndata = g.N_data;
  a.data_scale = (g.pde == PDE_DARCY) ? 2.0 / (g.noise * g.noise) : 0.0;
  a.z = g.z; a.data = g.data_u;
  grad_kernel<<<(N + 255) / 256, 256, 0, h->stream>>>(a);
  h->launches++;
  CUDA_TRY(h, cudaGetLastError());
  return GPP_OK;
}

// g = grad loss(z) and H = Hessian_GN(z, z) at g.z; requires F, s and coef of g.z to be current.
int gn_grad_hess(gpp_handle* h) {
  GnState& g = h->gn;
  const int ns = nslots_of(g);
  const int N = h->N;
  set_kind(g);
  int rc;
  // t = L^{-T} s
  for (int s = 0; s < ns; ++s) {
    GramSlot& sl = h->slot[s];
    CUDA_TRY(h, cudaMemcpyAsync(g.t[s], g.s[s], sizeof(double) * sl.M, cudaMemcpyDeviceToDevice, h->stream));
    rc = trsv_lower(h, sl.T, sl.ld, sl.M, g.t[s], true);
    if (rc) return rc;
  }
  // gradient
  {
    GParams a{};
    a.N = N; a.nz = g.nz; a.nslots = ns;
    for (int s = 0; s < ns; ++s) { a.nblk[s] = h->slot[s].lay.nblk; a.t[s] = g.t[s]; }
    memcpy(a.kind, g.coef_kind, sizeof(a.kind));
    a.coef = g.coef; a.g = g.g;
    a.data_block = (g.pde == PDE_DARCY) ? 3 : -1; a.ndata = g.N_data;
    a.data_scale = (g.pde == PDE_DARCY) ? 2.0 / (g.noise * g.noise) : 0.0;
    a.z = g.z; a.data = g.data_u;
    grad_kernel<<<(N + 255) / 256, 256, 0, h->stream>>>(a);
    h->launches++;
  }
  // Hessian
  {
    HParams a{};
    if (make_term_table(g.pde, &a.tt)) { h->err = "term table overflow"; return -1; }
    a.N = N; a.coef = g.coef;
    for (int s = 0; s < ns; ++s) { a.A[s] = h->slot[s].Ainv; a.ldA[s] = h->slot[s].ldA; }
    a.H = g.H; a.ldH = g.ldH;
    a.data_block = (g.pde == PDE_DARCY) ? 3 : -1; a.ndata = g.N_data;
    a.data_diag = (g.pde == PDE_DARCY) ? 2.0 / (g.noise * g.noise) : 0.0;
    dim3 grid((N + 63) / 64, (N + 15) / 16, g.nz * g.nz);
    hess_kernel<<<grid, 256, 0, h->stream>>>(a);
    h->launches++;
    CUDA_TRY(h, cudaGetLastError());
  }
  if (g.pde == PDE_ELLIPTIC_RELAXED) {
    const double* ss2 = g.coef + ((long)((1 * GPP_MAX_BLOCKS + 0) * GPP_MAX_ZBLOCKS + 0)) * N;
    const double* cc = g.coef + ((long)((1 * GPP_MAX_BLOCKS + 0) * GPP_MAX_ZBLOCKS + 1)) * N;
    relax_penalty_kernel<<<(N + 255) / 256, 256, 0, h->stream>>>(N, 2.0 / g.params[3], ss2, cc, g.H, g.ldH, g.g);
    h->launches++;
  }
  return GPP_OK;
}

// One GN step at g.z; requires F, s and coef of g.z to be current (gn_loss leaves them so).
int gn_step(gpp_handle* h, double step, double* loss_host) {
  GnState& g = h->gn;
  set_kind(g);
  int rc;
  static const bool trace = getenv("GPP_TRACE") != nullptr;
  auto mark = [&](int k) { if (trace) cudaEventRecord(h->ev[2 + k], h->stream); };
  if (!g.current) {            // z was replaced since the last loss evaluation: refresh F, s and the coefficients
    double dummy;
    rc = gn_loss(h, g.z, &dummy);
    if (rc) return rc;
  }
  mark(0);
  mark(1);
  if (h->dist_gn) {
    // sharded: gradient replicated, Hessian blocks by their owners, distributed Cholesky of H (dist.cu)
    rc = gn_grad(h);
    if (rc) return rc;
    mark(2);
    rc = dist_gn_hess_potrf(h);
    if (rc) return rc;
  } else {
    rc = gn_grad_hess(h);
    if (rc) return rc;
    mark(2);
    // delta = H^{-1} g via Cholesky (H is SPD: 2 S^T S + data term)
    rc = potrf_lower(h, g.H, g.ldH, g.n, &g.mapH);
    if (rc) return rc;
  }
  mark(3);
  rc = trsv_lower(h, g.H, g.ldH, g.n, g.g, false);
  if (rc) return rc;
  rc = trsv_lower(h, g.H, g.ldH, g.n, g.g, true);
  if (rc) return rc;
  axpy_kernel<<<(g.n + 255) / 256, 256, 0, h->stream>>>(g.z, g.g, step, g.n);
  h->launches++;
  CUDA_TRY(h, cudaGetLastError());
  g.current = false;
  mark(4);
  rc = gn_loss(h, g.z, loss_host);
  if (trace && !rc) {
    mark(5);
    cudaEventSynchronize(h->ev[7]);
    float t[5];
    for (int k = 0; k < 5; ++k) cudaEventElapsedTime(&t[k], h->ev[2 + k], h->ev[3 + k]);
    fprintf(stderr, "[gpp trace] gn_step: setup %.2f ms | trsv L^T + grad + hess %.2f | potrf(H) %.2f | trsv H x2 + axpy %.2f | F, trsv L, loss %.2f\n",
            t[0], t[1], t[2], t[3], t[4]);
  }
  return rc;
}
