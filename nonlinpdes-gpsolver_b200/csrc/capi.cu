// extern "C" entry points of libgpp_b200.so (declared in include/gpp.h).
#include "../../include/gpp.h"
#include "gpp_internal.cuh"

#include <cstring>

#include <nvtx3/nvToolsExt.h>   // header-only; ranges are no-ops unless a profiler (ncu / nsys) is attached

namespace {

// NVTX range per hot-path phase (the reference has no tracing at all, SURVEY section 5)
struct NvtxRange {
  explicit NvtxRange(const char* name) { nvtxRangePushA(name); }
  ~NvtxRange() { nvtxRangePop(); }
};

__global__ void get_diag_kernel(const double* __restrict__ T, long ld, int M, double* __restrict__ out) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < M) out[i] = T[(long)i * ld + i];
}
__global__ void add_diag_kernel(double* __restrict__ T, long ld, int M, const double* __restrict__ add) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < M) T[(long)i * ld + i] = T[(long)i * ld + i] + add[i];
}
// dense copy-out: mode 0 symmetric from lower, mode 1 lower with zeros above, mode 2 plain
__global__ void pack_kernel(const double* __restrict__ T, long ld, int M, int mode, double* __restrict__ out) {
  long e = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= (long)M * M) return;
  int i = (int)(e / M), j = (int)(e % M);
  double v;
  if (mode == 2 || j <= i) v = T[(long)i * ld + j];
  else v = (mode == 0) ? T[(long)j * ld + i] : 0.0;
  out[e] = v;
}
__global__ void unpack_kernel(const double* __restrict__ in, int M, double* __restrict__ T, long ld) {
  long e = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= (long)M * M) return;
  int i = (int)(e / M), j = (int)(e % M);
  if (j <= i) T[(long)i * ld + j] = in[e];
}

// grow-only device buffers (gpp_internal.cuh: dev_reserve): repeated solves on a handle never touch the allocator
int dev_alloc(gpp_handle* h, double** p, size_t n) { return dev_reserve(h, p, n); }
void dev_free(double*& p) { if (p) { cudaFree(p); p = nullptr; } }

int ensure_work(gpp_handle* h, size_t bytes) {
  if (h->work_bytes >= bytes) return GPP_OK;
  if (h->work) cudaFree(h->work);
  h->work = nullptr; h->work_bytes = 0;
  CUDA_TRY(h, cudaMalloc(&h->work, bytes));
  h->work_bytes = bytes;
  return GPP_OK;
}

bool bad_slot(gpp_handle* h, int slot, bool need_T = true) {
  if (!h) return true;
  if (slot < 0 || slot >= GPP_MAX_SLOTS) { h->err = "bad slot"; return true; }
  if (need_T && !h->slot[slot].T) { h->err = "slot not assembled"; return true; }
  return false;
}

}  // namespace

int gram_slot_prepare(gpp_handle* h, int slot, int layout, int kernel, const double* kparams) {
  if (bad_slot(h, slot, false)) return -2;
  if (!h->Xall) { h->err = "points not set"; return -1; }
  if (layout < 0 || layout > 3) { h->err = "bad layout"; return -3; }
  if (kernel < 0 || kernel > 1) { h->err = "bad kernel"; return -4; }
  if (!kparams) { h->err = "kparams missing"; return -5; }
  CUDA_TRY(h, cudaSetDevice(h->device));
  GramSlot& s = h->slot[slot];
  s.layout_id = layout;
  s.lay = make_layout(layout);
  s.N = h->N; s.Nb = (layout == LAY_DARCY_A) ? 0 : h->Nb;
  int o = 0;
  for (int p = 0; p < s.lay.nblk; ++p) { s.off[p] = o; o += s.N + (s.lay.with_bdy[p] ? s.Nb : 0); }
  s.off[s.lay.nblk] = o;
  s.M = o; s.ld = round_up(s.M, 16);
  int rc = dev_alloc(h, &s.T, (size_t)s.M * s.ld);
  if (rc) return rc;
  rc = make_tensor_map(h, &s.mapT, s.T, s.M, s.M, s.ld);     // host-side encode only; M / ld may have changed
  if (rc) return rc;
  s.Mint = s.lay.nblk * s.N;
  s.kernel_id = kernel;
  s.kp_b1 = kparams[0]; s.kp_b2 = kparams[1]; s.kp_e1 = kparams[2]; s.kp_e2 = kparams[3];
  s.factored = s.inverted = false;
  h->dist_gn = false;
  return GPP_OK;
}

extern "C" {

int gpp_create(int device, gpp_handle** out) {
  if (!out) return -2;
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) return GPP_CUDA_ERR;   // no CPU fallback
  if (device < 0 || device >= ndev) return -1;
  gpp_handle* h = new gpp_handle();
  h->device = device;
  if (cudaSetDevice(device) != cudaSuccess) { delete h; return GPP_CUDA_ERR; }
  cudaDeviceProp prop;
  cudaGetDeviceProperties(&prop, device);
  if (prop.major < 10) {   // sm_100a-only binary
    delete h;
    return GPP_CUDA_ERR + 1;
  }
  if (cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking) != cudaSuccess) { delete h; return GPP_CUDA_ERR; }
  h->cur = h->stream;
  {
    int lo = 0, hi = 0;
    cudaDeviceGetStreamPriorityRange(&lo, &hi);   // hi = greatest priority (numerically lowest)
    cudaStreamCreateWithPriority(&h->sP, cudaStreamNonBlocking, hi);
    cudaStreamCreateWithPriority(&h->sG[0], cudaStreamNonBlocking, lo);
    cudaStreamCreateWithPriority(&h->sG[1], cudaStreamNonBlocking, lo);
  }
  for (auto& e : h->ev) cudaEventCreate(&e);
  cudaMalloc(&h->d_info, sizeof(int));
  cudaMemset(h->d_info, 0, sizeof(int));
  cudaMalloc(&h->gn.scal, 64 * sizeof(double));
  *out = h;
  return GPP_OK;
}

int gpp_destroy(gpp_handle* h) {
  if (h) cudaSetDevice(h->device);
  if (!h) return -1;
  cudaSetDevice(h->device);
  cudaStreamSynchronize(h->stream);
  if (h->dist) gpp_dist_finalize(h);       // NCCL communicator + the distributed buffers
  dist_local_release(h);
  dev_free(h->Xd); dev_free(h->Xb); dev_free(h->Xall);
  for (auto& s : h->slot) { dev_free(s.T); dev_free(s.udiag); dev_free(s.Ainv); }
  GnState& g = h->gn;
  dev_free(g.rhs_f); dev_free(g.bdy_g); dev_free(g.data_u); dev_free(g.z); dev_free(g.coef); dev_free(g.H); dev_free(g.g);
  dev_free(g.scal);
  for (int s = 0; s < GPP_MAX_SLOTS; ++s) { dev_free(g.F[s]); dev_free(g.s[s]); dev_free(g.t[s]); }
  dev_free(h->var_W); dev_free(h->var_io); dev_free(h->var_aux);
  if (h->work) cudaFree(h->work);
  if (h->d_info) cudaFree(h->d_info);
  if (h->d_trsv_flag) cudaFree(h->d_trsv_flag);
  if (h->d_bar) cudaFree(h->d_bar);
  for (auto& e : h->ev) cudaEventDestroy(e);
  for (auto& e : h->evpool) cudaEventDestroy(e);
  if (h->sP) cudaStreamDestroy(h->sP);
  for (auto& sg : h->sG) if (sg) cudaStreamDestroy(sg);
  cudaStreamDestroy(h->stream);
  delete h;
  return GPP_OK;
}

const char* gpp_last_error(gpp_handle* h) { return h ? h->err.c_str() : "null handle"; }

int gpp_set_option(gpp_handle* h, const char* name, double value) {
  if (h) cudaSetDevice(h->device);
  if (!h || !name) return -1;
  if (!strcmp(name, "NB")) {
    int nb = (int)value;
    if (nb < 128 || nb % 128) { h->err = "NB must be a positive multiple of 128"; return -3; }
    h->NB = nb;
    return GPP_OK;
  }
  if (!strcmp(name, "lookahead")) { h->lookahead = value != 0.0; return GPP_OK; }
  if (!strcmp(name, "tiled_potrf")) { h->tiled_potrf = value != 0.0; return GPP_OK; }
  if (!strcmp(name, "tiled_max_n")) { h->tiled_max_n = (int)value; return GPP_OK; }
  if (!strcmp(name, "tiled_grid_limit")) { h->tiled_grid_limit = (int)value; return GPP_OK; }
  if (!strcmp(name, "persistent_gemm")) { h->persistent_gemm = value != 0.0; return GPP_OK; }
  if (!strcmp(name, "blocksum")) { h->blocksum = value != 0.0; return GPP_OK; }
  if (!strcmp(name, "rl_potrf")) { h->rl_potrf = value != 0.0; return GPP_OK; }
  if (!strcmp(name, "fused_trsm_rows")) { h->fused_trsm_rows = (int)value; return GPP_OK; }
  if (!strcmp(name, "gemm_tile")) {
    const int t = (int)value;
    if (t != 0 && t != 64 && t != 128) { h->err = "gemm_tile must be 0, 64 or 128"; return -3; }
    h->force_tile = t;
    return GPP_OK;
  }
  h->err = std::string("unknown option ") + name;
  return -2;
}

int gpp_sync(gpp_handle* h) {
  if (h) cudaSetDevice(h->device);
  if (!h) return -1;
  CUDA_TRY(h, cudaStreamSynchronize(h->stream));
  return GPP_OK;
}

long gpp_launch_count(gpp_handle* h) { return h ? h->launches : -1; }

int gpp_timer_start(gpp_handle* h) {
  if (h) cudaSetDevice(h->device);
  if (!h) return -1;
  CUDA_TRY(h, cudaEventRecord(h->ev[0], h->stream));
  return GPP_OK;
}
int gpp_timer_stop(gpp_handle* h, float* ms) {
  if (h) cudaSetDevice(h->device);
  if (!h || !ms) return -1;
  CUDA_TRY(h, cudaEventRecord(h->ev[1], h->stream));
  CUDA_TRY(h, cudaEventSynchronize(h->ev[1]));
  CUDA_TRY(h, cudaEventElapsedTime(ms, h->ev[0], h->ev[1]));
  return GPP_OK;
}

int gpp_timer2_start(gpp_handle* h) {
  if (h) cudaSetDevice(h->device);
  if (!h) return -1;
  CUDA_TRY(h, cudaEventRecord(h->ev[8], h->stream));
  return GPP_OK;
}
int gpp_timer2_stop(gpp_handle* h, float* ms) {
  if (h) cudaSetDevice(h->device);
  if (!h || !ms) return -1;
  CUDA_TRY(h, cudaEventRecord(h->ev[9], h->stream));
  CUDA_TRY(h, cudaEventSynchronize(h->ev[9]));
  CUDA_TRY(h, cudaEventElapsedTime(ms, h->ev[8], h->ev[9]));
  return GPP_OK;
}

int gpp_set_points(gpp_handle* h, const double* Xd, int N, const double* Xb, int Nb) {
  if (h) cudaSetDevice(h->device);
  if (!h) return -1;
  if (!Xd || N <= 0) { h->err = "X_domain missing"; return -2; }
  if (Nb < 0 || (Nb > 0 && !Xb)) { h->err = "X_boundary missing"; return -4; }
  CUDA_TRY(h, cudaSetDevice(h->device));
  h->N = N; h->Nb = Nb;
  int rc = dev_alloc(h, &h->Xall, (size_t)(N + Nb) * 2);
  if (rc) return rc;
  CUDA_TRY(h, cudaMemcpyAsync(h->Xall, Xd, sizeof(double) * 2 * N, cudaMemcpyHostToDevice, h->stream));
  if (Nb) CUDA_TRY(h, cudaMemcpyAsync(h->Xall + 2 * (size_t)N, Xb, sizeof(double) * 2 * Nb, cudaMemcpyHostToDevice, h->stream));
  CUDA_TRY(h, cudaStreamSynchronize(h->stream));
  for (auto& s : h->slot) { s.factored = s.inverted = false; }
  h->gn.ready = false;
  return GPP_OK;
}

int gpp_gram_assemble(gpp_handle* h, int slot, int layout, int kernel, const double* kparams) {
  NvtxRange nvtx_range("gpp:gram_assemble");
  if (h) cudaSetDevice(h->device);
  int rc = gram_slot_prepare(h, slot, layout, kernel, kparams);
  if (rc) return rc;
  return gram_assemble(h, h->slot[slot]);
}

int gpp_gram_size(gpp_handle* h, int slot, int* M, int* Mint) {
  if (h) cudaSetDevice(h->device);
  if (bad_slot(h, slot)) return -2;
  if (M) *M = h->slot[slot].M;
  if (Mint) *Mint = h->slot[slot].Mint;
  return GPP_OK;
}

int gpp_gram_get_diag(gpp_handle* h, int slot, double* out) {
  if (h) cudaSetDevice(h->device);
  if (bad_slot(h, slot)) return -2;
  if (!out) return -3;
  GramSlot& s = h->slot[slot];
  int rc = ensure_work(h, sizeof(double) * s.M);
  if (rc) return rc;
  get_diag_kernel<<<(s.M + 255) / 256, 256, 0, h->stream>>>(s.T, s.ld, s.M, h->work);
  h->launches++;
  CUDA_TRY(h, cudaMemcpyAsync(out, h->work, sizeof(double) * s.M, cudaMemcpyDeviceToHost, h->stream));
  CUDA_TRY(h, cudaStreamSynchronize(h->stream));
  return GPP_OK;
}

int gpp_gram_add_diag(gpp_handle* h, int slot, const double* add) {
  if (h) cudaSetDevice(h->device);
  if (bad_slot(h, slot)) return -2;
  if (!add) return -3;
  GramSlot& s = h->slot[slot];
  int rc = ensure_work(h, sizeof(double) * s.M);
  if (rc) return rc;
  CUDA_TRY(h, cudaMemcpyAsync(h->work, add, sizeof(double) * s.M, cudaMemcpyHostToDevice, h->stream));
  add_diag_kernel<<<(s.M + 255) / 256, 256, 0, h->stream>>>(s.T, s.ld, s.M, h->work);
  h->launches++;
  CUDA_TRY(h, cudaStreamSynchronize(h->stream));
  return GPP_OK;
}

int gpp_gram_download(gpp_handle* h, int slot, int what, double* out) {
  if (h) cudaSetDevice(h->device);
  if (bad_slot(h, slot)) return -2;
  if (!out || what < 0 || what > 2) return -3;
  GramSlot& s = h->slot[slot];
  const double* src = s.T; long ld = s.ld; int M = s.M; int mode = what;
  if (what == 2) {
    if (!s.inverted) { h->err = "inverse not computed"; return -4; }
    src = s.Ainv; ld = s.ldA; M = s.Mint;
  }
  const size_t bytes = sizeof(double) * (size_t)M * M;
  double* tmp = nullptr;
  CUDA_TRY(h, cudaMalloc(&tmp, bytes));
  const long tot = (long)M * M;
  pack_kernel<<<(unsigned)((tot + 255) / 256), 256, 0, h->stream>>>(src, ld, M, mode, tmp);
  h->launches++;
  cudaError_t e = cudaMemcpyAsync(out, tmp, bytes, cudaMemcpyDeviceToHost, h->stream);
  if (e == cudaSuccess) e = cudaStreamSynchronize(h->stream);
  cudaFree(tmp);
  CUDA_TRY(h, e);
  return GPP_OK;
}

int gpp_gram_upload(gpp_handle* h, int slot, const double* theta) {
  if (h) cudaSetDevice(h->device);
  if (bad_slot(h, slot)) return -2;
  if (!theta) return -3;
  GramSlot& s = h->slot[slot];
  const size_t bytes = sizeof(double) * (size_t)s.M * s.M;
  double* tmp = nullptr;
  CUDA_TRY(h, cudaMalloc(&tmp, bytes));
  cudaError_t e = cudaMemcpyAsync(tmp, theta, bytes, cudaMemcpyHostToDevice, h->stream);
  const long tot = (long)s.M * s.M;
  unpack_kernel<<<(unsigned)((tot + 255) / 256), 256, 0, h->stream>>>(tmp, s.M, s.T, s.ld);
  h->launches++;
  if (e == cudaSuccess) e = cudaStreamSynchronize(h->stream);
  cudaFree(tmp);
  CUDA_TRY(h, e);
  s.factored = s.inverted = false;
  return GPP_OK;
}

int gpp_potrf(gpp_handle* h, int slot, int* info) {
  NvtxRange nvtx_range("gpp:potrf");
  if (h) cudaSetDevice(h->device);
  if (bad_slot(h, slot)) return -2;
  CUDA_TRY(h, cudaSetDevice(h->device));
  GramSlot& s = h->slot[slot];
  if (s.factored) { h->err = "already factored"; return -3; }
  // large slots: right-looking schedule with block summation (robust at nuggets ~1e-13, see gpp_internal.cuh);
  // small ones: the persistent tiled kernel inside potrf_lower
  int rc = (h->rl_potrf && s.M > h->tiled_max_n) ? potrf_right_looking(h, s.T, s.ld, s.M, &s.mapT)
                                                  : potrf_lower(h, s.T, s.ld, s.M, &s.mapT);
  if (rc) return rc;
  int hinfo = 0;
  CUDA_TRY(h, cudaMemcpyAsync(&hinfo, h->d_info, sizeof(int), cudaMemcpyDeviceToHost, h->stream));
  CUDA_TRY(h, cudaStreamSynchronize(h->stream));
  if (info) *info = hinfo;
  s.factored = true;
  s.inverted = false;
  return GPP_OK;
}

int gpp_inverse(gpp_handle* h, int slot) {
  NvtxRange nvtx_range("gpp:inverse");
  if (h) cudaSetDevice(h->device);
  if (bad_slot(h, slot)) return -2;
  CUDA_TRY(h, cudaSetDevice(h->device));
  GramSlot& s = h->slot[slot];
  if (!s.factored) { h->err = "potrf first"; return -3; }
  const int NB = h->NB;
  const long nblk = (s.M + NB - 1) / NB;
  int rc = dev_alloc(h, &s.udiag, (size_t)nblk * NB * NB);
  if (rc) return rc;
  rc = make_tensor_map(h, &s.mapUdiag, s.udiag, s.M, NB, NB);
  if (rc) return rc;
  s.ldA = round_up(s.Mint, 16);
  rc = dev_alloc(h, &s.Ainv, (size_t)s.Mint * s.ldA);          // sized for the present Mint (grow-only)
  if (rc) return rc;
  rc = inverse_interior(h, s);
  if (rc) return rc;
  s.inverted = true;
  return GPP_OK;
}

int gpp_solve_vec(gpp_handle* h, int slot, const double* b, double* x) {
  if (h) cudaSetDevice(h->device);
  if (bad_slot(h, slot)) return -2;
  if (!b || !x) return -3;
  GramSlot& s = h->slot[slot];
  if (!s.factored) { h->err = "potrf first"; return -4; }
  int rc = ensure_work(h, sizeof(double) * s.M);
  if (rc) return rc;
  CUDA_TRY(h, cudaMemcpyAsync(h->work, b, sizeof(double) * s.M, cudaMemcpyHostToDevice, h->stream));
  rc = trsv_lower(h, s.T, s.ld, s.M, h->work, false);
  if (rc) return rc;
  rc = trsv_lower(h, s.T, s.ld, s.M, h->work, true);
  if (rc) return rc;
  CUDA_TRY(h, cudaMemcpyAsync(x, h->work, sizeof(double) * s.M, cudaMemcpyDeviceToHost, h->stream));
  CUDA_TRY(h, cudaStreamSynchronize(h->stream));
  return GPP_OK;
}

int gpp_gn_setup(gpp_handle* h, int pde, const double* params, const double* rhs_f, const double* bdy_g,
                 const double* data_u, int N_data, double noise) {
  if (h) cudaSetDevice(h->device);
  if (!h) return -1;
  if (pde < 0 || pde > 4) { h->err = "bad pde"; return -2; }
  if (!rhs_f || (h->Nb > 0 && !bdy_g)) { h->err = "rhs_f / bdy_g missing"; return -4; }
  CUDA_TRY(h, cudaSetDevice(h->device));
  GnState& g = h->gn;
  const int N = h->N, Nb = h->Nb;
  g.pde = pde;
  g.nz = pde_nz(pde);
  g.n = g.nz * N;
  memset(g.params, 0, sizeof(g.params));
  g.m_int = 0;
  if (pde == PDE_ELLIPTIC || pde == PDE_ELLIPTIC_RELAXED) {
    if (!params) return -3;
    g.params[0] = params[0]; g.params[1] = params[1]; g.params[2] = params[0] * params[1];
    if (pde == PDE_ELLIPTIC_RELAXED) {
      if (!(params[2] > 0.0)) { h->err = "pen_lambda must be positive"; return -3; }
      g.params[3] = params[2];
    }
    const double m = params[1];
    g.m_int = (m == (double)(int)m && m >= 1.0 && m <= 64.0) ? (int)m : 0;
  } else if (pde == PDE_BURGERS) {
    if (!params) return -3;
    g.params[0] = params[0]; g.params[1] = params[1]; g.params[2] = -params[0];
  } else if (pde == PDE_EIKONAL) {
    if (!params) return -3;
    g.params[0] = params[0];
  }
  const int need_slots = (pde == PDE_DARCY) ? 2 : 1;
  const int want_layout[2] = {(pde == PDE_ELLIPTIC || pde == PDE_ELLIPTIC_RELAXED) ? LAY_ELLIPTIC : (pde == PDE_BURGERS ? LAY_BURGERS : LAY_EIKONAL), LAY_DARCY_A};
  for (int s = 0; s < need_slots; ++s) {
    if (!h->slot[s].T || h->slot[s].layout_id != want_layout[s]) { h->err = "Gram slot missing or wrong layout for this PDE"; return -5; }
  }
  int rc;
  if ((rc = dev_alloc(h, &g.rhs_f, N))) return rc;
  if ((rc = dev_alloc(h, &g.bdy_g, Nb > 0 ? Nb : 1))) return rc;
  CUDA_TRY(h, cudaMemcpyAsync(g.rhs_f, rhs_f, sizeof(double) * N, cudaMemcpyHostToDevice, h->stream));
  if (Nb) CUDA_TRY(h, cudaMemcpyAsync(g.bdy_g, bdy_g, sizeof(double) * Nb, cudaMemcpyHostToDevice, h->stream));
  g.N_data = 0; g.noise = 1.0;
  if (pde == PDE_DARCY) {
    if (N_data < 0 || N_data > N || (N_data > 0 && !data_u) || !(noise > 0)) { h->err = "bad observation data"; return -6; }
    g.N_data = N_data; g.noise = noise;
    if ((rc = dev_alloc(h, &g.data_u, N_data > 0 ? N_data : 1))) return rc;
    if (N_data) CUDA_TRY(h, cudaMemcpyAsync(g.data_u, data_u, sizeof(double) * N_data, cudaMemcpyHostToDevice, h->stream));
  }
  if ((rc = dev_alloc(h, &g.z, g.n))) return rc;
  if ((rc = dev_alloc(h, &g.g, g.n))) return rc;
  if ((rc = dev_alloc(h, &g.coef, (size_t)GPP_MAX_SLOTS * GPP_MAX_BLOCKS * GPP_MAX_ZBLOCKS * N))) return rc;
  for (int s = 0; s < need_slots; ++s) {
    const int M = h->slot[s].M;
    if ((rc = dev_alloc(h, &g.F[s], M))) return rc;
    if ((rc = dev_alloc(h, &g.s[s], M))) return rc;
    if ((rc = dev_alloc(h, &g.t[s], M))) return rc;
  }
  g.ldH = round_up(g.n, 16);
  if ((rc = dev_alloc(h, &g.H, (size_t)g.n * g.ldH))) return rc;
  if ((rc = make_tensor_map(h, &g.mapH, g.H, g.n, g.n, g.ldH))) return rc;
  CUDA_TRY(h, cudaMemsetAsync(g.z, 0, sizeof(double) * g.n, h->stream));
  CUDA_TRY(h, cudaStreamSynchronize(h->stream));
  g.ready = true;
  g.current = false;
  return GPP_OK;
}

int gpp_gn_set_z(gpp_handle* h, const double* z) {
  if (h) cudaSetDevice(h->device);
  if (!h || !h->gn.ready) return -1;
  if (!z) return -2;
  CUDA_TRY(h, cudaMemcpyAsync(h->gn.z, z, sizeof(double) * h->gn.n, cudaMemcpyHostToDevice, h->stream));
  CUDA_TRY(h, cudaStreamSynchronize(h->stream));
  h->gn.current = false;
  return GPP_OK;
}

int gpp_gn_get_z(gpp_handle* h, double* z) {
  if (h) cudaSetDevice(h->device);
  if (!h || !h->gn.ready) return -1;
  if (!z) return -2;
  CUDA_TRY(h, cudaMemcpyAsync(z, h->gn.z, sizeof(double) * h->gn.n, cudaMemcpyDeviceToHost, h->stream));
  CUDA_TRY(h, cudaStreamSynchronize(h->stream));
  return GPP_OK;
}

static int gn_check(gpp_handle* h, bool need_inverse) {
  if (!h) return -1;
  if (!h->gn.ready) { h->err = "gpp_gn_setup first"; return -1; }
  const int ns = h->gn.pde == PDE_DARCY ? 2 : 1;
  for (int s = 0; s < ns; ++s) {
    if (!h->slot[s].factored) { h->err = "gpp_potrf first"; return -2; }
    if (need_inverse && !h->slot[s].inverted) { h->err = "gpp_inverse first"; return -3; }
  }
  return GPP_OK;
}

int gpp_gn_loss(gpp_handle* h, double* loss) {
  NvtxRange nvtx_range("gpp:gn_loss");
  if (h) cudaSetDevice(h->device);
  int rc = gn_check(h, false);
  if (rc) return rc;
  if (!loss) return -4;
  CUDA_TRY(h, cudaSetDevice(h->device));
  return gn_loss(h, h->gn.z, loss);
}

int gpp_gn_step(gpp_handle* h, double step, double* loss) {
  NvtxRange nvtx_range("gpp:gn_step");
  if (h) cudaSetDevice(h->device);
  int rc = gn_check(h, true);
  if (rc) return rc;
  if (!loss) return -4;
  CUDA_TRY(h, cudaSetDevice(h->device));
  return gn_step(h, step, loss);
}

int gpp_gn_grad_hess(gpp_handle* h, double* grad_out, double* hess_out) {
  if (h) cudaSetDevice(h->device);
  int rc = gn_check(h, true);
  if (rc) return rc;
  CUDA_TRY(h, cudaSetDevice(h->device));
  double dummy;
  rc = gn_loss(h, h->gn.z, &dummy);            // F, s = L^{-1} F and the coefficients at the current z
  if (rc) return rc;
  rc = gn_grad_hess(h);
  if (rc) return rc;
  GnState& g = h->gn;
  if (grad_out) CUDA_TRY(h, cudaMemcpyAsync(grad_out, g.g, sizeof(double) * g.n, cudaMemcpyDeviceToHost, h->stream));
  if (hess_out)
    CUDA_TRY(h, cudaMemcpy2DAsync(hess_out, (size_t)g.n * 8, g.H, g.ldH * 8, (size_t)g.n * 8, g.n, cudaMemcpyDeviceToHost, h->stream));
  CUDA_TRY(h, cudaStreamSynchronize(h->stream));
  return GPP_OK;
}

int gpp_gn_residual(gpp_handle* h, int slot, double* F_out) {
  if (h) cudaSetDevice(h->device);
  if (!h || !h->gn.ready) return -1;
  if (bad_slot(h, slot)) return -2;
  if (!F_out) return -3;
  int rc = gn_eval_F(h, h->gn.z, true);
  if (rc) return rc;
  if (!h->gn.F[slot]) { h->err = "slot has no residual"; return -4; }
  CUDA_TRY(h, cudaMemcpyAsync(F_out, h->gn.F[slot], sizeof(double) * h->slot[slot].M, cudaMemcpyDeviceToHost, h->stream));
  CUDA_TRY(h, cudaStreamSynchronize(h->stream));
  return GPP_OK;
}

int gpp_gn_coef(gpp_handle* h, int slot, int p, int q, double* c_out, int* present) {
  if (h) cudaSetDevice(h->device);
  if (!h || !h->gn.ready) return -1;
  if (slot < 0 || slot >= GPP_MAX_SLOTS || p < 0 || p >= GPP_MAX_BLOCKS || q < 0 || q >= GPP_MAX_ZBLOCKS) return -2;
  if (!c_out) return -3;
  h->gn.current = false;
  CUDA_TRY(h, cudaMemsetAsync(h->gn.coef, 0, sizeof(double) * GPP_MAX_SLOTS * GPP_MAX_BLOCKS * GPP_MAX_ZBLOCKS * (size_t)h->N, h->stream));
  int rc = gn_eval_F(h, h->gn.z, true);
  if (rc) return rc;
  const double* src = h->gn.coef + ((long)((slot * GPP_MAX_BLOCKS + p) * GPP_MAX_ZBLOCKS + q)) * h->N;
  CUDA_TRY(h, cudaMemcpyAsync(c_out, src, sizeof(double) * h->N, cudaMemcpyDeviceToHost, h->stream));
  CUDA_TRY(h, cudaStreamSynchronize(h->stream));
  if (present) {
    *present = 0;
    for (int i = 0; i < h->N; ++i) if (c_out[i] != 0.0) { *present = 1; break; }
  }
  return GPP_OK;
}

int gpp_predict(gpp_handle* h, int slot, const double* Xtest, int ntest, const double* w, double* out) {
  NvtxRange nvtx_range("gpp:predict");
  if (h) cudaSetDevice(h->device);
  if (bad_slot(h, slot)) return -2;
  if (!Xtest || ntest <= 0 || !w || !out) return -3;
  CUDA_TRY(h, cudaSetDevice(h->device));
  GramSlot& s = h->slot[slot];
  int rc = ensure_work(h, sizeof(double) * ((size_t)3 * ntest + s.M));
  if (rc) return rc;
  double* d_xt = h->work; double* d_out = d_xt + 2 * (size_t)ntest; double* d_w = d_out + ntest;
  CUDA_TRY(h, cudaMemcpyAsync(d_xt, Xtest, sizeof(double) * 2 * ntest, cudaMemcpyHostToDevice, h->stream));
  CUDA_TRY(h, cudaMemcpyAsync(d_w, w, sizeof(double) * s.M, cudaMemcpyHostToDevice, h->stream));
  rc = gram_predict(h, s, d_xt, ntest, d_w, d_out);
  if (rc) return rc;
  CUDA_TRY(h, cudaMemcpyAsync(out, d_out, sizeof(double) * ntest, cudaMemcpyDeviceToHost, h->stream));
  CUDA_TRY(h, cudaStreamSynchronize(h->stream));
  return GPP_OK;
}

int gpp_theta_test(gpp_handle* h, int slot, const double* Xtest, int ntest, double* out) {
  if (h) cudaSetDevice(h->device);
  if (bad_slot(h, slot)) return -2;
  if (!Xtest || ntest <= 0 || !out) return -3;
  CUDA_TRY(h, cudaSetDevice(h->device));
  GramSlot& s = h->slot[slot];
  const size_t nout = (size_t)ntest * s.M;
  int rc = ensure_work(h, sizeof(double) * ((size_t)2 * ntest + nout));
  if (rc) return rc;
  double* d_xt = h->work; double* d_o = d_xt + 2 * (size_t)ntest;
  CUDA_TRY(h, cudaMemcpyAsync(d_xt, Xtest, sizeof(double) * 2 * ntest, cudaMemcpyHostToDevice, h->stream));
  CUDA_TRY(h, cudaMemsetAsync(d_o, 0, sizeof(double) * nout, h->stream));
  rc = gram_theta_test(h, s, d_xt, ntest, d_o, s.M);
  if (rc) return rc;
  CUDA_TRY(h, cudaMemcpyAsync(out, d_o, sizeof(double) * nout, cudaMemcpyDeviceToHost, h->stream));
  CUDA_TRY(h, cudaStreamSynchronize(h->stream));
  return GPP_OK;
}

int gpp_predict_var(gpp_handle* h, int slot, const double* Xtest, int ntest, double* var_out) {
  NvtxRange nvtx_range("gpp:predict_var");
  if (h) cudaSetDevice(h->device);
  if (bad_slot(h, slot)) return -2;
  if (!Xtest || ntest <= 0 || !var_out) return -3;
  if (!h->slot[slot].factored) { h->err = "potrf first"; return -4; }
  CUDA_TRY(h, cudaSetDevice(h->device));
  int rc = dev_alloc(h, &h->var_io, (size_t)3 * ntest);
  if (rc) return rc;
  double* d_xt = h->var_io; double* d_var = d_xt + 2 * (size_t)ntest;
  CUDA_TRY(h, cudaMemcpyAsync(d_xt, Xtest, sizeof(double) * 2 * ntest, cudaMemcpyHostToDevice, h->stream));
  rc = predict_var(h, slot, d_xt, 0, ntest, d_var);
  if (rc) return rc;
  CUDA_TRY(h, cudaMemcpyAsync(var_out, d_var, sizeof(double) * ntest, cudaMemcpyDeviceToHost, h->stream));
  CUDA_TRY(h, cudaStreamSynchronize(h->stream));
  return GPP_OK;
}

int gpp_kernel_eval(gpp_handle* h, int kernel, const double* kparams, int op_x, int op_y, const double* x1,
                    const double* x2, const double* y1, const double* y2, long n, double* out) {
  if (h) cudaSetDevice(h->device);
  if (!h) return -1;
  if (kernel < 0 || kernel > 1 || !kparams) return -2;
  if (op_x < 0 || op_x > 4 || op_y < 0 || op_y > 4) { h->err = "bad operator id"; return -4; }
  if (n <= 0 || !x1 || !x2 || !y1 || !y2 || !out) return -6;
  CUDA_TRY(h, cudaSetDevice(h->device));
  int rc = ensure_work(h, sizeof(double) * 5 * (size_t)n);
  if (rc) return rc;
  const double* src[4] = {x1, x2, y1, y2};
  for (int k = 0; k < 4; ++k)
    CUDA_TRY(h, cudaMemcpyAsync(h->work + (size_t)k * n, src[k], sizeof(double) * n, cudaMemcpyHostToDevice, h->stream));
  rc = gram_kernel_eval(h, kernel, kparams, op_x, op_y, h->work, n, h->work + 4 * (size_t)n);
  if (rc) return rc;
  CUDA_TRY(h, cudaMemcpyAsync(out, h->work + 4 * (size_t)n, sizeof(double) * n, cudaMemcpyDeviceToHost, h->stream));
  CUDA_TRY(h, cudaStreamSynchronize(h->stream));
  return GPP_OK;
}

}  // extern "C"
