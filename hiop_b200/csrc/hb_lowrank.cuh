// Shared between hb_lowrank.cu and hb_krylov.cu: the quasi-Newton KKT handle and the two Jacobian gemv helpers.
#pragma once
#include "hb_common.cuh"

struct hb_lowrank
{
  hb_ctx* ctx = nullptr;
  long long n = 0;
  int meq = 0, mineq = 0, m = 0, lmax = 0, l = 0;
  double sigma = 1.0;
  // borrowed
  const double *ixl = nullptr, *ixu = nullptr, *idl = nullptr, *idu = nullptr;
  const double *J = nullptr, *St = nullptr, *Yt = nullptr;
  const double *zl = nullptr, *sxl = nullptr, *zu = nullptr, *sxu = nullptr, *vl = nullptr, *sdl = nullptr, *vu = nullptr, *sdu = nullptr;
  // owned
  double *Dx = nullptr, *DhInv = nullptr, *Dd = nullptr, *Dd_inv = nullptr;
  double* Jpack = nullptr;
  const double** rowptr_dev = nullptr;
  const double** rowptr_host = nullptr; // pinned
  bool rows_aligned = false, rowptr_dirty = true;
  double *Caug = nullptr, *SSt = nullptr, *Ld = nullptr, *Dd_sec = nullptr, *V = nullptr, *Mdir = nullptr, *U = nullptr, *Z = nullptr;
  int *ipivV = nullptr, *ipivM = nullptr, *info = nullptr; // info[0]: V, info[1]: N chol, info[2]: M
  double *Nmat = nullptr, *F = nullptr, *svec = nullptr, *rhs = nullptr, *dy = nullptr, *work = nullptr, *stats = nullptr;
  double *nv1 = nullptr, *nv2 = nullptr; // n-vector scratch
  double *p2l = nullptr, *md_partial = nullptr;
  double *mi1 = nullptr, *mi2 = nullptr, *mi3 = nullptr; // m_ineq scratch
  int md_grid = 0;
  bool have_update = false, cond_valid = false, mdir_valid = false;
  int condense_mode = -1; // -1 = auto, 0 = FP64 DMMA, 6/7/8 = INT8-slice tcgen05
  int condense_used = 0;
  long long n_global = -1; // sum of n over the ranks (the auto rule must not depend on the world size); resolved at the first condensation
  bool check_pending = false; // an asynchronous condensation left its info words unchecked
  int fallbacks = 0;          // AUTO-mode condensations the FP64 kernel redid: the int8-slice Cholesky broke down or its slices did not fit
  int condense_chunks = 0;    // column chunks of the last int8-slice condensation (1 = unchunked); 0 = the FP64 kernel ran
  double* tri = nullptr;      // packed upper triangle of C_aug for the all-reduce
  double* tdot = nullptr;     // [J; S; Y] (DhInv .* rx) from the fused row-maximum sweep of an int8-slice condensation (m + 2 lmax)
  bool tdot_valid = false;
  // host staging (hb_lowrank_kkt_system_host)
  double* hbuf[16] = {nullptr};
  double* hJ = nullptr;
  int last_refine = 0;
  double last_resid = 0.0;
  int* info_host = nullptr; // pinned 4 ints
  double* stats_host = nullptr; // pinned 4 doubles
  // BiCGStab workspace (hb_krylov.cu), allocated on first use
  double* kry = nullptr;
  double* kry_m = nullptr; // 2 m-vectors
  // secant memory owned by the engine (hb_secant.cu): S_t, Y_t (lmax x n), previous iterate / gradient / Jacobian
  double *sec_S = nullptr, *sec_Y = nullptr, *sec_xprev = nullptr, *sec_gprev = nullptr, *sec_Jprev = nullptr;
  double sec_L[64 * 64] = {0}, sec_D[64] = {0}; // host copies of L (row-major, stride l) and D; lmax <= 64 in this mode
  // chunked, copy-overlapped condensation of hb_lowrank_kkt_system_host
  cudaStream_t copy_stream = nullptr;
  cudaEvent_t chunk_ev[32] = {nullptr};
  double* Ctmp = nullptr;
  const double** chunk_rowptr_dev = nullptr;
  const double** chunk_rowptr_host = nullptr; // pinned, 32 x (m + 2 lmax)
  double* Finv = nullptr;  // 16 x 16 inverses of the diagonal of F (cooperative Cholesky / solve)
  bool have_finv = false;
  double* lsq_M = nullptr; // m x m LSQ matrix / Cholesky factor + 2 m-vectors (hb_lsq.cu)
  int sec_lcurr = -1, sec_strategy = 1;
  double sec_sigma0 = 1.0;
};


// y = beta*y + alpha*A x over the local columns (+ all-reduce, beta*y on rank 0 only); A is m x n_local row-major
int hb_lr_gemv_rows(hb_lowrank* k, const double* A, int m, double beta, double* y, double alpha, const double* x);
// y = beta*y + alpha*A^T x (local columns only, no reduction)
int hb_lr_gemv_cols(hb_lowrank* k, const double* A, int m, double beta, double* y, double alpha, const double* x);
// k->p2l (device, 2l doubles) = [sigma_s * S (w.*x); Y (w.*x)], all-reduced; w may be NULL
int hb_lr_multidot(hb_lowrank* k, const double* w, const double* x, double sigma_s);
// device table of row pointers [J rows (m); S rows (l); Y rows (l)] -> k->rowptr_dev, k->rows_aligned
int hb_lr_refresh_rowptr(hb_lowrank* k);
// sum of n over the ranks (resolved once, by an all-reduce, when there is a communicator)
int hb_lr_global_n(hb_lowrank* k, long long* n_global);
