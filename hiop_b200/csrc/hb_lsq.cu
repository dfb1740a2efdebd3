// Least-squares multiplier update of the quasi-Newton driver on the device (SURVEY 8 f2).
//
// Reference: hiopDualsLsqUpdateLinsysRedDense::do_lsq_update   src/Optimization/hiopDualsUpdater.cpp:232-332
//            hiopDualsLsqUpdateLinsysRedDenseSymPD::{factorize_mat, solve_with_factors} (DPOTRF / DPOTRS)  :690-735
//
//   [ Jc Jc^T   Jc Jd^T     ] [yc]     [ Jc  0 ] [ grad_f - zl + zu ]
//   [   .       Jd Jd^T + I ] [yd] = - [ Jd  I ] [     vl - vu      ]
//
// The reference runs three DGEMMs (Jc Jc^T, Jc Jd^T, Jd Jd^T) that each stream the Jacobians; here J J^T is one pass of the
// same symmetric kernel that condenses the KKT system (diagonal = I), followed by the blocked Cholesky of hb_dense.cu.
#include "hb_lowrank.cuh"
#include "hb_dense.cuh"
#include "../../include/hiopb200.h"

int hb_syrk_rows(hb_ctx* c, int M, long long K, const double* const* rowptr_dev, bool aligned16, const double* d, double* C, int ldc);
int hb_syrk_rows_ozaki(hb_ctx* c, int M, long long K, const double* const* rowptr_dev, bool rows_aligned16, const double* d, double* C, int ldc, int S,
                       const double* dot_x, double* dot_out, int* chunks_out);

namespace {
constexpr int ET = 256;
// vecx = (grad_f - zl) + zu                                                             :281-283
__global__ void __launch_bounds__(ET)
k_lsq_vecx(long long n, const double* __restrict__ g, const double* __restrict__ zl, const double* __restrict__ zu, double* __restrict__ out)
{
  const long long stride = (long long)gridDim.x * ET;
  for(long long i = (long long)blockIdx.x * ET + threadIdx.x; i < n; i += stride) out[i] = __dadd_rn(__dsub_rn(g[i], zl[i]), zu[i]);
}
// M[me+i][me+i] += 1;  rhs[me+i] -= vl[i] - vu[i]                                       :246, 284-289
__global__ void k_lsq_dpart(int me, int mi, int m, double* __restrict__ M, double* __restrict__ rhs, const double* __restrict__ vl,
                            const double* __restrict__ vu)
{
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if(i < mi) {
    M[(size_t)(me + i) * m + me + i] += 1.0;
    rhs[me + i] = __dsub_rn(rhs[me + i], __dsub_rn(vl[i], vu[i]));
  }
}
} // namespace

extern "C" int hb_lowrank_lsq_duals(hb_lowrank* k, const double* grad_f, const double* zl, const double* zu, const double* vl, const double* vu,
                                    double* yc, double* yd)
{
  HB_REQUIRE(k, "null handle");
  HB_REQUIRE(k->m == 0 || k->J, "hb_lowrank_lsq_duals: register the Jacobian with hb_lowrank_set_jacobian first");
  HB_REQUIRE(k->n == 0 || (grad_f && zl && zu), "hb_lowrank_lsq_duals: null x block");
  HB_REQUIRE(k->mineq == 0 || (vl && vu && yd), "hb_lowrank_lsq_duals: null d block");
  HB_REQUIRE(k->meq == 0 || yc, "hb_lowrank_lsq_duals: null yc");
  hb_ctx* c = k->ctx;
  const int m = k->m, me = k->meq, mi = k->mineq;
  const long long n = k->n;
  if(m == 0) return HB_OK;
  if(!k->lsq_M && cudaMalloc(&k->lsq_M, sizeof(double) * ((size_t)m * m + 2 * m)) != cudaSuccess) {
    cudaGetLastError();
    return hb_fail(HB_ERR_ALLOC, "LSQ workspace allocation failed%s", "");
  }
  double* M = k->lsq_M;
  double* rhs = M + (size_t)m * m;
  HB_CHECK(hb_lr_refresh_rowptr(k));
  // J J^T: rows 0..m-1 of the row-pointer table are the Jacobian rows
  int mode = k->condense_mode;
  if(mode < 0) {
    long long ng = n;
    HB_CHECK(hb_lr_global_n(k, &ng));
    mode = (ng >= 32768 && m >= 64) ? 8 : 0;
  }
  if(mode == 0) HB_CHECK(hb_syrk_rows(c, m, n, k->rowptr_dev, k->rows_aligned, nullptr, M, m));
  else HB_CHECK(hb_syrk_rows_ozaki(c, m, n, k->rowptr_dev, k->rows_aligned, nullptr, M, m, mode, nullptr, nullptr, nullptr));
  HB_CHECK(hb_allreduce_sum(c, M, (long long)m * m));
  // rhs = -J vecx (all-reduced), then the d-side terms on the replicated part
  if(n > 0) {
    long long g = (n + ET - 1) / ET;
    const long long cap = (long long)c->num_sms * 8;
    k_lsq_vecx<<<(int)(g > cap ? cap : g), ET, 0, c->stream>>>(n, grad_f, zl, zu, k->nv1);
    HB_LAUNCHED();
  }
  HB_CHECK(hb_lr_gemv_rows(k, k->J, m, 0.0, rhs, -1.0, k->nv1));
  if(mi > 0) {
    k_lsq_dpart<<<(mi + 127) / 128, 128, 0, c->stream>>>(me, mi, m, M, rhs, vl, vu);
    HB_LAUNCHED();
  }
  HB_CUDA(cudaMemsetAsync(k->info + 3, 0, sizeof(int), c->stream));
  HB_CHECK(hb_dense_factor_blocked(c, m, M, m, false, nullptr, k->info + 3));
  HB_CHECK(hb_dense_tri_solve(c, m, M, m, false, rhs));
  HB_CUDA(cudaMemcpyAsync(k->info_host + 3, k->info + 3, sizeof(int), cudaMemcpyDeviceToHost, c->stream));
  if(me) HB_CUDA(cudaMemcpyAsync(yc, rhs, sizeof(double) * me, cudaMemcpyDeviceToDevice, c->stream));
  if(mi) HB_CUDA(cudaMemcpyAsync(yd, rhs + me, sizeof(double) * mi, cudaMemcpyDeviceToDevice, c->stream));
  HB_CUDA(cudaStreamSynchronize(c->stream));
  if(k->info_host[3] != 0) { // "dpotrf (Chol fact) detected %d minor being indefinite" :722-725 -> the driver keeps the old duals
    snprintf(g_hb_err, sizeof(g_hb_err), "hb_lowrank_lsq_duals: J J^T + I is not SPD (leading minor %d)", k->info_host[3]);
    return HB_ERR_NUMERIC;
  }
  return HB_OK;
}
