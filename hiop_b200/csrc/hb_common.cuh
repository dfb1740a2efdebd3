// Shared internals of libhiopb200.so (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <cstdint>
#include <cstdio>
#include <cstring>
#include <string>
#include <vector>

#include "../../include/hiopb200.h"

#define HB_NUM_SMS_DEFAULT 148

extern thread_local char g_hb_err[512];
extern long long g_hb_launches;

inline int hb_fail(int code, const char* fmt, const char* a = "", int line = 0)
{
  snprintf(g_hb_err, sizeof(g_hb_err), fmt, a, line);
  return code;
}

#define HB_CUDA(call)                                                                              \
  do {                                                                                             \
    cudaError_t e__ = (call);                                                                      \
    if(e__ != cudaSuccess) {                                                                       \
      snprintf(g_hb_err, sizeof(g_hb_err), "%s at %s:%d", cudaGetErrorString(e__), __FILE__, __LINE__); \
      return HB_ERR_CUDA;                                                                          \
    }                                                                                              \
  } while(0)

#define HB_CHECK(expr)                                                                             \
  do {                                                                                             \
    int rc__ = (expr);                                                                             \
    if(rc__ != HB_OK) return rc__;                                                                 \
  } while(0)

#define HB_REQUIRE(cond, msg)                                                                      \
  do {                                                                                             \
    if(!(cond)) {                                                                                  \
      snprintf(g_hb_err, sizeof(g_hb_err), "%s (%s:%d)", msg, __FILE__, __LINE__);                 \
      return HB_ERR_INVALID;                                                                       \
    }                                                                                              \
  } while(0)

// count a launch and check for launch errors
#define HB_LAUNCHED()                                                                              \
  do {                                                                                             \
    g_hb_launches++;                                                                               \
    cudaError_t e__ = cudaGetLastError();                                                          \
    if(e__ != cudaSuccess) {                                                                       \
      snprintf(g_hb_err, sizeof(g_hb_err), "launch failed: %s at %s:%d", cudaGetErrorString(e__), __FILE__, __LINE__); \
      return HB_ERR_CUDA;                                                                          \
    }                                                                                              \
  } while(0)

struct hb_ctx
{
  int device = 0;
  int num_sms = HB_NUM_SMS_DEFAULT;
  cudaStream_t stream = nullptr;
  // scratch for reductions: per-CTA partials + a pinned host landing slot
  double* red_dev = nullptr;     // RED_SLOTS doubles
  double* red_host = nullptr;    // pinned, 64 doubles
  // generic workspace (grown on demand)
  void* ws = nullptr;
  size_t ws_bytes = 0;
  // optional kernel timing (roofline reporting)
  bool timing = false;
  cudaEvent_t ev_syrk0 = nullptr, ev_syrk1 = nullptr;
  bool syrk_timed = false;
  // phase timeline (hb_ctx_phase_timeline): events recorded at fixed points of one update + condense + solve when enabled
  bool phases = false;
  cudaEvent_t ev_phase[16] = {nullptr};
  unsigned phase_mask = 0;
  // per-context state of the int8-slice condensation (hb_ozaki.cu): slice buffer, exponents, tensor maps, work list
  void* oz_state = nullptr;
  void (*oz_free)(void*) = nullptr;
  size_t oz_ws_limit = 0; // bytes of int8 slices the condensation may hold (hb_ctx_set_oz_workspace_limit); 0 = AUTO
  // NCCL
  void* nccl_comm = nullptr;
  int nranks = 1, rank = 0;
};

static constexpr int HB_RED_SLOTS = 4096;

int hb_ws_reserve(hb_ctx* ctx, size_t bytes);

// phase marks of the quasi-Newton step (ids are the HB_PH_* below); a no-op unless hb_ctx_phase_timeline switched them on
enum { HB_PH_START = 0, HB_PH_UPDATE, HB_PH_OZ_ROWMAX, HB_PH_OZ_SLICE, HB_PH_CAUG, HB_PH_ALLREDUCE, HB_PH_VN, HB_PH_CHOL, HB_PH_HSOLVE1, HB_PH_JX, HB_PH_SPDSOLVE, HB_PH_JTY, HB_PH_HSOLVE2, HB_PH_COUNT };
inline void hb_phase_mark(hb_ctx* c, int id)
{
  if(c->phases && c->ev_phase[id]) {
    cudaEventRecord(c->ev_phase[id], c->stream);
    c->phase_mask |= 1u << id;
  }
}

// ---- small device helpers ---------------------------------------------------------------------------------
__device__ __forceinline__ double hb_warp_sum(double v)
{
#pragma unroll
  for(int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ double hb_warp_max(double v)
{
#pragma unroll
  for(int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
__device__ __forceinline__ double hb_warp_min(double v)
{
#pragma unroll
  for(int o = 16; o > 0; o >>= 1) v = fmin(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

// Block-wide sum in a FIXED order (warp shuffles then warp 0) -> deterministic for a fixed launch geometry.
template <int THREADS>
__device__ __forceinline__ double hb_block_sum(double v, double* sm /* >= THREADS/32 doubles */)
{
  v = hb_warp_sum(v);
  const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
  __syncthreads();
  if(l == 0) sm[w] = v;
  __syncthreads();
  double r = 0.0;
  if(w == 0) {
    r = (l < THREADS / 32) ? sm[l] : 0.0;
    r = hb_warp_sum(r);
  }
  return r; // valid on warp 0 (all lanes)
}

// stream-K style even split of `total` items over `parts`
__host__ __device__ inline long long hb_part_begin(long long total, int parts, int p)
{
  return (total / parts) * p + (p < (int)(total % parts) ? p : (total % parts));
}
