// Context, memory and communicator plumbing of libhiopb200.so.
#include "hb_common.cuh"

#include <cstdlib>
#include <dlfcn.h>

thread_local char g_hb_err[512] = "";
long long g_hb_launches = 0;

extern "C" const char* hb_version(void) { return "hiopb200 0.1.0 (sm_100a)"; }
extern "C" const char* hb_last_error(void) { return g_hb_err; }
extern "C" long long hb_launch_count(void) { return g_hb_launches; }

extern "C" int hb_ctx_create(int device, hb_ctx** out)
{
  HB_REQUIRE(out != nullptr, "hb_ctx_create: out is null");
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if(e != cudaSuccess || ndev == 0) {
    snprintf(g_hb_err, sizeof(g_hb_err), "hb_ctx_create: no CUDA device available (%s); this engine has no CPU fallback",
             e == cudaSuccess ? "device count 0" : cudaGetErrorString(e));
    return HB_ERR_CUDA;
  }
  HB_REQUIRE(device >= 0 && device < ndev, "hb_ctx_create: bad device ordinal");
  HB_CUDA(cudaSetDevice(device));
  cudaDeviceProp prop;
  HB_CUDA(cudaGetDeviceProperties(&prop, device));
  if(prop.major != 10) {
    snprintf(g_hb_err, sizeof(g_hb_err), "hb_ctx_create: device %s is sm_%d%d; this library is built for sm_100a only", prop.name,
             prop.major, prop.minor);
    return HB_ERR_CUDA;
  }
  hb_ctx* c = new hb_ctx;
  c->device = device;
  c->num_sms = prop.multiProcessorCount;
  if(const char* e = getenv("HB_OZ_WORKSPACE_MB")) c->oz_ws_limit = (size_t)strtoull(e, nullptr, 10) << 20;
  HB_CUDA(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
  HB_CUDA(cudaMalloc(&c->red_dev, sizeof(double) * HB_RED_SLOTS));
  HB_CUDA(cudaMallocHost(&c->red_host, sizeof(double) * 64));
  *out = c;
  return HB_OK;
}

extern "C" int hb_ctx_destroy(hb_ctx* c)
{
  if(!c) return HB_OK;
  cudaSetDevice(c->device);
  cudaStreamSynchronize(c->stream);
  if(c->oz_state && c->oz_free) c->oz_free(c->oz_state);
  for(cudaEvent_t e : c->ev_phase) if(e) cudaEventDestroy(e);
  if(c->ws) cudaFree(c->ws);
  if(c->ev_syrk0) { cudaEventDestroy(c->ev_syrk0); cudaEventDestroy(c->ev_syrk1); }
  cudaFree(c->red_dev);
  cudaFreeHost(c->red_host);
  cudaStreamDestroy(c->stream);
  delete c;
  return HB_OK;
}

extern "C" int hb_ctx_enable_timing(hb_ctx* c, int on)
{
  HB_REQUIRE(c, "null ctx");
  if(on && !c->ev_syrk0) {
    HB_CUDA(cudaEventCreate(&c->ev_syrk0));
    HB_CUDA(cudaEventCreate(&c->ev_syrk1));
  }
  c->timing = on != 0;
  c->syrk_timed = false;
  return HB_OK;
}
extern "C" int hb_ctx_last_syrk_ms(hb_ctx* c, float* ms)
{
  HB_REQUIRE(c && ms, "hb_ctx_last_syrk_ms: null argument");
  if(!c->timing || !c->syrk_timed) return hb_fail(HB_ERR_STATE, "hb_ctx_last_syrk_ms: no timed SYRK launch recorded%s", "");
  HB_CUDA(cudaEventSynchronize(c->ev_syrk1));
  HB_CUDA(cudaEventElapsedTime(ms, c->ev_syrk0, c->ev_syrk1));
  return HB_OK;
}

// Timeline of one quasi-Newton step: with on != 0 the engine records an event after each phase of hb_lowrank_update / condense /
// solve_compressed; hb_ctx_phase_timeline(ctx, 0, ms) waits for them and returns the phase durations (ms) in the order
// update, row maxima (+ fused row dots), slicing, GEMM + fix-up [= C_aug; the first two only with the int8-slice kernel, otherwise the whole
// condensation is in the third], all-reduce, V/U/N assembly, Cholesky, H^-1 rx, J dx (+ all-reduce), SPD solve, J^T dy, H^-1 rx (second).
// A mark that was not passed contributes 0 and its time is counted in the next recorded phase. When the int8 slices are made and
// multiplied in several column chunks (hb_lowrank_last_condense_chunks > 1) the slicing entry is 0 and the GEMM entry holds the
// slicing and the GEMM of all chunks.
extern "C" int hb_ctx_phase_timeline(hb_ctx* c, int on, float* ms_host10)
{
  HB_REQUIRE(c, "null ctx");
  if(on) {
    for(int i = 0; i < HB_PH_COUNT; i++)
      if(!c->ev_phase[i]) HB_CUDA(cudaEventCreate(&c->ev_phase[i]));
    c->phase_mask = 0;
    c->phases = true;
    return HB_OK;
  }
  c->phases = false;
  if(ms_host10) {
    HB_CUDA(cudaStreamSynchronize(c->stream));
    int prev = (c->phase_mask & 1u) ? 0 : -1;
    for(int i = 1; i < HB_PH_COUNT; i++) {
      ms_host10[i - 1] = 0.f;
      if(!(c->phase_mask >> i & 1u)) continue;
      if(prev >= 0) HB_CUDA(cudaEventElapsedTime(&ms_host10[i - 1], c->ev_phase[prev], c->ev_phase[i]));
      prev = i;
    }
  }
  return HB_OK;
}

extern "C" int hb_ctx_sync(hb_ctx* c)
{
  HB_REQUIRE(c, "null ctx");
  HB_CUDA(cudaStreamSynchronize(c->stream));
  return HB_OK;
}
extern "C" void* hb_ctx_stream(hb_ctx* c) { return c ? (void*)c->stream : nullptr; }
extern "C" int hb_ctx_device(hb_ctx* c) { return c ? c->device : -1; }

int hb_ws_reserve(hb_ctx* c, size_t bytes)
{
  if(bytes <= c->ws_bytes) return HB_OK;
  if(c->ws) {
    HB_CUDA(cudaStreamSynchronize(c->stream));
    HB_CUDA(cudaFree(c->ws));
    c->ws = nullptr;
    c->ws_bytes = 0;
  }
  size_t want = bytes + (bytes >> 3);
  if(cudaMalloc(&c->ws, want) != cudaSuccess) {
    cudaGetLastError();
    snprintf(g_hb_err, sizeof(g_hb_err), "workspace allocation of %zu bytes failed", want);
    return HB_ERR_ALLOC;
  }
  c->ws_bytes = want;
  return HB_OK;
}

extern "C" int hb_malloc(hb_ctx* c, size_t bytes, void** p)
{
  HB_REQUIRE(c && p, "hb_malloc: null argument");
  HB_CUDA(cudaSetDevice(c->device));
  if(cudaMalloc(p, bytes ? bytes : 8) != cudaSuccess) {
    cudaGetLastError();
    snprintf(g_hb_err, sizeof(g_hb_err), "hb_malloc: cudaMalloc of %zu bytes failed", bytes);
    return HB_ERR_ALLOC;
  }
  return HB_OK;
}
extern "C" int hb_free(hb_ctx* c, void* p)
{
  HB_REQUIRE(c, "null ctx");
  if(p) {
    HB_CUDA(cudaStreamSynchronize(c->stream));
    HB_CUDA(cudaFree(p));
  }
  return HB_OK;
}
extern "C" int hb_malloc_host(hb_ctx* c, size_t bytes, void** p)
{
  HB_REQUIRE(c && p, "hb_malloc_host: null argument");
  if(cudaMallocHost(p, bytes ? bytes : 8) != cudaSuccess) {
    cudaGetLastError();
    snprintf(g_hb_err, sizeof(g_hb_err), "hb_malloc_host: cudaMallocHost of %zu bytes failed", bytes);
    return HB_ERR_ALLOC;
  }
  return HB_OK;
}
extern "C" int hb_free_host(hb_ctx* c, void* p)
{
  HB_REQUIRE(c, "null ctx");
  if(p) HB_CUDA(cudaFreeHost(p));
  return HB_OK;
}
extern "C" int hb_memcpy_h2d(hb_ctx* c, void* dst, const void* src, size_t bytes)
{
  HB_REQUIRE(c, "null ctx");
  if(bytes) HB_CUDA(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, c->stream));
  return HB_OK;
}
extern "C" int hb_memcpy_d2h(hb_ctx* c, void* dst, const void* src, size_t bytes)
{
  HB_REQUIRE(c, "null ctx");
  if(bytes) HB_CUDA(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, c->stream));
  return HB_OK;
}
extern "C" int hb_memcpy_d2d(hb_ctx* c, void* dst, const void* src, size_t bytes)
{
  HB_REQUIRE(c, "null ctx");
  if(bytes) HB_CUDA(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToDevice, c->stream));
  return HB_OK;
}
extern "C" int hb_memset(hb_ctx* c, void* dst, int byte, size_t bytes)
{
  HB_REQUIRE(c, "null ctx");
  if(bytes) HB_CUDA(cudaMemsetAsync(dst, byte, bytes, c->stream));
  return HB_OK;
}

// ---------------------------------------------------------------------------------------------------------
// NCCL, resolved at run time: if the host process (torch) already carries a libnccl we bind to that copy so that
// a single NCCL lives in the process; otherwise the system libnccl.so.2 is opened. No link-time dependency, so the
// single-GPU path never needs NCCL.
// ---------------------------------------------------------------------------------------------------------
namespace {
typedef struct { char internal[128]; } ncclUniqueId_t;
typedef int (*fn_get_uid)(ncclUniqueId_t*);
typedef int (*fn_comm_init)(void**, int, ncclUniqueId_t, int);
typedef int (*fn_comm_destroy)(void*);
typedef int (*fn_allreduce)(const void*, void*, size_t, int, int, void*, cudaStream_t);
typedef const char* (*fn_errstr)(int);
struct NcclApi
{
  void* h = nullptr;
  fn_get_uid get_uid = nullptr;
  fn_comm_init comm_init = nullptr;
  fn_comm_destroy comm_destroy = nullptr;
  fn_allreduce allreduce = nullptr;
  fn_errstr errstr = nullptr;
  bool tried = false;
} g_nccl;

int nccl_load()
{
  if(g_nccl.h) return HB_OK;
  if(g_nccl.tried) return hb_fail(HB_ERR_COMM, "NCCL library could not be loaded%s", "");
  g_nccl.tried = true;
  void* h = dlopen(nullptr, RTLD_NOW); // symbols already in the process (torch's bundled NCCL)?
  if(h && !dlsym(h, "ncclAllReduce")) h = nullptr;
  const char* names[] = {"libnccl.so.2", "libnccl.so", "/usr/lib/x86_64-linux-gnu/libnccl.so.2"};
  for(int i = 0; !h && i < 3; i++) {
    h = dlopen(names[i], RTLD_NOW | RTLD_NOLOAD);
    if(!h) h = dlopen(names[i], RTLD_NOW | RTLD_GLOBAL);
  }
  if(!h) return hb_fail(HB_ERR_COMM, "NCCL library could not be loaded: %s", dlerror());
  g_nccl.get_uid = (fn_get_uid)dlsym(h, "ncclGetUniqueId");
  g_nccl.comm_init = (fn_comm_init)dlsym(h, "ncclCommInitRank");
  g_nccl.comm_destroy = (fn_comm_destroy)dlsym(h, "ncclCommDestroy");
  g_nccl.allreduce = (fn_allreduce)dlsym(h, "ncclAllReduce");
  g_nccl.errstr = (fn_errstr)dlsym(h, "ncclGetErrorString");
  if(!g_nccl.get_uid || !g_nccl.comm_init || !g_nccl.allreduce) return hb_fail(HB_ERR_COMM, "NCCL symbols missing%s", "");
  g_nccl.h = h;
  return HB_OK;
}
} // namespace

extern "C" int hb_comm_unique_id(void* id128)
{
  HB_REQUIRE(id128, "null id buffer");
  HB_CHECK(nccl_load());
  ncclUniqueId_t id;
  int rc = g_nccl.get_uid(&id);
  if(rc != 0) return hb_fail(HB_ERR_COMM, "ncclGetUniqueId failed: %s", g_nccl.errstr ? g_nccl.errstr(rc) : "?");
  memcpy(id128, &id, 128);
  return HB_OK;
}

extern "C" int hb_comm_init(hb_ctx* c, int nranks, int rank, const void* id128)
{
  HB_REQUIRE(c && nranks >= 1 && rank >= 0 && rank < nranks, "hb_comm_init: bad arguments");
  c->nranks = nranks;
  c->rank = rank;
  if(nranks == 1) return HB_OK;
  HB_REQUIRE(id128, "hb_comm_init: null unique id");
  HB_CHECK(nccl_load());
  HB_CUDA(cudaSetDevice(c->device));
  ncclUniqueId_t id;
  memcpy(&id, id128, 128);
  int rc = g_nccl.comm_init(&c->nccl_comm, nranks, id, rank);
  if(rc != 0) return hb_fail(HB_ERR_COMM, "ncclCommInitRank failed: %s", g_nccl.errstr ? g_nccl.errstr(rc) : "?");
  return HB_OK;
}
extern "C" int hb_comm_size(hb_ctx* c) { return c ? c->nranks : 0; }
extern "C" int hb_comm_rank(hb_ctx* c) { return c ? c->rank : -1; }

extern "C" int hb_allreduce_sum(hb_ctx* c, double* buf, long long count)
{
  HB_REQUIRE(c, "null ctx");
  if(c->nranks == 1 || count == 0) return HB_OK;
  if(!c->nccl_comm) return hb_fail(HB_ERR_COMM, "hb_allreduce_sum: communicator not initialised%s", "");
  // ncclFloat64 = 8, ncclSum = 0
  int rc = g_nccl.allreduce(buf, buf, (size_t)count, 8, 0, c->nccl_comm, c->stream);
  if(rc != 0) return hb_fail(HB_ERR_COMM, "ncclAllReduce failed: %s", g_nccl.errstr ? g_nccl.errstr(rc) : "?");
  return HB_OK;
}

int hb_allreduce_op(hb_ctx* c, double* buf, long long count, int op /*0 sum,2 max,3 min*/)
{
  if(c->nranks == 1 || count == 0) return HB_OK;
  if(!c->nccl_comm) return hb_fail(HB_ERR_COMM, "communicator not initialised%s", "");
  int rc = g_nccl.allreduce(buf, buf, (size_t)count, 8, op, c->nccl_comm, c->stream);
  if(rc != 0) return hb_fail(HB_ERR_COMM, "ncclAllReduce failed: %s", g_nccl.errstr ? g_nccl.errstr(rc) : "?");
  return HB_OK;
}
