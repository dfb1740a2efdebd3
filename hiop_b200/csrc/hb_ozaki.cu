// C = A diag(d) A^T on the 5th-generation tensor cores (tcgen05.mma.kind::i8, accumulators in TMEM, operands by TMA):
// FP64 emulation by integer slicing (Ozaki scheme).
//
//   B = A diag(sqrt(d));   row i:  b_ik = 2^{e_i} * sum_p q_p(i,k) 2^{-(6+7p)} + O(2^{e_i - 6 - 7S}),  q_p int8, |q_p| <= 64
//   C_ij = 2^{e_i+e_j} * sum_{t=0}^{S-1} 2^{-(12+7t)} T_t(i,j),     T_t = sum_{p+q=t} Q_p Q_q^T   (exact int32)
//
// tcgen05.mma has no f64 kind; this is the only way the K ~ 1e6, M ~ 1e3 condensation can use the tcgen05 pipe. Every
// integer product and accumulation is exact (K is cut into chunks so that (t+1)*Kc*2^12 < 2^31); the only error is the
// truncation of b after 6+7(S-1) bits relative to each row's largest entry (S=7: 2^-48, S=8: 2^-55) plus the final FP64
// recombination. The exact FP64 DMMA kernel (hb_syrk.cu) stays as the reference path and as the fallback.
//
// Pipeline of k_oz_gemm (256 threads, one CTA per SM, 128x64 output tiles, split-K):
//   warp 0 (1 thread)  TMA producer: per 128-byte K block one box {128 B x 64 rows x S slices} (B) and S boxes
//                      {128 B x 128 rows} (A) from the 3-D tensor map (k, row, slice), SWIZZLE_128B, mbarrier completion
//   warp 1 (1 thread)  MMA issuer: tcgen05.mma.cta_group::1.kind::i8 (M=128, N=64..256 = stacked slices, K=32),
//                      one TMEM accumulator (64 columns) per t = p+q; tcgen05.commit frees the stage / signals the epilogue
//   warps 4-7          epilogue: at every K-chunk boundary tcgen05.ld the S accumulators, recombine them in FP64 and
//                      accumulate into the CTA's FP64 partial tile (workspace, L2 resident)
// A last kernel sums the split-K partials in fixed order, applies 2^{e_i+e_j} and mirrors the tile (deterministic).
// When the slices of all K columns do not fit the slice budget, K is sliced and multiplied in column chunks that reuse one buffer, the
// GEMM of every chunk after the first adding to the partial tiles (see hb_syrk_rows_ozaki).
#include "hb_common.cuh"
#include <cuda.h>
#include <cstdlib>

namespace {

constexpr int TM = 128, TN = 64;
constexpr int KS = 128;           // bytes of K per block (one SWIZZLE_128B row = four MMA K steps)
constexpr int A_TILE = TM * KS;   // 16 KB per slice
constexpr int B_TILE = TN * KS;   // 8 KB per slice
constexpr int OZ_THREADS = 256;
// device memory the AUTO slice budget leaves free: the split-K partial tiles (<= 1 GB by the split rule) and the small buffers
constexpr size_t OZ_FREE_MARGIN = (size_t)1 << 30;

__device__ __forceinline__ uint32_t s2u(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(unsigned long long* b, unsigned c) { asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;\n" ::"r"(s2u(b)), "r"(c)); }
__device__ __forceinline__ void mbar_expect_tx(unsigned long long* b, unsigned bytes)
{
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n" ::"r"(s2u(b)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(unsigned long long* b) { asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];\n" ::"r"(s2u(b)) : "memory"); }
__device__ __forceinline__ bool mbar_try_wait(unsigned long long* b, unsigned parity)
{
  unsigned ok;
  asm volatile(
      "{\n.reg .pred p;\nmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\nselp.u32 %0, 1, 0, p;\n}\n"
      : "=r"(ok)
      : "r"(s2u(b)), "r"(parity), "r"(0x989680u)
      : "memory");
  return ok != 0;
}
__device__ __forceinline__ void mbar_wait(unsigned long long* b, unsigned parity)
{
  while(!mbar_try_wait(b, parity)) {}
}
// wait used by the epilogue warps (they idle for a whole K chunk): back off between polls so that the four warps do not
// steal issue slots from the single-thread TMA / MMA warps sharing their SM sub-partitions
__device__ __forceinline__ void mbar_wait_sleep(unsigned long long* b, unsigned parity)
{
  while(!mbar_try_wait(b, parity)) __nanosleep(2000);
}
__device__ __forceinline__ void tma_load_3d(void* dst, const CUtensorMap* map, int c0, int c1, int c2, unsigned long long* bar)
{
  asm volatile("cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];\n" ::"r"(s2u(dst)),
               "l"(map), "r"(c0), "r"(c1), "r"(c2), "r"(s2u(bar))
               : "memory");
}
__device__ __forceinline__ void umma_commit(unsigned long long* bar)
{
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n" ::"r"(s2u(bar)) : "memory");
}
// K-major SWIZZLE_128B operand descriptor (rows 128 B apart, 8-row groups 1024 B apart), sm_100 descriptor version 1.
// K steps inside the 128-byte swizzle row advance the start address by 32 bytes. The SWIZZLE_64B / SWIZZLE_32B variants of the
// same formula are validated by tools/tc_i8_tma_test{,32}.cu.
__device__ __forceinline__ uint64_t make_desc_sw(uint32_t smem_addr)
{
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr >> 4) & 0x3FFF);
  d |= (uint64_t)1 << 16;
  d |= (uint64_t)((1024 >> 4) & 0x3FFF) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)2 << 61; // SWIZZLE_128B
  return d;
}
__device__ __forceinline__ void umma_i8(uint32_t tmem_c, uint64_t da, uint64_t db, uint32_t idesc, uint32_t accumulate)
{
  asm volatile(
      "{\n.reg .pred pp;\nsetp.ne.b32 pp, %4, 0;\n"
      "tcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, {%5, %6, %7, %8}, pp;\n}\n" ::"r"(tmem_c),
      "l"(da), "l"(db), "r"(idesc), "r"(accumulate), "r"(0), "r"(0), "r"(0), "r"(0)
      : "memory");
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&v)[32])
{
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];\n"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]),
        "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]),
        "=r"(v[23]), "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
      : "r"(taddr));
}

// ---------------------------------------------------------------------------------------------------------------------
// slicing
// ---------------------------------------------------------------------------------------------------------------------
// row maxima of |a_ik| * sd_k  (sd = sqrt(d) or 1): integer atomicMax on the bit pattern of a non-negative double
__global__ void __launch_bounds__(256)
k_oz_rowmax(const double* const* __restrict__ rowptr, int M, long long K, const double* __restrict__ sd, unsigned long long* __restrict__ mx)
{
  const int row = blockIdx.y;
  const double* a = rowptr[row];
  double m = 0.0;
  const long long stride = (long long)gridDim.x * 256;
  for(long long k = (long long)blockIdx.x * 256 + threadIdx.x; k < K; k += stride) m = fmax(m, fabs(a[k]) * (sd ? sd[k] : 1.0));
  m = hb_warp_max(m);
  if((threadIdx.x & 31) == 0 && m > 0.0) atomicMax(&mx[row], (unsigned long long)__double_as_longlong(m));
}
// Row maxima AND the row dot products with t = d .* x in the same pass over the rows (a5/a13: J (H+Dx)^-1-weighted rhs, step 2 of
// solveCompressed, costs no second sweep over J when the condensation is pending anyway). A CTA owns RD_COLS columns: each lane keeps
// the sqrt(d) and d.*x values of its columns in registers and the 16 warps stream the rows past them, RD_ROWS rows in flight per warp.
// partial[chunk][row] is combined in a fixed order by k_oz_dot_final; the maxima go through the same order-independent atomicMax.
constexpr int RD_THREADS = 512, RD_COLS = 256, RD_ROWS = 4;
template <bool VEC>
__global__ void __launch_bounds__(RD_THREADS)
k_oz_rowmax_dot(const double* const* __restrict__ rowptr, int M, long long K, const double* __restrict__ d, const double* __restrict__ x,
                unsigned long long* __restrict__ mx, double* __restrict__ partial)
{
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const long long k0 = (long long)blockIdx.x * RD_COLS;
  const int len = (int)min((long long)RD_COLS, K - k0);
  double sd[8], w[8];
  // slot p of a lane: VEC -> the pair of columns 2*(lane + 32*(p/2)) + (p&1); scalar -> column lane + 32*p (relative to k0)
#define RD_OFF(p) (VEC ? 2 * (lane + 32 * ((p) >> 1)) + ((p) & 1) : lane + 32 * (p))
#pragma unroll
  for(int p = 0; p < 8; p++) {
    const int off = RD_OFF(p);
    if(off < len) {
      const double dv = d ? d[k0 + off] : 1.0;
      sd[p] = d ? sqrt(dv) : 1.0;
      w[p] = dv * x[k0 + off];
    } else {
      sd[p] = 0.0;
      w[p] = 0.0;
    }
  }
  const int wstride = (RD_THREADS / 32) * gridDim.y;
  for(int i0 = warp + (RD_THREADS / 32) * blockIdx.y; i0 < M; i0 += wstride * RD_ROWS) {
    double v[RD_ROWS][8];
#pragma unroll
    for(int r = 0; r < RD_ROWS; r++) {
      const int i = i0 + r * wstride;
      const double* row = i < M ? rowptr[i] + k0 : nullptr;
#pragma unroll
      for(int p = 0; p < (VEC ? 4 : 8); p++) {
        if(VEC) {
          double2 t = make_double2(0.0, 0.0);
          if(row && RD_OFF(2 * p) < len) t = *reinterpret_cast<const double2*>(row + RD_OFF(2 * p));
          v[r][2 * p] = t.x;
          v[r][2 * p + 1] = t.y;
        } else {
          v[r][p] = (row && RD_OFF(p) < len) ? row[RD_OFF(p)] : 0.0;
        }
      }
    }
#pragma unroll
    for(int r = 0; r < RD_ROWS; r++) {
      const int i = i0 + r * wstride;
      double mm = 0.0, acc = 0.0;
#pragma unroll
      for(int p = 0; p < 8; p++) {
        mm = fmax(mm, fabs(v[r][p]) * sd[p]);
        acc += v[r][p] * w[p];
      }
      mm = hb_warp_max(mm);
      acc = hb_warp_sum(acc);
      if(lane == 0 && i < M) {
        if(mm > 0.0) atomicMax(&mx[i], (unsigned long long)__double_as_longlong(mm));
        partial[(size_t)blockIdx.x * M + i] = acc;
      }
    }
  }
#undef RD_OFF
}
// out[i] = sum_chunks partial[c][i]: 32 rows x 8 chunk classes per CTA, fixed-order combine
__global__ void __launch_bounds__(256)
k_oz_dot_final(int M, int nchunks, const double* __restrict__ partial, double* __restrict__ out)
{
  __shared__ double sm[8][33];
  const int ri = threadIdx.x & 31, part = threadIdx.x >> 5;
  const int i = blockIdx.x * 32 + ri;
  double s = 0.0;
  if(i < M)
    for(int c = part; c < nchunks; c += 8) s += partial[(size_t)c * M + i];
  sm[part][ri] = s;
  __syncthreads();
  if(part == 0 && i < M) {
    double t = 0.0;
#pragma unroll
    for(int p = 0; p < 8; p++) t += sm[p][ri];
    out[i] = t;
  }
}
__global__ void k_oz_exponents(int M, const unsigned long long* __restrict__ mx, int* __restrict__ e)
{
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if(i >= M) return;
  const double m = __longlong_as_double((long long)mx[i]);
  int ex = 0;
  if(m > 0.0) frexp(m, &ex); // m = f * 2^ex, f in [0.5, 1)  ->  |b| / 2^ex < 1
  e[i] = ex;
}
__global__ void k_sqrt(long long n, const double* __restrict__ d, double* __restrict__ sd)
{
  const long long stride = (long long)gridDim.x * blockDim.x;
  for(long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) sd[i] = sqrt(d[i]);
}

// Q[p][row][k - k0] (int8, row pitch ldq bytes, slice pitch Mpad*ldq) for the column window [k0, k0 + Kw), zero-padded up to
// Kwpad (a multiple of KS). One thread = 8 consecutive k of one row: a warp reads 2 KB of the FP64 row with 16-byte loads and writes
// 256 contiguous bytes per slice. The digits depend only on a_ik, sd_k and the row exponent e_i, so a window of a column-chunked
// condensation holds exactly the bytes the one-window (unchunked) call writes for those columns.
//
// Digits without the conversion pipe: with b = a*sd / 2^e (|b| < 1), hi = rint(b * 2^27) carries the first four slices
// (6+7+7+7 bits) and lo = rint((b*2^27 - hi) * 2^(7(S-4))) the remaining S-4. Both roundings use the 1.5*2^52 magic-number
// add (two DADDs at full FP64 rate; the integer is the low word of the sum -- no F2I/FRND, which issue at 1/4 rate and made
// the first version of this kernel conversion-bound at 3.9 ms for 8 GB). Each 32-bit integer is then cut into balanced
// base-128 digits d in [-64, 63] from the least significant end; the leading digit of either word is bounded by 64.
// sum_p q_p 2^-(6+7p) = b rounded to the last slice's grid, exactly.
template <int ND>
__device__ __forceinline__ void oz_digits(int v, int (&d)[ND])
{
#pragma unroll
  for(int j = ND - 1; j > 0; j--) {
    d[j] = ((v + 64) & 127) - 64;
    v = (v - d[j]) >> 7;
  }
  d[0] = v;
}
template <int S>
__global__ void __launch_bounds__(256)
k_oz_slice(const double* const* __restrict__ rowptr, int M, int Mpad, long long kwin, long long K, long long Kpad, long long ldq,
           const double* __restrict__ sd, const int* __restrict__ e, int8_t* __restrict__ Q, int vec_ok)
{
  static_assert(S >= 5 && S <= 8, "slices");
  constexpr int NLO = S - 4;
  const int row = blockIdx.y;
  const long long k0 = ((long long)blockIdx.x * 256 + threadIdx.x) * 8;
  if(k0 >= Kpad) return;
  double x[8];
#pragma unroll
  for(int j = 0; j < 8; j++) x[j] = 0.0;
  if(sd) sd += kwin; // kwin is a multiple of KS: 16-byte alignment of the rows and of sd is kept
  if(row < M) {
    const double* a = rowptr[row] + kwin;
    const double sc = ldexp(1.0, 27 - e[row]);
    if(vec_ok && k0 + 7 < K) {
#pragma unroll
      for(int j = 0; j < 8; j += 2) {
        const double2 av = *reinterpret_cast<const double2*>(a + k0 + j);
        double2 sv = make_double2(1.0, 1.0);
        if(sd) sv = *reinterpret_cast<const double2*>(sd + k0 + j);
        x[j] = __dmul_rn(__dmul_rn(av.x, sv.x), sc);
        x[j + 1] = __dmul_rn(__dmul_rn(av.y, sv.y), sc);
      }
    } else {
#pragma unroll
      for(int j = 0; j < 8; j++)
        if(k0 + j < K) x[j] = __dmul_rn(__dmul_rn(a[k0 + j], sd ? sd[k0 + j] : 1.0), sc);
    }
  }
  const double MAGIC = 6755399441055744.0; // 1.5 * 2^52
  unsigned w[S][2];
#pragma unroll
  for(int h = 0; h < 2; h++) {
    int dh[4][4], dl[4][NLO];
#pragma unroll
    for(int j = 0; j < 4; j++) {
      const double xs = x[4 * h + j];
      const double t = __dadd_rn(xs, MAGIC);
      const int hi = __double2loint(t);
      const double rem = __dsub_rn(xs, __dsub_rn(t, MAGIC));                       // exact, |rem| <= 0.5
      const int lo = __double2loint(__fma_rn(rem, (double)(1 << (7 * NLO)), MAGIC));
      oz_digits<4>(hi, dh[j]);
      oz_digits<NLO>(lo, dl[j]);
    }
#pragma unroll
    for(int p = 0; p < 4; p++)
      w[p][h] = __byte_perm(__byte_perm(dh[0][p], dh[1][p], 0x0040), __byte_perm(dh[2][p], dh[3][p], 0x0040), 0x5410);
#pragma unroll
    for(int p = 0; p < NLO; p++)
      w[4 + p][h] = __byte_perm(__byte_perm(dl[0][p], dl[1][p], 0x0040), __byte_perm(dl[2][p], dl[3][p], 0x0040), 0x5410);
  }
#pragma unroll
  for(int p = 0; p < S; p++) *reinterpret_cast<uint2*>(Q + ((size_t)p * Mpad + row) * ldq + k0) = make_uint2(w[p][0], w[p][1]);
}

// ---------------------------------------------------------------------------------------------------------------------
// the tcgen05 GEMM
// ---------------------------------------------------------------------------------------------------------------------
struct OzItem
{
  int bi, bj;       // 128-row block, 64-column block
  int k_begin;      // first K stage (units of KS bytes)
  int k_count;
  int slot;         // FP64 partial tile (TM x TN doubles)
};

template <int S>
struct OzCfg
{
  static constexpr int B_BLOCK = S * B_TILE;                       // all S slices of the 64 B-rows for one K block
  static constexpr int RING = (226 * 1024 - 2 * B_BLOCK) / A_TILE; // A tiles in flight (7 / 7 / 6 for S = 6 / 7 / 8)
  static constexpr int SMEM = 2 * B_BLOCK + RING * A_TILE + 512;
};

// K is swept in blocks of KS = 128 bytes (one SWIZZLE_128B row: TMA delivers twice the bytes per row request of the first,
// 64-byte version, which was bound by the TMA row rate -- the stage time did not change when the row length was halved).
// Per K block the B operand (S slices x 64 rows, 8S KB) is double-buffered and stays resident while the S A tiles (16 KB
// each) stream through a ring; slice p is multiplied against the stacked slices 0..S-1-p of B (N up to 256 per MMA).
template <int S>
__global__ void __launch_bounds__(OZ_THREADS, 1)
k_oz_gemm(const __grid_constant__ CUtensorMap mapA, const __grid_constant__ CUtensorMap mapB, const OzItem* __restrict__ items, int n_items,
          int chunk_blocks, int accumulate, double* __restrict__ partial)
{
  using Cfg = OzCfg<S>;
  constexpr int RING = Cfg::RING;
  extern __shared__ __align__(1024) uint8_t smem[];
  uint8_t* bbuf = smem;                       // 2 x B_BLOCK
  uint8_t* aring = smem + 2 * Cfg::B_BLOCK;   // RING x A_TILE
  unsigned long long* bfull = reinterpret_cast<unsigned long long*>(aring + RING * A_TILE);
  unsigned long long* bempty = bfull + 2;
  unsigned long long* afull = bempty + 2;
  unsigned long long* aempty = afull + RING;
  unsigned long long* accfull = aempty + RING;
  unsigned long long* accempty = accfull + 1;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(accempty + 1);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  if(tid == 0) {
    for(int s = 0; s < 2; s++) { mbar_init(&bfull[s], 1); mbar_init(&bempty[s], 1); }
    for(int s = 0; s < RING; s++) { mbar_init(&afull[s], 1); mbar_init(&aempty[s], 1); }
    mbar_init(accfull, 1);
    mbar_init(accempty, 4);
    asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
  }
  if(warp == 2) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;\n" ::"r"(s2u(tmem_slot)), "r"(512));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;\n" ::);
  }
  asm volatile("tcgen05.fence::before_thread_sync;\n" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory");
  const uint32_t tmem = *tmem_slot;

  if(warp == 0 && lane == 0) {
    // ================= TMA producer =================
    int bs = 0, as = 0;
    unsigned bph = 0, aph = 0;
    for(int w = blockIdx.x; w < n_items; w += gridDim.x) {
      const OzItem itm = items[w];
      for(int it = 0; it < itm.k_count; it++) {
        const int kc = (itm.k_begin + it) * KS;
        mbar_wait(&bempty[bs], bph ^ 1);
        mbar_expect_tx(&bfull[bs], Cfg::B_BLOCK);
        tma_load_3d(bbuf + bs * Cfg::B_BLOCK, &mapB, kc, itm.bj * TN, 0, &bfull[bs]); // box {128 B, 64 rows, S slices}
        if(++bs == 2) { bs = 0; bph ^= 1; }
#pragma unroll 1
        for(int p = 0; p < S; p++) {
          mbar_wait(&aempty[as], aph ^ 1);
          mbar_expect_tx(&afull[as], A_TILE);
          tma_load_3d(aring + as * A_TILE, &mapA, kc, itm.bi * TM, p, &afull[as]);    // box {128 B, 128 rows, 1 slice}
          if(++as == RING) { as = 0; aph ^= 1; }
        }
      }
    }
  } else if(warp == 1 && lane == 0) {
    // ================= MMA issuer =================
    // idesc: c=S32 [4,6), a=INT8 [7,10), b=INT8 [10,13), K-major both, n_dim=N>>3 [17,23), m_dim=M>>4 [24,29)
    const uint32_t idesc0 = (2u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(TM >> 4) << 24);
    int bs = 0, as = 0;
    unsigned bph = 0, aph = 0, accphase = 0;
    for(int w = blockIdx.x; w < n_items; w += gridDim.x) {
      const OzItem itm = items[w];
      int in_chunk = 0;
      for(int it = 0; it < itm.k_count; it++) {
        if(in_chunk == 0) {
          // accumulators are about to be overwritten: the epilogue must have drained the previous chunk
          mbar_wait(accempty, accphase ^ 1);
          asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory");
        }
        mbar_wait(&bfull[bs], bph);
        const uint32_t sb = s2u(bbuf + bs * Cfg::B_BLOCK);
#pragma unroll
        for(int p = 0; p < S; p++) {
          mbar_wait(&afull[as], aph);
          asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory");
          const uint32_t sa = s2u(aring + as * A_TILE);
          // Slice stacking: B tiles of consecutive slices are contiguous in shared memory and their accumulators (t = p+q)
          // are contiguous in TMEM, so one instruction with N = 64*nq computes A_p * [B_q0 .. B_q0+nq-1]^T.
#pragma unroll
          for(int ks = 0; ks < KS / 32; ks++) {
#pragma unroll
            for(int q0 = 0; q0 < S - p; q0 += 4) {
              const int nq = (S - p - q0) < 4 ? (S - p - q0) : 4;
              const uint32_t idesc = idesc0 | ((uint32_t)((TN * nq) >> 3) << 17);
              const uint32_t acc = (in_chunk > 0 || ks > 0 || p > 0) ? 1u : 0u;
              umma_i8(tmem + (uint32_t)((p + q0) * TN), make_desc_sw(sa + ks * 32), make_desc_sw(sb + q0 * B_TILE + ks * 32), idesc, acc);
            }
          }
          umma_commit(&aempty[as]);
          if(++as == RING) { as = 0; aph ^= 1; }
        }
        umma_commit(&bempty[bs]);
        if(++bs == 2) { bs = 0; bph ^= 1; }
        in_chunk++;
        if(in_chunk == chunk_blocks || it == itm.k_count - 1) {
          umma_commit(accfull);
          accphase ^= 1;
          in_chunk = 0;
        }
      }
    }
  } else if(warp >= 4) {
    // ================= epilogue (TMEM lanes 32*(warp%4) .. +31 = tile rows) =================
    const int wq = warp & 3;
    const int row = wq * 32 + lane;
    unsigned accphase = 0;
    for(int w = blockIdx.x; w < n_items; w += gridDim.x) {
      const OzItem itm = items[w];
      double* slot = partial + (size_t)itm.slot * (TM * TN) + (size_t)row * TN;
      const int nchunks = (itm.k_count + chunk_blocks - 1) / chunk_blocks;
      for(int c = 0; c < nchunks; c++) {
        mbar_wait_sleep(accfull, accphase);
        accphase ^= 1;
        asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory");
        double acc[TN];
#pragma unroll
        for(int j = 0; j < TN; j++) acc[j] = 0.0;
#pragma unroll
        for(int t = S - 1; t >= 0; t--) { // smallest weights first
          const double wt = ldexp(1.0, -(12 + 7 * t));
#pragma unroll
          for(int c0 = 0; c0 < TN; c0 += 32) {
            uint32_t v[32];
            tmem_ld32(tmem + ((uint32_t)(wq * 32) << 16) + (uint32_t)(t * TN + c0), v);
            asm volatile("tcgen05.wait::ld.sync.aligned;\n" ::: "memory");
#pragma unroll
            for(int j = 0; j < 32; j++) acc[c0 + j] += (double)(int)v[j] * wt;
          }
        }
        asm volatile("tcgen05.fence::before_thread_sync;\n" ::: "memory");
        __syncwarp();
        if(lane == 0) mbar_arrive(accempty);
        if(c == 0 && !accumulate) {
#pragma unroll
          for(int j = 0; j < TN; j += 2) *reinterpret_cast<double2*>(slot + j) = make_double2(acc[j], acc[j + 1]);
        } else {
#pragma unroll
          for(int j = 0; j < TN; j += 2) {
            double2 o = *reinterpret_cast<double2*>(slot + j);
            o.x += acc[j];
            o.y += acc[j + 1];
            *reinterpret_cast<double2*>(slot + j) = o;
          }
        }
      }
    }
  }
  asm volatile("tcgen05.fence::before_thread_sync;\n" ::: "memory");
  __syncthreads();
  if(warp == 2) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;\n" ::"r"(tmem), "r"(512));
}

// C(i,j) = 2^{e_i+e_j} * sum over splits of the partial tiles; upper part computed, mirrored.
__global__ void __launch_bounds__(256)
k_oz_fixup(int M, int n_tiles, const int2* __restrict__ tile_ij, int splits, const double* __restrict__ partial, const int* __restrict__ e,
           double* __restrict__ C, int ldc)
{
  const int t = blockIdx.x;
  const int2 ij = tile_ij[t];
  for(int el = threadIdx.x; el < TM * TN; el += 256) {
    const int r = el / TN, c = el % TN;
    const int gi = ij.x * TM + r, gj = ij.y * TN + c;
    if(gi >= M || gj >= M || gj < gi) continue;
    double v = 0.0;
    for(int s = 0; s < splits; s++) v += partial[((size_t)(t * splits + s)) * (TM * TN) + el];
    v = ldexp(v, e[gi] + e[gj]);
    C[(size_t)gi * ldc + gj] = v;
    C[(size_t)gj * ldc + gi] = v;
  }
}

typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*, const cuuint32_t*,
                                    const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
PFN_encodeTiled g_encode = nullptr;

struct OzState
{
  int M = -1, S = 0, splits = 0, n_tiles = 0, n_items = 0;
  long long K = -1, Kpad = 0;
  long long Kc = 0;  // columns per slicing chunk (Kpad: unchunked); row pitch of Q
  int Mpad = 0;
  int8_t* Q = nullptr; // S x Mpad x Kc int8 slices of the current column chunk
  size_t Qbytes = 0;
  double* sd = nullptr;
  long long sd_n = 0;
  unsigned long long* mx = nullptr;
  int* e = nullptr;
  int mcap = 0;
  double* dot_partial = nullptr; // [chunks][M] partial row dots of the fused row-maximum pass
  size_t dot_cap = 0;
  OzItem* d_items = nullptr; // 2 x n_items: the work list of a full chunk, then that of the (possibly shorter) last chunk
  int2* d_tiles = nullptr;
  CUtensorMap mapA, mapB;
};
// one state per CONTEXT (it used to be per device: two contexts on one GPU would have shared the slice buffer across their streams)
void oz_state_free(void* p)
{
  OzState* st = static_cast<OzState*>(p);
  if(!st) return;
  cudaFree(st->Q); cudaFree(st->sd); cudaFree(st->mx); cudaFree(st->e); cudaFree(st->d_items); cudaFree(st->d_tiles); cudaFree(st->dot_partial);
  delete st;
}
OzState& oz_state(hb_ctx* c)
{
  if(!c->oz_state) {
    c->oz_state = new OzState;
    c->oz_free = oz_state_free;
  }
  return *static_cast<OzState*>(c->oz_state);
}

template <int S>
int launch_gemm(hb_ctx* c, OzState& st, const OzItem* items, int chunk_blocks, int accumulate, double* partial)
{
  const size_t smem = OzCfg<S>::SMEM;
  static bool attr[16] = {false}; // function attributes are per device
  if(c->device >= 16 || !attr[c->device]) {
    HB_CUDA(cudaFuncSetAttribute(k_oz_gemm<S>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    if(c->device < 16) attr[c->device] = true;
  }
  const int G = st.n_items < c->num_sms ? st.n_items : c->num_sms;
  k_oz_gemm<S><<<G, OZ_THREADS, smem, c->stream>>>(st.mapA, st.mapB, items, st.n_items, chunk_blocks, accumulate, partial);
  HB_LAUNCHED();
  return HB_OK;
}

} // namespace

// Explicit bound on the int8 slice buffer (0 = AUTO). A buffer held above the new bound is released now.
extern "C" int hb_ctx_set_oz_workspace_limit(hb_ctx* c, size_t bytes)
{
  HB_REQUIRE(c, "null ctx");
  c->oz_ws_limit = bytes;
  if(bytes && c->oz_state) {
    OzState& st = oz_state(c);
    if(st.Qbytes > bytes) {
      HB_CUDA(cudaStreamSynchronize(c->stream));
      HB_CUDA(cudaFree(st.Q));
      st.Q = nullptr;
      st.Qbytes = 0;
      st.M = -1; // the tensor maps pointed into the released buffer
    }
  }
  return HB_OK;
}

// Same contract as hb_syrk_rows (C = A diag(d) A^T, both triangles), computed with S int8 slices on tcgen05.
// dot_x/dot_out (optional, device): dot_out[i] = sum_k row_i[k] d[k] dot_x[k] over the local columns, produced by the row-maximum pass
// chunks_out (optional, host): how many column chunks were sliced (1 = the whole of K at once)
//
// Column chunks. The slice buffer of all K columns (S * Mpad * Kpad bytes, as large as A in FP64 at S = 8) is allocated when it fits
// the budget: hb_ctx_set_oz_workspace_limit / HB_OZ_WORKSPACE_MB, or, without one, the free device memory minus OZ_FREE_MARGIN.
// Otherwise K is cut into chunks of a whole number of int32-safe recombination chunks (chunk_stages * KS columns) and each chunk is
// sliced into a buffer of S * Mpad * Kc bytes and multiplied in turn; the first GEMM writes the FP64 partial tiles, the later ones add
// to them. The row exponents come from one sweep over all columns first, so every digit is the one the unchunked call makes; only the
// grouping of the FP64 partial sums changes. HB_ERR_ALLOC when not even one recombination chunk (or all of K, if smaller) fits.
int hb_syrk_rows_ozaki(hb_ctx* c, int M, long long K, const double* const* rowptr_dev, bool rows_aligned16, const double* d, double* C, int ldc, int S,
                       const double* dot_x, double* dot_out, int* chunks_out)
{
  HB_REQUIRE(c && M >= 0 && K >= 0 && ldc >= M && (S == 6 || S == 7 || S == 8), "hb_syrk_rows_ozaki: bad arguments");
  if(chunks_out) *chunks_out = 1;
  if(M == 0) return HB_OK;
  if(K == 0) {
    HB_CUDA(cudaMemset2DAsync(C, sizeof(double) * ldc, 0, sizeof(double) * M, M, c->stream));
    return HB_OK;
  }
  if(!g_encode) {
    cudaDriverEntryPointQueryResult qres;
    HB_CUDA(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", (void**)&g_encode, cudaEnableDefault, &qres));
    if(!g_encode) return hb_fail(HB_ERR_CUDA, "cuTensorMapEncodeTiled is not available in this driver%s", "");
  }
  OzState& st = oz_state(c);
  const int Mpad = ((M + TM - 1) / TM) * TM;
  const long long Kpad = ((K + KS - 1) / KS) * KS;
  // (t+1) * Kc * 2^12 < 2^31 with t+1 <= S  ->  Kc <= 2^19 / S columns
  int chunk_stages = (int)((524288 / S) / KS);
  // strict: S products of |q q'| <= 2^12 per column must stay BELOW 2^31 (S = 8 gives exactly 2^31 with 512 stages of 128 columns when
  // every digit is -64, see tests/test_cpu_oz_model.py)
  while((long long)S * chunk_stages * KS * 4096 >= (1LL << 31)) chunk_stages--;
  // column chunk width: all of K when its slices are already held or fit the budget, else the most recombination chunks that fit
  long long Kc = Kpad;
  if(st.Qbytes < (size_t)S * Mpad * Kpad) {
    size_t budget = c->oz_ws_limit;
    if(!budget) {
      size_t free_b = 0, total_b = 0;
      HB_CUDA(cudaMemGetInfo(&free_b, &total_b));
      budget = st.Qbytes + (free_b > OZ_FREE_MARGIN ? free_b - OZ_FREE_MARGIN : 0);
    }
    if((size_t)S * Mpad * Kpad > budget) {
      const long long rcols = (long long)chunk_stages * KS;
      const long long nr = (long long)(budget / ((size_t)S * Mpad * rcols));
      if(nr == 0 || Kpad <= rcols) {
        const long long minc = Kpad < rcols ? Kpad : rcols;
        snprintf(g_hb_err, sizeof(g_hb_err), "hb_syrk_rows_ozaki: the int8 slices of one %lld-column chunk (%llu bytes) exceed the %llu-byte budget",
                 minc, (unsigned long long)S * Mpad * minc, (unsigned long long)budget);
        return HB_ERR_ALLOC;
      }
      Kc = nr * rcols;
    }
  }
  const size_t qbytes = (size_t)S * Mpad * Kc;
  if(st.Qbytes < qbytes) {
    HB_CUDA(cudaStreamSynchronize(c->stream));
    cudaFree(st.Q);
    st.Q = nullptr; st.Qbytes = 0;
    if(cudaMalloc(&st.Q, qbytes) != cudaSuccess) { cudaGetLastError(); return hb_fail(HB_ERR_ALLOC, "hb_syrk_rows_ozaki: cannot allocate the int8 slice buffer%s", ""); }
    st.Qbytes = qbytes;
    st.M = -1;
  }
  const int ncc = (int)((Kpad + Kc - 1) / Kc); // column chunks
  if(chunks_out) *chunks_out = ncc;
  if(st.sd_n < K) {
    HB_CUDA(cudaStreamSynchronize(c->stream));
    cudaFree(st.sd);
    HB_CUDA(cudaMalloc(&st.sd, sizeof(double) * K));
    st.sd_n = K;
  }
  if(st.mcap < Mpad) {
    HB_CUDA(cudaStreamSynchronize(c->stream));
    cudaFree(st.mx); cudaFree(st.e);
    HB_CUDA(cudaMalloc(&st.mx, sizeof(unsigned long long) * Mpad));
    HB_CUDA(cudaMalloc(&st.e, sizeof(int) * Mpad));
    st.mcap = Mpad;
  }
  if(st.M != M || st.K != K || st.S != S || st.Kc != Kc) {
    // schedule: tiles (bi, bj) with bj >= 2 bi cover the upper triangle; split the K stages of one column chunk so that ~all SMs get one
    // item (unchunked: the chunk is all of K)
    HB_CUDA(cudaStreamSynchronize(c->stream));
    const int nbi = Mpad / TM, nbj = Mpad / TN;
    std::vector<int2> tiles;
    for(int bi = 0; bi < nbi; bi++)
      for(int bj = 2 * bi; bj < nbj; bj++)
        if(bj * TN < M) tiles.push_back(make_int2(bi, bj));
    const int nt = (int)tiles.size();
    const long long kstages = Kc / KS;
    // K splits. Default: one wave, splits = SMs / tiles (every CTA gets one item; 72 tiles x 2 splits = 144 of 148 SMs at m = 1000).
    // Where that leaves the machine badly filled (81 tiles at m = 1024: one split, 81 of 148 SMs busy) several waves of the persistent
    // CTAs are considered: the makespan is ceil(tiles * splits / SMs) / splits of one tile's full-K time, e.g. 9 splits = 729 items = 4.9
    // waves -> 0.556 against the ideal 81/148 = 0.547. Bounds there: >= 64 K stages per split, partial-tile workspace <= 1 GB, <= 16
    // splits; ties go to the smaller count.
    int splits = c->num_sms / (nt > 0 ? nt : 1);
    if(splits < 1) splits = 1;
    if(splits > kstages) splits = (int)(kstages > 0 ? kstages : 1);
    {
      const long long items0 = (long long)nt * splits;
      const long long waves0 = (items0 + c->num_sms - 1) / c->num_sms;
      const double util0 = nt > 0 ? (double)items0 / (double)(waves0 * c->num_sms) : 1.0;
      if(util0 < 0.7) {
        double best = (double)waves0 / splits;
        const int smax = getenv("HB_OZ_MAX_SPLITS") ? atoi(getenv("HB_OZ_MAX_SPLITS")) : 16;
        for(int sp = 1; sp <= smax; sp++) {
          if(sp > 1 && (kstages / sp < 64 || (size_t)nt * sp * TM * TN * sizeof(double) > ((size_t)1 << 30))) break;
          const long long waves = ((long long)nt * sp + c->num_sms - 1) / c->num_sms;
          const double cost = (double)waves / sp;
          if(cost < best * (1.0 - 1e-3)) { best = cost; splits = sp; }
        }
      }
    }
    if(splits > kstages) splits = (int)(kstages > 0 ? kstages : 1);
    // the same tile x split list and slots for every chunk; the last chunk may be shorter (items with k_count = 0 do nothing)
    const long long last_stages = (Kpad - (long long)(ncc - 1) * Kc) / KS;
    std::vector<OzItem> items;
    for(long long cst : {kstages, last_stages})
      // split-major order: the CTAs of one split sweep the same K range concurrently (operand reuse in L2)
      for(int s = 0; s < splits; s++)
        for(int t = 0; t < nt; t++) {
          OzItem it;
          it.bi = tiles[t].x; it.bj = tiles[t].y;
          const long long b = hb_part_begin(cst, splits, s), e2 = hb_part_begin(cst, splits, s + 1);
          it.k_begin = (int)b; it.k_count = (int)(e2 - b);
          it.slot = t * splits + s;
          items.push_back(it);
        }
    cudaFree(st.d_items); cudaFree(st.d_tiles);
    HB_CUDA(cudaMalloc(&st.d_items, sizeof(OzItem) * items.size()));
    HB_CUDA(cudaMalloc(&st.d_tiles, sizeof(int2) * nt));
    HB_CUDA(cudaMemcpy(st.d_items, items.data(), sizeof(OzItem) * items.size(), cudaMemcpyHostToDevice));
    HB_CUDA(cudaMemcpy(st.d_tiles, tiles.data(), sizeof(int2) * nt, cudaMemcpyHostToDevice));
    // the maps describe the chunk buffer (row pitch Kc); every chunk is sliced into the same buffer, so they stay valid
    cuuint64_t dims[3] = {(cuuint64_t)Kc, (cuuint64_t)Mpad, (cuuint64_t)S};
    cuuint64_t strides[2] = {(cuuint64_t)Kc, (cuuint64_t)Kc * Mpad};
    cuuint32_t boxA[3] = {KS, TM, 1}, boxB[3] = {KS, TN, (cuuint32_t)S}, es[3] = {1, 1, 1};
    CUresult r1 = g_encode(&st.mapA, CU_TENSOR_MAP_DATA_TYPE_UINT8, 3, st.Q, dims, strides, boxA, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
                           CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    CUresult r2 = g_encode(&st.mapB, CU_TENSOR_MAP_DATA_TYPE_UINT8, 3, st.Q, dims, strides, boxB, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
                           CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if(r1 != CUDA_SUCCESS || r2 != CUDA_SUCCESS) return hb_fail(HB_ERR_CUDA, "cuTensorMapEncodeTiled failed%s", "");
    st.M = M; st.K = K; st.S = S; st.Mpad = Mpad; st.Kpad = Kpad; st.Kc = Kc; st.splits = splits; st.n_tiles = nt; st.n_items = nt * splits;
  }
  // 1. sqrt(d), row maxima and exponents over all K columns
  const double* sd = nullptr;
  if(d) {
    k_sqrt<<<c->num_sms * 8, 256, 0, c->stream>>>(K, d, st.sd);
    HB_LAUNCHED();
    sd = st.sd;
  }
  HB_CUDA(cudaMemsetAsync(st.mx, 0, sizeof(unsigned long long) * Mpad, c->stream));
  {
    if(dot_x && dot_out && K > 0) {
      const int nchunks = (int)((K + RD_COLS - 1) / RD_COLS);
      if(st.dot_cap < (size_t)nchunks * M) {
        HB_CUDA(cudaStreamSynchronize(c->stream));
        cudaFree(st.dot_partial);
        HB_CUDA(cudaMalloc(&st.dot_partial, sizeof(double) * (size_t)nchunks * M));
        st.dot_cap = (size_t)nchunks * M;
      }
      int rsplit = (2 * c->num_sms + nchunks - 1) / nchunks; // short shards: split the rows of a chunk over several CTAs
      rsplit = rsplit < 1 ? 1 : (rsplit > 8 ? 8 : rsplit);
      // pairs of columns need 16-byte aligned rows AND an even first column per lane (RD_COLS is even)
      if(rows_aligned16 && (K & 1) == 0)
        k_oz_rowmax_dot<true><<<dim3(nchunks, rsplit), RD_THREADS, 0, c->stream>>>(rowptr_dev, M, K, d, dot_x, st.mx, st.dot_partial);
      else
        k_oz_rowmax_dot<false><<<dim3(nchunks, rsplit), RD_THREADS, 0, c->stream>>>(rowptr_dev, M, K, d, dot_x, st.mx, st.dot_partial);
      HB_LAUNCHED();
      k_oz_dot_final<<<(M + 31) / 32, 256, 0, c->stream>>>(M, nchunks, st.dot_partial, dot_out);
      HB_LAUNCHED();
    } else {
      long long gx = (K + 256 * 64 - 1) / (256 * 64);
      if(gx < 1) gx = 1;
      if(gx > 64) gx = 64;
      k_oz_rowmax<<<dim3((unsigned)gx, M), 256, 0, c->stream>>>(rowptr_dev, M, K, sd, st.mx);
      HB_LAUNCHED();
    }
    k_oz_exponents<<<(Mpad + 127) / 128, 128, 0, c->stream>>>(M, st.mx, st.e);
    HB_LAUNCHED();
    hb_phase_mark(c, HB_PH_OZ_ROWMAX);
  }
  // 2. per column chunk: slices, then the tcgen05 GEMM into the FP64 partial tiles (the first chunk writes them, the later ones add)
  const int vec_ok = rows_aligned16 ? 1 : 0;
  // timed window (hb_ctx_last_syrk_ms): the GEMM; in chunked mode the slicing and GEMMs of all chunks
  if(c->timing && ncc > 1) HB_CUDA(cudaEventRecord(c->ev_syrk0, c->stream));
  for(int q = 0; q < ncc; q++) {
    const long long k0 = (long long)q * Kc;
    const long long kw = (K - k0 < Kc) ? K - k0 : Kc;
    const long long kwpad = ((kw + KS - 1) / KS) * KS;
    const unsigned sx = (unsigned)((kwpad / 8 + 255) / 256);
    if(S == 6) k_oz_slice<6><<<dim3(sx, Mpad), 256, 0, c->stream>>>(rowptr_dev, M, Mpad, k0, kw, kwpad, Kc, sd, st.e, st.Q, vec_ok);
    else if(S == 7) k_oz_slice<7><<<dim3(sx, Mpad), 256, 0, c->stream>>>(rowptr_dev, M, Mpad, k0, kw, kwpad, Kc, sd, st.e, st.Q, vec_ok);
    else k_oz_slice<8><<<dim3(sx, Mpad), 256, 0, c->stream>>>(rowptr_dev, M, Mpad, k0, kw, kwpad, Kc, sd, st.e, st.Q, vec_ok);
    HB_LAUNCHED();
    if(q == 0) {
      // the slicing phase mark only when the slicing is one phase; in chunked mode the slicing counts under the GEMM phase
      if(ncc == 1) hb_phase_mark(c, HB_PH_OZ_SLICE);
      HB_CHECK(hb_ws_reserve(c, sizeof(double) * (size_t)st.n_items * TM * TN));
      if(c->timing && ncc == 1) HB_CUDA(cudaEventRecord(c->ev_syrk0, c->stream));
    }
    const OzItem* items = st.d_items + (q == ncc - 1 ? st.n_items : 0);
    if(S == 6) HB_CHECK(launch_gemm<6>(c, st, items, chunk_stages, q > 0, (double*)c->ws));
    else if(S == 7) HB_CHECK(launch_gemm<7>(c, st, items, chunk_stages, q > 0, (double*)c->ws));
    else HB_CHECK(launch_gemm<8>(c, st, items, chunk_stages, q > 0, (double*)c->ws));
  }
  if(c->timing) {
    HB_CUDA(cudaEventRecord(c->ev_syrk1, c->stream));
    c->syrk_timed = true;
  }
  // 3. split-K reduction, row scales, symmetrisation
  k_oz_fixup<<<st.n_tiles, 256, 0, c->stream>>>(M, st.n_tiles, st.d_tiles, st.splits, (const double*)c->ws, st.e, C, ldc);
  HB_LAUNCHED();
  return HB_OK;
}
