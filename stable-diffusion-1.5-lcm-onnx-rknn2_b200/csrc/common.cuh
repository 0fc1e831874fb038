// Common device/host helpers for the dreamlab_b200 kernels (sm_100a only).
// Thin inline-PTX wrappers: mbarrier, TMA (cp.async.bulk.tensor), tcgen05 (UMMA/TMEM).
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdint.h>
#include <stdio.h>

#include "dreamlab_b200.h"

namespace dl {

// ----------------------------------------------------------------------------------------------
// host-side error plumbing (C-ABI returns int status; text via dl_last_error())
// ----------------------------------------------------------------------------------------------
void set_error(const char* fmt, ...);
int check_launch(const char* what);          // cudaGetLastError → status
const char* last_error();

#define DL_CHECK_ARG(cond, ...)                                  \
  do {                                                           \
    if (!(cond)) { ::dl::set_error(__VA_ARGS__); return 1; }     \
  } while (0)

// driver entry point (no -lcuda link: libcuda is absent in the CPU build container)
typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*,
                                    const cuuint64_t*, const cuuint64_t*, const cuuint32_t*,
                                    const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                    CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
PFN_encodeTiled get_encode_tiled();

// Encode a bf16 tensor map, up to 4 dims (innermost first), 128B swizzle, zero OOB fill.
int make_tmap_bf16(CUtensorMap* out, const void* base, int rank, const uint64_t* dims,
                   const uint64_t* strides_bytes /* rank-1 entries */, const uint32_t* box,
                   CUtensorMapSwizzle swizzle = CU_TENSOR_MAP_SWIZZLE_128B);

int num_sms();

// ----------------------------------------------------------------------------------------------
// device helpers
// ----------------------------------------------------------------------------------------------
#ifdef __CUDACC__

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

__device__ __forceinline__ bool elect_one() {
  uint32_t pred = 0;
  asm volatile(
      "{\n\t.reg .pred P;\n\t"
      "elect.sync _|P, 0xffffffff;\n\t"
      "selp.b32 %0, 1, 0, P;\n\t}"
      : "=r"(pred));
  return pred != 0;
}

// ---- mbarrier ----
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void fence_barrier_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void fence_proxy_async_smem() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)),
               "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred P;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 P, [%1], %2;\n\t"
      "selp.b32 %0, 1, 0, P;\n\t}"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
// Bounded wait: a protocol bug becomes a trap (launch error) instead of a hung GPU.
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  if (mbar_try_wait(bar, parity)) return;
  uint64_t t0 = 0;
  uint32_t spins = 0;
  while (!mbar_try_wait(bar, parity)) {
    if (++spins == 4096) {
      uint64_t now;
      asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(now));
      if (t0 == 0) t0 = now;
      else if (now - t0 > 4000000000ull) {   // 4 s
        printf("dreamlab_b200: mbarrier wait timeout (block %d,%d,%d thread %d)\n", blockIdx.x,
               blockIdx.y, blockIdx.z, threadIdx.x);
        __trap();
      }
      spins = 0;
    }
  }
}

// ---- TMA ----
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* m) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(m)) : "memory");
}
__device__ __forceinline__ void tma_load_2d(void* dst, const CUtensorMap* m, uint64_t* bar, int c0,
                                            int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes"
      " [%0], [%1, {%3, %4}], [%2];" ::"r"(smem_u32(dst)),
      "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tma_load_3d(void* dst, const CUtensorMap* m, uint64_t* bar, int c0,
                                            int c1, int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes"
      " [%0], [%1, {%3, %4, %5}], [%2];" ::"r"(smem_u32(dst)),
      "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}
__device__ __forceinline__ void tma_load_4d(void* dst, const CUtensorMap* m, uint64_t* bar, int c0,
                                            int c1, int c2, int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.tile.mbarrier::complete_tx::bytes"
      " [%0], [%1, {%3, %4, %5, %6}], [%2];" ::"r"(smem_u32(dst)),
      "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
      : "memory");
}

// TMA store: shared (swizzled per the tensor map) -> global tile; bulk-group completion
__device__ __forceinline__ void tma_store_4d(const CUtensorMap* m, const void* src, int c0, int c1,
                                             int c2, int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.global.shared::cta.bulk_group [%0, {%2, %3, %4, %5}], [%1];" ::"l"(
          reinterpret_cast<uint64_t>(m)),
      "r"(smem_u32(src)), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
      : "memory");
}
__device__ __forceinline__ void bulk_commit_group() {
  asm volatile("cp.async.bulk.commit_group;" ::: "memory");
}
template <int N>
__device__ __forceinline__ void bulk_wait_group_read() {
  asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory");
}
__device__ __forceinline__ void bulk_wait_group_all() {
  asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
}
__device__ __forceinline__ void named_bar_sync(int id, int nthreads) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}

// 1-D bulk async copy global -> shared (TMA engine, no tensor map), completes on an mbarrier
__device__ __forceinline__ void bulk_load_1d(void* dst, const void* src, uint32_t bytes,
                                             uint64_t* bar) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::
      "r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(src)), "r"(bytes), "r"(smem_u32(bar))
      : "memory");
}

// ---- tcgen05 / TMEM ----
__device__ __forceinline__ void tmem_alloc(uint32_t* smem_dst, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(
                   smem_u32(smem_dst)),
               "r"(ncols)
               : "memory");
}
__device__ __forceinline__ void tmem_relinquish() {
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols)
               : "memory");
}
__device__ __forceinline__ void tc_fence_before() {
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_after() {
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
}
// tcgen05.commit: arrive on mbarrier when all prior tcgen05 async ops of this thread retire.
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(
                   smem_u32(bar))
               : "memory");
}
// D[tmem] (+)= A[smem] * B[smem], bf16 inputs, fp32 accumulate
__device__ __forceinline__ void umma_ss(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc,
                                        uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(d_tmem),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// D[tmem] (+)= A[tmem] * B[smem]
__device__ __forceinline__ void umma_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t bdesc,
                                        uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}" ::"r"(d_tmem),
      "r"(a_tmem), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}

// K-major, 128B-swizzled operand tile: rows are 128 B (64 bf16), 8-row atoms of 1024 B.
// (canonical layout ((8,n),2):((8,SBO),1) in 16-byte units; version=1 for sm_100)
__device__ __forceinline__ uint64_t umma_desc_kmajor_sw128(uint32_t smem_addr, uint32_t sbo_bytes) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr >> 4) & 0x3FFF);
  d |= (uint64_t)1 << 16;                              // LBO (ignored for swizzled K-major)
  d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32;    // SBO: stride between 8-row groups
  d |= (uint64_t)1 << 46;                              // descriptor version (Blackwell)
  d |= (uint64_t)2 << 61;                              // SWIZZLE_128B
  return d;
}
// MN-major, 128B-swizzled operand tile: 64 MN-elements contiguous (128 B) per K row,
// 8 K-rows per 1024 B atom. LBO = byte stride between 64-wide MN chunks, SBO = between 8-row K groups.
__device__ __forceinline__ uint64_t umma_desc_mnmajor_sw128(uint32_t smem_addr, uint32_t lbo_bytes,
                                                            uint32_t sbo_bytes) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr >> 4) & 0x3FFF);
  d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16;
  d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)2 << 61;
  return d;
}
// Split form of the same descriptors: the upper word (SBO, version, swizzle) is loop-invariant,
// the lower word is (address >> 4) | LBO << 16 — advancing along K is a 32-bit add.
__device__ __forceinline__ uint32_t umma_desc_hi_sw128(uint32_t sbo_bytes) {
  return ((sbo_bytes >> 4) & 0x3FFF) | (1u << 14) | (2u << 29);
}
__device__ __forceinline__ uint32_t umma_desc_lo(uint32_t smem_addr, uint32_t lbo_bytes = 16) {
  return ((smem_addr >> 4) & 0x3FFF) | (((lbo_bytes >> 4) & 0x3FFF) << 16);
}
__device__ __forceinline__ void umma_ss_lohi(uint32_t d_tmem, uint32_t a_lo, uint32_t b_lo,
                                             uint32_t desc_hi, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t.reg .b64 da, db;\n\t"
      "mov.b64 da, {%1, %3};\n\t"
      "mov.b64 db, {%2, %3};\n\t"
      "setp.ne.b32 p, %5, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %4, p;\n\t}" ::"r"(d_tmem),
      "r"(a_lo), "r"(b_lo), "r"(desc_hi), "r"(idesc), "r"(accumulate)
      : "memory");
}
// TS form: A from TMEM, B descriptor split
__device__ __forceinline__ void umma_ts_lohi(uint32_t d_tmem, uint32_t a_tmem, uint32_t b_lo,
                                             uint32_t desc_hi, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t.reg .b64 db;\n\t"
      "mov.b64 db, {%2, %3};\n\t"
      "setp.ne.b32 p, %5, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], db, %4, p;\n\t}" ::"r"(d_tmem),
      "r"(a_tmem), "r"(b_lo), "r"(desc_hi), "r"(idesc), "r"(accumulate)
      : "memory");
}

// instruction descriptor: bf16 x bf16 -> fp32, M x N, majors: 0 = K-major, 1 = MN-major
__device__ __host__ __forceinline__ uint32_t umma_idesc_bf16(uint32_t M, uint32_t N,
                                                             uint32_t a_mn_major = 0,
                                                             uint32_t b_mn_major = 0) {
  return (1u << 4) | (1u << 7) | (1u << 10) | (a_mn_major << 15) | (b_mn_major << 16) |
         ((N >> 3) << 17) | ((M >> 4) << 24);
}

// TMEM -> registers: this warp's 32 lanes x 16 consecutive fp32 columns
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]),
        "=r"(r[7]), "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]),
        "=r"(r[14]), "=r"(r[15])
      : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]),
        "=r"(r[7]), "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]),
        "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]),
        "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]),
        "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld_wait() {
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}
// registers -> TMEM: this warp's 32 lanes x 16 consecutive 32-bit columns
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};" ::"r"(taddr),
      "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]),
      "r"(r[8]), "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15])
      : "memory");
}
__device__ __forceinline__ void tmem_st8(uint32_t taddr, const uint32_t (&r)[8]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"r"(taddr),
      "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7])
      : "memory");
}
__device__ __forceinline__ void tmem_st_wait() {
  asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
}

// ---- small numeric helpers ----
// packed bf16 in, packed bf16 out: saves the fp32 -> bf16 conversion of the results (in sm_100a SASS it is
// still two MUFU.EX2.BF16, one per half, + a PRMT — not two exponentials per XU op)
__device__ __forceinline__ uint32_t ex2_bf16x2(uint32_t packed) {
  uint32_t r;
  asm("ex2.approx.ftz.bf16x2 %0, %1;" : "=r"(r) : "r"(packed));
  return r;
}
__device__ __forceinline__ float fast_exp2(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
// 2^x WITHOUT the MUFU pipe (16 lanes / clk / SM, and `ex2.approx.*x2` is lowered to two MUFU ops on
// sm_100a, so the packed form saves no XU cycles): Cody-Waite split x = n + f with |f| <= 0.5 by
// the 1.5 * 2^23 rounding constant, degree-3 minimax polynomial of 2^f (max rel err 7.7e-5, far
// below the bf16 rounding of P), n added into the exponent field as an integer.  ~8 FMA / ALU
// pipe instructions.  x <= -125 (masked keys: -inf) returns ~2^-125, which rounds away in P.
__device__ __forceinline__ float poly_exp2(float x) {
  x = fmaxf(x, -125.0f);
  const float r = x + 12582912.0f;                     // low mantissa bits of r hold round(x)
  const float f = x - (r - 12582912.0f);
  float p = fmaf(0.05508873611688614f, f, 0.242604061961174f);
  p = fmaf(p, f, 0.6932762265205383f);
  p = fmaf(p, f, 0.9999289512634277f);
  return __int_as_float(__float_as_int(p) + (__float_as_int(r) << 23));
}
// silu(x) = x*sigmoid(x) = h + h*tanh(h), h = x/2: ONE MUFU op (tanh.approx, rel err 2^-11, below
// bf16 output rounding).  exp + reciprocal (2 MUFU + a precise divide) made GroupNorm+SiLU
// MUFU-/ALU-bound instead of HBM-bound.
__device__ __forceinline__ float silu_f(float x) {
  const float h = 0.5f * x;
  float t;
  asm("tanh.approx.f32 %0, %1;" : "=f"(t) : "f"(h));
  return fmaf(h, t, h);
}
// Exact (erf) GELU evaluated through a fitted tanh form:
//   gelu(x) = x*Phi(x) ~= h + h*tanh(x*(a + b*t + c*t^2)),  h = x/2, t = min(x^2, 100)
// (a, b, c) minimise the max abs error against 0.5*x*(1+erf(x/sqrt2)): 2.5e-5 over all x, plus
// tanh.approx's 2^-11 relative error — far below the bf16 precision of the GEGLU output.
// 8 instructions, one of them on the otherwise idle MUFU pipe (libm erff: ~40; a polynomial
// erf: 17) — the GEGLU epilogue was ALU-bound.
__device__ __forceinline__ float gelu_erf_f(float x) {
  const float t = fminf(x * x, 100.0f);
  float p = fmaf(-3.51516780e-04f, t, 3.70056460e-02f);
  p = fmaf(p, t, 7.97507884e-01f);
  float th;
  asm("tanh.approx.f32 %0, %1;" : "=f"(th) : "f"(x * p));
  const float h = 0.5f * x;
  return fmaf(h, th, h);
}
__device__ __forceinline__ uint32_t pack_bf16x2(float lo, float hi) {
  __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&v);
}
__device__ __forceinline__ float2 unpack_bf16x2(uint32_t u) {
  __nv_bfloat162 v = *reinterpret_cast<__nv_bfloat162*>(&u);
  return __bfloat1622float2(v);
}
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

// LCMScheduler.step's predicted_original_sample from the model output mo (DL_PRED_*), each mul / sub / div rounded
// on its own as the fp32 torch ops are, then `clip_sample`'s clamp to [-r, r].
template <int PRED>
__device__ __forceinline__ float lcm_x0(float mo, float x, float sqrt_alpha_t, float sqrt_beta_t, int clip,
                                        float r) {
  static_assert(PRED == DL_PRED_EPSILON || PRED == DL_PRED_V || PRED == DL_PRED_SAMPLE, "prediction type");
  float x0;
  if constexpr (PRED == DL_PRED_EPSILON) {
    x0 = __fdiv_rn(__fsub_rn(x, __fmul_rn(sqrt_beta_t, mo)), sqrt_alpha_t);
  } else if constexpr (PRED == DL_PRED_V) {
    x0 = __fsub_rn(__fmul_rn(sqrt_alpha_t, x), __fmul_rn(sqrt_beta_t, mo));
  } else {
    x0 = mo;
  }
  if (clip) x0 = fminf(fmaxf(x0, -r), r);
  return x0;
}

#endif  // __CUDACC__

}  // namespace dl
