// t4r_common.cuh -- sm_100a device primitives shared by the t4r_b200 kernels.
//
// Hand-written PTX wrappers for mbarrier, TMA (cp.async.bulk.tensor), tcgen05
// (alloc / mma / commit / ld / fences) and small warp-level helpers.  No CUTLASS,
// no CuTe: the descriptor bit layouts below were checked against
// cute/arch/mma_sm100_desc.hpp (SmemDescriptor / InstrDescriptor) but nothing is
// included from there.
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdint.h>

namespace t4r {

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

__device__ __forceinline__ int lane_id() { return threadIdx.x & 31; }
__device__ __forceinline__ int warp_id() { return threadIdx.x >> 5; }

// ----------------------------------------------------------------------------
// mbarrier
// ----------------------------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_barrier_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.b32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
// Bounded wait: a broken pipeline traps (kernel aborts with an error the host
// sees) instead of spinning forever on a shared GPU box.
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  uint32_t spins = 0;
  while (!mbar_try_wait(bar, parity)) {
    if (++spins > (1u << 26)) __trap();
  }
}

// ----------------------------------------------------------------------------
// TMA: 2-D tiled bulk tensor load, completion on an mbarrier
// ----------------------------------------------------------------------------
__device__ __forceinline__ void tma_prefetch_desc(const void* tmap) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(tmap)) : "memory");
}
__device__ __forceinline__ void tma_load_2d(void* smem_dst, const void* tmap, uint64_t* bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(tmap)), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
      : "memory");
}

// ----------------------------------------------------------------------------
// tcgen05 / TMEM
// ----------------------------------------------------------------------------
__device__ __forceinline__ void tmem_alloc(uint32_t* smem_dst, uint32_t ncols) {  // whole warp
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_dst)),
               "r"(ncols)
               : "memory");
}
__device__ __forceinline__ void tmem_relinquish() {  // whole warp
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {  // whole warp
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tc_fence_before_sync() {
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_after_sync() {
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
}
// D[tmem] (+)= A[smem desc] * B[smem desc]; one thread issues for the CTA.
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                          uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// all previously issued MMAs of this thread complete -> one arrive on the mbarrier
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
               : "memory");
}

// ----------------------------------------------------------------------------
// CTA pairs (cta_group::2): two SMs of a TPC cooperate on one 256-row MMA tile.  Addresses of a CTA's
// shared memory inside the cluster window differ from its peer's in bit 24 only; clearing it turns the
// address of an object in CTA 1 into the address of the same object in CTA 0 (the leader).
// ----------------------------------------------------------------------------
constexpr uint32_t kPeerBitMask = 0xFEFFFFFFu;
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {  // every thread of both CTAs
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// TMA load issued by either CTA of a pair; the transaction bytes are credited to the LEADER's barrier
__device__ __forceinline__ void tma_load_2d_pair(void* smem_dst, const void* tmap, uint64_t* leader_bar_local, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(tmap)), "r"(smem_u32(leader_bar_local) & kPeerBitMask),
        "r"(c0), "r"(c1)
      : "memory");
}
// arrive on the leader CTA's copy of a barrier (from either CTA)
__device__ __forceinline__ void mbar_arrive_leader(uint64_t* bar_local) {
  asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(smem_u32(bar_local) & kPeerBitMask) : "memory");
}
__device__ __forceinline__ void tmem_alloc_pair(uint32_t* smem_dst, uint32_t ncols) {  // one warp in EACH CTA
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_dst)), "r"(ncols)
               : "memory");
}
__device__ __forceinline__ void tmem_relinquish_pair() {
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc_pair(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
// D[256 x N] (+)= A[256 x 16] * B[N x 16]^T: rows 0-127 of A / D live in the leader, 128-255 in the peer; each CTA
// holds N/2 rows of B.  Issued by one thread of the leader; descriptors are offsets valid in both CTAs.
__device__ __forceinline__ void umma_bf16_pair(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                               uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// completion of all MMAs issued so far by this thread -> arrive on the barrier at this offset in BOTH CTAs
__device__ __forceinline__ void umma_commit_pair(uint64_t* bar_local) {
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
               ::"r"(smem_u32(bar_local)), "h"(static_cast<uint16_t>(3))
               : "memory");
}

// UMMA shared-memory matrix descriptor for a K-major operand tile stored as rows
// of 128 bytes with the 128-byte swizzle (what TMA SWIZZLE_128B produces):
//   bits [0,14)  start address >> 4
//   bits [16,30) leading byte offset >> 4  (unused for swizzled K-major; 1)
//   bits [32,46) stride byte offset >> 4   (8 rows * 128 B = 1024 -> 64)
//   bits [46,48) descriptor version = 1 (sm_100)
//   bits [61,64) layout type: 2 = SWIZZLE_128B
__device__ __forceinline__ uint64_t umma_desc_sw128(uint32_t smem_addr) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((smem_addr >> 4) & 0x3FFFu);
  d |= static_cast<uint64_t>(1) << 16;
  d |= static_cast<uint64_t>(1024 >> 4) << 32;
  d |= static_cast<uint64_t>(1) << 46;
  d |= static_cast<uint64_t>(2) << 61;
  return d;
}
// Instruction descriptor, kind::f16: A,B = bf16 (format 1), D = f32 (format 1),
// both operands K-major, M = 128, N = n.
__host__ __device__ constexpr uint32_t umma_idesc_bf16(int m, int n) {
  return (1u << 4) | (1u << 7) | (1u << 10) | (static_cast<uint32_t>(n >> 3) << 17) |
         (static_cast<uint32_t>(m >> 4) << 24);
}

// kind::f16 with fp16 operands (format 0) and kind::f8f6f4 with e4m3 operands (format 0): the bit patterns
// coincide -- the KIND in the instruction selects the interpretation (cute/arch/mma_sm100_desc.hpp:
// F32F16Format F16 = 0, MXF8F6F4Format E4M3 = 0).  Used by the 2-unit product (nprod = 2, t4r_mixed_pack.cuh).
__host__ __device__ constexpr uint32_t umma_idesc_f16(int m, int n) {
  return (1u << 4) | (static_cast<uint32_t>(n >> 3) << 17) | (static_cast<uint32_t>(m >> 4) << 24);
}
__host__ __device__ constexpr uint32_t umma_idesc_e4m3(int m, int n) {
  return (1u << 4) | (static_cast<uint32_t>(n >> 3) << 17) | (static_cast<uint32_t>(m >> 4) << 24);
}
// D[tmem] (+)= A * B with 8-bit operands: K = 32 per instruction (32 bytes of each K-major operand row, the same
// shared-memory footprint per instruction as a K = 16 bf16 MMA), twice the MACs of a kind::f16 MMA per issue slot.
__device__ __forceinline__ void umma_f8(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                        uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f8f6f4 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void umma_f8_pair(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                             uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f8f6f4 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}

// ----------------------------------------------------------------------------
// split-bf16 helpers: x = hi + lo with hi = bf16(x), lo = bf16(x - hi)
// (three bf16 products hi*hi + hi*lo + lo*hi carry ~2^-16 relative error)
// ----------------------------------------------------------------------------
__device__ __forceinline__ void split_bf16(float x, __nv_bfloat16& hi, __nv_bfloat16& lo) {
  hi = __float2bfloat16_rn(x);
  lo = __float2bfloat16_rn(x - __bfloat162float(hi));
}
// Split two floats at once: hi/lo words hold element a in bits [0,16) and b in [16,32) (memory order a, b).
// cvt.rn.bf16x2.f32 is one full-rate F2FP per PAIR; the scalar __float2bfloat16_rn lowers to F2F.BF16.F32
// on the quarter-rate XU pipe (2 per element), which made every plane-writing epilogue XU-bound.
// Same round-to-nearest-even results as split_bf16.
__device__ __forceinline__ void split_bf16x2(float a, float b, uint32_t& hi, uint32_t& lo) {
  asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(hi) : "f"(b), "f"(a));
  const float ra = a - __uint_as_float(hi << 16);
  const float rb = b - __uint_as_float(hi & 0xffff0000u);
  asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(lo) : "f"(rb), "f"(ra));
}
__device__ __forceinline__ uint32_t pack_bf16x2(__nv_bfloat16 a, __nv_bfloat16 b) {
  return static_cast<uint32_t>(__bfloat16_as_ushort(a)) | (static_cast<uint32_t>(__bfloat16_as_ushort(b)) << 16);
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

// 2^x on the SFU (ex2.approx.ftz: 2 ulp, exact 0 for x = -inf); used for the online softmax
__device__ __forceinline__ float fast_exp2(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

// erf via Abramowitz & Stegun 7.1.26 (|abs error| <= 1.5e-7; ~14 instructions with two SFU
// ops instead of erff's ~30 with a branch).  The GELU epilogue of the 4d-wide FFN GEMM is
// instruction-bound, and 1.5e-7 is far inside the 1e-3 parity budget.
__device__ __forceinline__ float fast_erf(float x) {
  const float ax = fabsf(x);
  float t;  // 1 / (1 + p|x|): argument >= 1, so the branch-free SFU reciprocal (1 ulp) is safe
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(t) : "f"(fmaf(0.3275911f, ax, 1.0f)));
  float p = fmaf(1.061405429f, t, -1.453152027f);
  p = fmaf(p, t, 1.421413741f);
  p = fmaf(p, t, -0.284496736f);
  p = fmaf(p, t, 0.254829592f);
  p *= t;
  const float e = fast_exp2(-ax * ax * 1.4426950408889634f);
  const float r = fmaf(-p, e, 1.0f);
  return copysignf(r, x);
}
__device__ __forceinline__ float gelu_erf(float x) { return 0.5f * x * (1.0f + fast_erf(x * 0.70710678118654752440f)); }

// Packed-pair forms (Blackwell fma.rn.f32x2 / mul / add: two fp32 lanes per issue slot).  The epilogue warps of the
// feed-forward kernels are issue/latency bound (two warps per scheduler), so halving the FMA-type instruction count
// is what shortens the GELU chunk.  Same A&S 7.1.26 polynomial as fast_erf (evaluated in -t, which only flips signs);
// the final 0.5 x (1 + erf) is one fused multiply-add here, so results agree with gelu_erf to 1 ulp.
__device__ __forceinline__ float2 gelu_erf2(float2 x) {
  const float2 z = __fmul2_rn(x, make_float2(0.70710678118654752440f, 0.70710678118654752440f));
  const float2 ax = make_float2(fabsf(z.x), fabsf(z.y));
  const float2 nd = __ffma2_rn(make_float2(-0.3275911f, -0.3275911f), ax, make_float2(-1.0f, -1.0f));
  float2 nt;  // -1 / (1 + p|z|)
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(nt.x) : "f"(nd.x));
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(nt.y) : "f"(nd.y));
  float2 q = __ffma2_rn(make_float2(1.061405429f, 1.061405429f), nt, make_float2(1.453152027f, 1.453152027f));
  q = __ffma2_rn(q, nt, make_float2(1.421413741f, 1.421413741f));
  q = __ffma2_rn(q, nt, make_float2(0.284496736f, 0.284496736f));
  q = __ffma2_rn(q, nt, make_float2(0.254829592f, 0.254829592f));
  q = __fmul2_rn(q, nt);  // = -p(t)
  const float2 a2 = __fmul2_rn(ax, ax);
  const float2 ea = __fmul2_rn(a2, make_float2(-1.4426950408889634f, -1.4426950408889634f));
  const float2 e = make_float2(fast_exp2(ea.x), fast_exp2(ea.y));
  const float2 r = __ffma2_rn(q, e, make_float2(1.0f, 1.0f));  // 1 - p e  (>= 0)
  const float2 erf2 = make_float2(copysignf(r.x, z.x), copysignf(r.y, z.y));
  const float2 h = __fmul2_rn(x, make_float2(0.5f, 0.5f));
  return __ffma2_rn(h, erf2, h);
}
__device__ __forceinline__ void split_bf16x2(float2 v, uint32_t& hi, uint32_t& lo) {
  asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(hi) : "f"(v.y), "f"(v.x));
  const float2 f = make_float2(__uint_as_float(hi << 16), __uint_as_float(hi & 0xffff0000u));
  const float2 r = __ffma2_rn(f, make_float2(-1.0f, -1.0f), v);  // v - f, exact product
  asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(lo) : "f"(r.y), "f"(r.x));
}

}  // namespace t4r
