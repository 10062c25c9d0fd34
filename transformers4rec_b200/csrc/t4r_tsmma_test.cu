// t4r_tsmma_test.cu -- probe for the A-from-TMEM ("TS") form of tcgen05.mma used by the fused FFN:
//   D[128, N] = A[128, 64] * B[N, 64]^T with A written to TMEM by tcgen05.st (bf16 pairs packed per
//   32-bit column, one row per lane) and B staged by TMA (128-byte swizzle).  Debug entry point only.
#include <cuda.h>

#include "t4r_common.cuh"
#include "t4r_tmem_ld.cuh"
#include "t4r_internal.h"

namespace t4r {

__device__ __forceinline__ void tmem_st8(uint32_t taddr, const uint32_t (&r)[8]) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"r"(taddr), "r"(r[0]),
               "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7])
               : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void umma_bf16_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t bdesc, uint32_t idesc,
                                             uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}"
      ::"r"(tmem_d), "r"(tmem_a), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}

template <int N>
__global__ void __launch_bounds__(128, 1)
tsmma_test_kernel(const __grid_constant__ CUtensorMap tmB, const float* __restrict__ A, float* __restrict__ D) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  uint64_t* bar_b = reinterpret_cast<uint64_t*>(smem + N * 128);
  uint64_t* bar_d = bar_b + 1;
  uint32_t* slot = reinterpret_cast<uint32_t*>(bar_d + 1);
  const int warp = warp_id(), lane = lane_id();
  if (threadIdx.x == 0) {
    mbar_init(bar_b, 1);
    mbar_init(bar_d, 1);
    fence_barrier_init();
  }
  if (warp == 0) {
    tmem_alloc(slot, 512);
    tmem_relinquish();
  }
  tc_fence_before_sync();
  __syncthreads();
  tc_fence_after_sync();
  const uint32_t tmem = *slot;
  const uint32_t d_col = 0, a_col = 256;  // D: N columns at 0; A: 32 columns (64 bf16) at 256
  if (threadIdx.x == 0) {
    mbar_arrive_expect_tx(bar_b, N * 128);
    tma_load_2d(smem, &tmB, bar_b, 0, 0);
  }
  // every thread owns one row of A: round to bf16, pack pairs, store 32 columns to its TMEM lane
  {
    const float* row = A + static_cast<int64_t>(threadIdx.x) * 64;
    const uint32_t taddr = tmem + (static_cast<uint32_t>(warp * 32) << 16) + a_col;
#pragma unroll
    for (int c = 0; c < 4; ++c) {
      uint32_t r[8];
#pragma unroll
      for (int j = 0; j < 8; ++j)
        r[j] = pack_bf16x2(__float2bfloat16_rn(row[c * 16 + 2 * j]), __float2bfloat16_rn(row[c * 16 + 2 * j + 1]));
      tmem_st8(taddr + c * 8, r);
    }
    tmem_st_wait();
  }
  tc_fence_before_sync();
  __syncthreads();
  tc_fence_after_sync();
  if (threadIdx.x == 0) {
    mbar_wait(bar_b, 0);
    tc_fence_after_sync();
    constexpr uint32_t idesc = umma_idesc_bf16(128, N);
#pragma unroll
    for (int k4 = 0; k4 < 4; ++k4)
      umma_bf16_ts(tmem + d_col, tmem + a_col + k4 * 8, umma_desc_sw128(smem_u32(smem) + k4 * 32), idesc, k4 != 0);
    umma_commit(bar_d);
  }
  __syncwarp();
  mbar_wait(bar_d, 0);
  tc_fence_after_sync();
  {
    const uint32_t taddr = tmem + (static_cast<uint32_t>(warp * 32) << 16) + d_col;
    for (int c = 0; c < N / 32; ++c) {
      float v[32];
      tmem_ld<32>(taddr + c * 32, v);
      for (int j = 0; j < 32; ++j) D[static_cast<int64_t>(threadIdx.x) * N + c * 32 + j] = v[j];
    }
  }
  tc_fence_before_sync();
  __syncthreads();
  tc_fence_after_sync();
  if (warp == 0) tmem_dealloc(tmem, 512);
}

int make_tmap_public(CUtensorMap* map, const __nv_bfloat16* base, int64_t rows, int Kp, int box_rows);

}  // namespace t4r

/* debug: D[128, N] = bf16(A[128, 64]) * B_hi[N, 64]^T via the TS form (A in TMEM); N in {64, 128, 256} */
extern "C" int t4r_debug_ts_mma(const float* A, const void* b_planes, int N, float* D, void* stream) {
  using namespace t4r;
  T4R_REQUIRE(A && b_planes && D && (N == 64 || N == 128 || N == 256), "debug_ts_mma: bad arguments");
  CUtensorMap tb;
  T4R_TRY(make_tmap_public(&tb, static_cast<const __nv_bfloat16*>(b_planes), N, 64, N));
  const int smem = N * 128 + 1024 + 64;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  if (N == 64) {
    T4R_CUDA(cudaFuncSetAttribute(tsmma_test_kernel<64>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    tsmma_test_kernel<64><<<1, 128, smem, s>>>(tb, A, D);
  } else if (N == 128) {
    T4R_CUDA(cudaFuncSetAttribute(tsmma_test_kernel<128>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    tsmma_test_kernel<128><<<1, 128, smem, s>>>(tb, A, D);
  } else {
    T4R_CUDA(cudaFuncSetAttribute(tsmma_test_kernel<256>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    tsmma_test_kernel<256><<<1, 128, smem, s>>>(tb, A, D);
  }
  T4R_LAUNCH_CHECK("tsmma_test_kernel");
  return 0;
}
