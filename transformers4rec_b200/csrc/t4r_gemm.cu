// t4r_gemm.cu -- persistent, warp-specialised tcgen05 GEMM for sm_100a.
//
//   C[M, N] = epilogue( A[M, K] * B[N, K]^T )
//
// A and B arrive as split-bf16 planes (hi, lo; see include/t4r_b200.h), are staged
// into shared memory by TMA (128-byte swizzle, K-major), multiplied by
// tcgen05.mma (kind::f16, bf16 x bf16 -> fp32 in TMEM; three products per K step:
// hi*hi + hi*lo + lo*hi) and drained by four epilogue warps with tcgen05.ld.
//
// Roles (320 threads): warp 0 = TMA producer, warp 1 = MMA issuer, warps 2-9 =
// epilogue (TMEM lane quadrant = warp_id % 4; warps 2-5 own the first half of a
// tile's columns, warps 6-9 the second half).  Two accumulator stages in TMEM let
// the epilogue of tile i overlap the main loop of tile i+1.  Tiles are visited
// m-fastest so CTAs running at the same time share the B tile in L2.
//
// Epilogues: dense (bias / ReLU / GELU / mask-replace / residual / LayerNorm, fp32
// and split-bf16 outputs) and head (online log-sum-exp partials + label rank).
#include <cuda.h>
#include <math.h>
#include <stdlib.h>
#include <mutex>
#include <unordered_map>

#include "t4r_common.cuh"
#include "t4r_tmem_ld.cuh"
#include "t4r_internal.h"

namespace t4r {

// ----------------------------------------------------------------------------
// tensor maps (driver entry point resolved at run time: no link-time libcuda)
// ----------------------------------------------------------------------------
typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                    const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                    CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static PFN_encodeTiled get_encode_fn() {
  static PFN_encodeTiled fn = nullptr;
  static std::once_flag once;
  std::call_once(once, []() {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult qres;
    cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres);
    if (e == cudaSuccess && qres == cudaDriverEntryPointSuccess) fn = reinterpret_cast<PFN_encodeTiled>(p);
  });
  return fn;
}

// Descriptors are pure functions of (base, rows, Kp, box_rows): encoded once and kept (the same weights, the same
// workspace slices and the same grow-only activation buffers come back every step; cuTensorMapEncodeTiled costs a
// microsecond or two of host time per call and a GEMM launch needs four to six of them -- the launch-bound small
// configurations spent a third of their host time here).  Bounded: the table is dropped when it reaches 8192 entries.
struct TmapKey {
  const void* base; int64_t rows; int Kp, box_rows;
  bool operator==(const TmapKey& o) const {
    return base == o.base && rows == o.rows && Kp == o.Kp && box_rows == o.box_rows;
  }
};
struct TmapKeyHash {
  size_t operator()(const TmapKey& k) const {
    uint64_t h = reinterpret_cast<uintptr_t>(k.base) * 0x9E3779B97F4A7C15ull;
    h ^= static_cast<uint64_t>(k.rows) * 0xC2B2AE3D27D4EB4Full + (static_cast<uint64_t>(k.Kp) << 20) +
         (static_cast<uint64_t>(k.box_rows) << 8);
    return static_cast<size_t>(h ^ (h >> 29));
  }
};
static std::mutex g_tmap_mu;
static std::unordered_map<TmapKey, CUtensorMap, TmapKeyHash> g_tmap_cache;

static int make_tmap_uncached(CUtensorMap* map, const __nv_bfloat16* base, int64_t rows, int Kp, int box_rows);
static int make_tmap(CUtensorMap* map, const __nv_bfloat16* base, int64_t rows, int Kp, int box_rows) {
  const TmapKey key{base, rows, Kp, box_rows};
  {
    std::lock_guard<std::mutex> lk(g_tmap_mu);
    auto it = g_tmap_cache.find(key);
    if (it != g_tmap_cache.end()) { *map = it->second; return 0; }
  }
  T4R_TRY(make_tmap_uncached(map, base, rows, Kp, box_rows));
  std::lock_guard<std::mutex> lk(g_tmap_mu);
  if (g_tmap_cache.size() >= 8192) g_tmap_cache.clear();
  g_tmap_cache.emplace(key, *map);
  return 0;
}

// box = 64 bf16 (128 bytes) of K x box_rows rows, 128-byte swizzle
static int make_tmap_uncached(CUtensorMap* map, const __nv_bfloat16* base, int64_t rows, int Kp, int box_rows) {
  PFN_encodeTiled fn = get_encode_fn();
  if (!fn) {
    set_error("cuTensorMapEncodeTiled entry point not available (no CUDA driver?)");
    return T4R_ERR_CUDA;
  }
  if ((reinterpret_cast<uintptr_t>(base) & 15) != 0) {
    set_error("operand planes must be 16-byte aligned");
    return T4R_ERR_INVALID;
  }
  cuuint64_t gdim[2] = {static_cast<cuuint64_t>(Kp), static_cast<cuuint64_t>(rows)};
  cuuint64_t gstride[1] = {static_cast<cuuint64_t>(Kp) * 2};
  cuuint32_t box[2] = {64u, static_cast<cuuint32_t>(box_rows)};
  cuuint32_t estr[2] = {1u, 1u};
  CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<__nv_bfloat16*>(base), gdim, gstride, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled failed (CUresult %d) rows=%lld Kp=%d box_rows=%d", (int)r, (long long)rows, Kp,
              box_rows);
    return T4R_ERR_CUDA;
  }
  return 0;
}

int make_tmap_public(CUtensorMap* map, const __nv_bfloat16* base, int64_t rows, int Kp, int box_rows) {
  return make_tmap(map, base, rows, Kp, box_rows);
}

// ----------------------------------------------------------------------------
// kernel
// ----------------------------------------------------------------------------
constexpr int BM = 128;
#ifndef T4R_HEAD_RESIDENT_DEFAULT
#define T4R_HEAD_RESIDENT_DEFAULT 1  // resident-A head kernel (validated on B200 in round 2; T4R_HEAD_RESIDENT=0 selects the streaming CTA-pair kernel)
#endif
#ifndef T4R_GEMM_2CTA_DEFAULT
#define T4R_GEMM_2CTA_DEFAULT 1
#endif

// One pipeline stage holds 64 bf16 of K: shared-memory operand rows of 128 bytes.
template <int BN>
struct GemmCfg {
  static constexpr int A_PLANE_BYTES = BM * 128;
  static constexpr int B_PLANE_BYTES = BN * 128;
  static constexpr int STAGE_BYTES = 2 * A_PLANE_BYTES + 2 * B_PLANE_BYTES;
  static constexpr int STAGES = (BN == 256) ? 2 : ((BN == 128) ? 3 : 4);
  static constexpr int KSTEPS = 4;   // UMMA K = 16 bf16 = 32 bytes
  static constexpr int TMEM_COLS = 2 * BN;  // two accumulator stages (power of two)
  static constexpr int SMEM_BYTES = STAGES * STAGE_BYTES + 1024 /*align*/ + 256 /*barriers*/ + 4096 /*LN exchange*/ + 8 * 32 * 20 * 4 /*epilogue staging*/;
};

// T4R_GEMM_DEBUG & 2: cycle counters of one epilogue warp (CTA 0, warp 2), see tools/microbench.py
__device__ unsigned long long g_dbg_cycles[8];
// T4R_GEMM_DEBUG & 2 in ffn_fused_kernel: [0..7] one epilogue warp of CTA 0 (wait S, tmem_ld, GELU math, wait G free,
// tmem_st, wait Y, final epilogue, chunks); [8..15] its MMA thread (wait S free, GEMM1 issue incl. TMA waits, wait G,
// wait Y free, GEMM2 issue incl. TMA waits, tiles)
__device__ unsigned long long g_dbg_ffn[16];

struct GemmDev {
  int head_chunk;  // resident-A head kernel: column tiles per unit
  int M;
  int64_t N;
  int nkb;
  int nprod;
  const int32_t* m_dev;
  GemmEpilogue ep;
};

// value of one 32-column chunk: acc + bias -> act -> mask replace (residual is added separately).
// nvalid < 32 only for the last chunk of an N that is not a multiple of 32: those columns read
// nothing and come out as exact zeros (they are the zero padding of the split planes).
__device__ __forceinline__ void dense_chunk(float (&v)[32], const GemmEpilogue& ep, int64_t ncol0, int code,
                                            int nvalid = 32) {
  if (nvalid < 32) {
#pragma unroll
    for (int j = 0; j < 32; ++j) {
      float x = 0.f;
      if (j < nvalid) {
        x = v[j] + (ep.bias ? __ldg(ep.bias + ncol0 + j) : 0.f);
        if (ep.act == T4R_ACT_GELU) x = gelu_erf(x);
        else if (ep.act == T4R_ACT_RELU) x = fmaxf(x, 0.f);
        if (code == 1) x = __ldg(ep.mask_vec + ncol0 + j);
        else if (code == 2) x = 0.f;
      }
      v[j] = x;
    }
    return;
  }
  if (ep.bias) {
    const float4* b4 = reinterpret_cast<const float4*>(ep.bias + ncol0);
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      float4 b = __ldg(b4 + j);
      v[4 * j + 0] += b.x; v[4 * j + 1] += b.y; v[4 * j + 2] += b.z; v[4 * j + 3] += b.w;
    }
  }
  // the activation switch stays OUTSIDE the element loops: a per-element branch splits the
  // unrolled loop into 32 basic blocks and ptxas can no longer interleave the 32 independent
  // chains (measured: 6.5k cycles per 32-element GELU chunk vs ~0.7k after hoisting)
  if (ep.act == T4R_ACT_GELU) {
#pragma unroll
    for (int j = 0; j < 32; ++j) v[j] = gelu_erf(v[j]);
  } else if (ep.act == T4R_ACT_RELU) {
#pragma unroll
    for (int j = 0; j < 32; ++j) v[j] = fmaxf(v[j], 0.f);
  }
  if (code == 1) {
    const float4* m4 = reinterpret_cast<const float4*>(ep.mask_vec + ncol0);
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      float4 b = __ldg(m4 + j);
      v[4 * j + 0] = b.x; v[4 * j + 1] = b.y; v[4 * j + 2] = b.z; v[4 * j + 3] = b.w;
    }
  } else if (code == 2) {
#pragma unroll
    for (int j = 0; j < 32; ++j) v[j] = 0.f;
  }
}

// ---------------------------------------------------------------------------
// Coalesced global access for the epilogue.  After tcgen05.ld a thread holds one
// output ROW (32 consecutive columns); storing that directly makes every warp store
// touch 32 different 128-byte lines with 16 bytes each (measured: the store queue, not
// the tensor pipe, then bounds the dense GEMMs).  Each warp therefore transposes
// 32 rows x 16 columns at a time through a private 32 x 20-word shared-memory tile
// (row stride 20 words: conflict-free row writes) and stores 8 rows x 64 contiguous
// bytes per instruction.  All helpers are warp-collective.
// ---------------------------------------------------------------------------
constexpr int STG_LD = 20;                       // words per staged row
constexpr int STG_WORDS = 32 * STG_LD;           // per warp

// stage: thread-row -> row-segment ownership (registers), no global access
__device__ __forceinline__ void warp_stage_f32(float* stg, const float (&v)[32], float scale, int lane, float4 (&t)[8]) {
#pragma unroll
  for (int h = 0; h < 2; ++h) {
    __syncwarp();
#pragma unroll
    for (int j = 0; j < 4; ++j)
      *reinterpret_cast<float4*>(stg + lane * STG_LD + 4 * j) =
          make_float4(v[h * 16 + 4 * j] * scale, v[h * 16 + 4 * j + 1] * scale, v[h * 16 + 4 * j + 2] * scale,
                      v[h * 16 + 4 * j + 3] * scale);
    __syncwarp();
#pragma unroll
    for (int it = 0; it < 4; ++it) {
      const int r = it * 8 + (lane >> 2), c4 = lane & 3;
      t[h * 4 + it] = *reinterpret_cast<const float4*>(stg + r * STG_LD + 4 * c4);
    }
  }
}
__device__ __forceinline__ void warp_commit_f32(const float4 (&t)[8], float* gbase, int64_t ld, int rows_valid, int lane) {
#pragma unroll
  for (int h = 0; h < 2; ++h)
#pragma unroll
    for (int it = 0; it < 4; ++it) {
      const int r = it * 8 + (lane >> 2), c4 = lane & 3;
      if (r < rows_valid) *reinterpret_cast<float4*>(gbase + r * ld + h * 16 + 4 * c4) = t[h * 4 + it];
    }
}
__device__ __forceinline__ void warp_store_f32(float* stg, const float (&v)[32], float scale, float* gbase, int64_t ld,
                                               int rows_valid, int lane) {
  float4 t[8];
  warp_stage_f32(stg, v, scale, lane, t);
  warp_commit_f32(t, gbase, ld, rows_valid, lane);  // all 8 global stores back to back, after the last warp barrier
}

__device__ __forceinline__ void warp_load_f32(float* stg, const float* gbase, int64_t ld, int rows_valid, int lane,
                                              float (&out)[32]) {
#pragma unroll
  for (int h = 0; h < 2; ++h) {
    __syncwarp();
#pragma unroll
    for (int it = 0; it < 4; ++it) {
      const int r = it * 8 + (lane >> 2), c4 = lane & 3;
      float4 t = make_float4(0.f, 0.f, 0.f, 0.f);
      if (r < rows_valid) t = *reinterpret_cast<const float4*>(gbase + r * ld + h * 16 + 4 * c4);
      *reinterpret_cast<float4*>(stg + r * STG_LD + 4 * c4) = t;
    }
    __syncwarp();
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const float4 t = *reinterpret_cast<const float4*>(stg + lane * STG_LD + 4 * j);
      out[h * 16 + 4 * j] = t.x; out[h * 16 + 4 * j + 1] = t.y; out[h * 16 + 4 * j + 2] = t.z; out[h * 16 + 4 * j + 3] = t.w;
    }
  }
}

// residual kept only as split planes: out[j] = hi[j] + lo[j] (exact to 16 mantissa bits)
__device__ __forceinline__ void warp_load_planes(float* stg_f, const __nv_bfloat16* hi_base, int64_t plane_stride,
                                                 int64_t ld, int rows_valid, int lane, float (&out)[32]) {
  uint32_t* stg = reinterpret_cast<uint32_t*>(stg_f);
#pragma unroll
  for (int pl = 0; pl < 2; ++pl) {
    const __nv_bfloat16* base = hi_base + pl * plane_stride;
    __syncwarp();
#pragma unroll
    for (int it = 0; it < 4; ++it) {
      const int r = it * 8 + (lane >> 2), c = lane & 3;
      uint4 t = make_uint4(0u, 0u, 0u, 0u);
      if (r < rows_valid) t = *reinterpret_cast<const uint4*>(base + r * ld + 8 * c);
      *reinterpret_cast<uint4*>(stg + r * STG_LD + 4 * c) = t;
    }
    __syncwarp();
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const uint4 t = *reinterpret_cast<const uint4*>(stg + lane * STG_LD + 4 * j);
      const uint32_t w[4] = {t.x, t.y, t.z, t.w};
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const float a = __uint_as_float(w[k] << 16), b = __uint_as_float(w[k] & 0xffff0000u);
        if (pl == 0) { out[8 * j + 2 * k] = a; out[8 * j + 2 * k + 1] = b; }
        else { out[8 * j + 2 * k] += a; out[8 * j + 2 * k + 1] += b; }
      }
    }
  }
}

// split v into bf16 hi/lo and store both planes (32 columns = 64 bytes per row and plane)
__device__ __forceinline__ void warp_store_planes(float* stg_f, const float (&v)[32], __nv_bfloat16* hi_base,
                                                  int64_t plane_stride, int64_t ld, int rows_valid, int lane) {
  uint32_t* stg = reinterpret_cast<uint32_t*>(stg_f);
  uint32_t h[16], l[16];
#pragma unroll
  for (int j = 0; j < 16; ++j) split_bf16x2(v[2 * j], v[2 * j + 1], h[j], l[j]);
  uint4 t[8];
#pragma unroll
  for (int pl = 0; pl < 2; ++pl) {
    __syncwarp();
#pragma unroll
    for (int j = 0; j < 4; ++j)
      *reinterpret_cast<uint4*>(stg + lane * STG_LD + 4 * j) =
          pl == 0 ? make_uint4(h[4 * j], h[4 * j + 1], h[4 * j + 2], h[4 * j + 3])
                  : make_uint4(l[4 * j], l[4 * j + 1], l[4 * j + 2], l[4 * j + 3]);
    __syncwarp();
#pragma unroll
    for (int it = 0; it < 4; ++it) {
      const int r = it * 8 + (lane >> 2), c = lane & 3;
      t[pl * 4 + it] = *reinterpret_cast<const uint4*>(stg + r * STG_LD + 4 * c);
    }
  }
  // global stores last, back to back (no warp barrier between them)
#pragma unroll
  for (int pl = 0; pl < 2; ++pl) {
    __nv_bfloat16* base = hi_base + pl * plane_stride;
#pragma unroll
    for (int it = 0; it < 4; ++it) {
      const int r = it * 8 + (lane >> 2), c = lane & 3;
      if (r < rows_valid) *reinterpret_cast<uint4*>(base + r * ld + 8 * c) = t[pl * 4 + it];
    }
  }
}

__device__ __forceinline__ void tmem_st8(uint32_t taddr, const uint32_t (&r)[8]) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"r"(taddr), "r"(r[0]),
               "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7])
               : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// ---------------------------------------------------------------------------
// LayerNorm epilogue, chunked: the half-row is processed 32 columns at a time and parked back in its TMEM columns
// between the two passes (tcgen05.st), instead of living in 128 registers.  That removes the spills of the
// single-pass form and leaves room to issue the coalesced residual loads of chunk c + 1 before chunk c is processed:
// the staged residual read used to expose the global-load latency twice per 32 columns (measured 18-22 k of the
// 35-40 k cycles this epilogue cost per 128 x 256 tile).  Statistics: exact two-pass mean / M2 per 32-column chunk,
// chunks and the two half-rows merged with the pairwise (Chan et al.) update.
// ---------------------------------------------------------------------------
__device__ __forceinline__ void tmem_st32(uint32_t taddr, const float (&v)[32]) {
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    uint32_t r[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) r[j] = __float_as_uint(v[q * 8 + j]);
    tmem_st8(taddr + q * 8, r);
  }
}
// coalesced loads of one 32-row x 32-column residual block into registers (8 rows x 64 B per instruction)
__device__ __forceinline__ void residual_issue(const GemmEpilogue& ep, int64_t row0, int64_t ncol0, int rows_valid, int lane,
                                               uint4 (&raw)[8]) {
#pragma unroll
  for (int it = 0; it < 4; ++it) {
    const int r = it * 8 + (lane >> 2), c = lane & 3;
    const bool ok = r < rows_valid;
    if (ep.residual) {
      const float* g = ep.residual + (row0 + r) * ep.ldr + ncol0 + 4 * c;
      raw[it] = ok ? __ldg(reinterpret_cast<const uint4*>(g)) : make_uint4(0u, 0u, 0u, 0u);
      raw[4 + it] = ok ? __ldg(reinterpret_cast<const uint4*>(g + 16)) : make_uint4(0u, 0u, 0u, 0u);
    } else {
      const __nv_bfloat16* g = ep.residual_planes + (row0 + r) * ep.ldrp + ncol0 + 8 * c;
      raw[it] = ok ? __ldg(reinterpret_cast<const uint4*>(g)) : make_uint4(0u, 0u, 0u, 0u);
      raw[4 + it] = ok ? __ldg(reinterpret_cast<const uint4*>(g + ep.residual_plane_stride)) : make_uint4(0u, 0u, 0u, 0u);
    }
  }
}
// transpose the block through the warp's staging tile and add it to the thread's row
__device__ __forceinline__ void residual_add(const GemmEpilogue& ep, float* stg_f, const uint4 (&raw)[8], int lane,
                                             float (&v)[32]) {
  uint32_t* stg = reinterpret_cast<uint32_t*>(stg_f);
#pragma unroll
  for (int h = 0; h < 2; ++h) {
    __syncwarp();
#pragma unroll
    for (int it = 0; it < 4; ++it) {
      const int r = it * 8 + (lane >> 2), c = lane & 3;
      *reinterpret_cast<uint4*>(stg + r * STG_LD + 4 * c) = raw[h * 4 + it];
    }
    __syncwarp();
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const uint4 t = *reinterpret_cast<const uint4*>(stg + lane * STG_LD + 4 * j);
      const uint32_t w[4] = {t.x, t.y, t.z, t.w};
      if (ep.residual) {  // fp32: half h holds columns [16 h, 16 h + 16)
#pragma unroll
        for (int k = 0; k < 4; ++k) v[h * 16 + 4 * j + k] += __uint_as_float(w[k]);
      } else {            // planes: half 0 = hi, half 1 = lo, eight bf16 per 16 bytes
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          v[8 * j + 2 * k] += __uint_as_float(w[k] << 16);
          v[8 * j + 2 * k + 1] += __uint_as_float(w[k] & 0xffff0000u);
        }
      }
    }
  }
}

// A tile's row is split into two column groups (warps 2-5 and 6-9).  xch_grp0 = this row's slot in group 0 of the
// exchange area [2][128]; grp = own group.
template <int BN>
__device__ __forceinline__ void epilogue_ln_chunked(const GemmDev& p, uint32_t taddr, int64_t row0, int rows_valid, int lane,
                                                    int64_t n0, float* stg, float2* xch_grp0, int grp) {
  constexpr int COLS = BN / 2, NCH = COLS / 32;
  const GemmEpilogue& ep = p.ep;
  if (ep.debug & 1) rows_valid = 0;
  const bool row_ok = lane < rows_valid;
  const int64_t row = row0 + lane;
  int code = 0;
  if (row_ok && ep.row_code) code = ep.row_code[row];
  const bool has_res = ep.residual || ep.residual_planes;
  const bool lprof = (ep.debug & 2) && blockIdx.x == 0 && threadIdx.x == 64;
  const long long l0 = lprof ? clock64() : 0;
  // ---- pass 1: bias (+act, mask) + residual, statistics, park the pre-LN values in TMEM
  uint4 nxt[8];
  if (has_res) residual_issue(ep, row0, n0, rows_valid, lane, nxt);
  float mean_h = 0.f, m2_h = 0.f;
#pragma unroll
  for (int c = 0; c < NCH; ++c) {
    uint4 cur[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) cur[j] = nxt[j];
    if (has_res && c + 1 < NCH) residual_issue(ep, row0, n0 + (c + 1) * 32, rows_valid, lane, nxt);
    float v[32];
    tmem_ld<32>(taddr + c * 32, v);
    dense_chunk(v, ep, n0 + c * 32, code);
    if (has_res) residual_add(ep, stg, cur, lane, v);
    float s = 0.f;
#pragma unroll
    for (int j = 0; j < 32; ++j) s += v[j];
    const float mc = s * (1.f / 32.f);
    float q = 0.f;
#pragma unroll
    for (int j = 0; j < 32; ++j) {
      const float d = v[j] - mc;
      q = fmaf(d, d, q);
    }
    // merge chunk c (32 values) into the running (mean, M2) of 32 c values
    const float delta = mc - mean_h;
    mean_h += delta * (1.f / static_cast<float>(c + 1));
    m2_h += q + delta * delta * (32.f * static_cast<float>(c) / static_cast<float>(c + 1));
    tmem_st32(taddr + c * 32, v);
  }
  tmem_st_wait();
  const long long l1 = lprof ? clock64() : 0;
  // ---- combine the two groups of the row (equal counts)
  xch_grp0[grp * 128] = make_float2(mean_h, m2_h);
  asm volatile("bar.sync 1, %0;" ::"n"(2 * 128) : "memory");
  const float2 o = xch_grp0[(grp ^ 1) * 128];
  const float delta = o.x - mean_h;
  const float mean = 0.5f * (mean_h + o.x);
  const float m2 = m2_h + o.y + delta * delta * (0.5f * COLS);
  const float rstd = rsqrtf(m2 * (1.f / BN) + ep.ln_eps);
  const long long l2 = lprof ? clock64() : 0;
  // ---- pass 2: normalise and store
#pragma unroll
  for (int c = 0; c < NCH; ++c) {
    float v[32];
    tmem_ld<32>(taddr + c * 32, v);
    const int64_t ncol0 = n0 + c * 32;
    if (ep.out_pre) warp_store_f32(stg, v, 1.f, ep.out_pre + row0 * ep.ldp + ncol0, ep.ldp, rows_valid, lane);
    const float4* g4 = reinterpret_cast<const float4*>(ep.ln_gamma + ncol0);
    const float4* b4 = reinterpret_cast<const float4*>(ep.ln_beta + ncol0);
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const float4 g = __ldg(g4 + j), b = __ldg(b4 + j);
      v[4 * j + 0] = (v[4 * j + 0] - mean) * rstd * g.x + b.x;
      v[4 * j + 1] = (v[4 * j + 1] - mean) * rstd * g.y + b.y;
      v[4 * j + 2] = (v[4 * j + 2] - mean) * rstd * g.z + b.z;
      v[4 * j + 3] = (v[4 * j + 3] - mean) * rstd * g.w + b.w;
    }
    if (ep.out_f32) warp_store_f32(stg, v, ep.out_scale, ep.out_f32 + row0 * ep.ldo + ncol0, ep.ldo, rows_valid, lane);
    if (ep.out_planes)
      warp_store_planes(stg, v, ep.out_planes + row0 * ep.ldpl + ncol0, ep.plane_stride, ep.ldpl, rows_valid, lane);
  }
  if (lprof) {  // phases: pass 1 (bias + residual + stats + park) | exchange | pass 2 (normalise + stores)
    g_dbg_cycles[2] += 0; g_dbg_cycles[3] += l1 - l0; g_dbg_cycles[4] += l2 - l1; g_dbg_cycles[5] += clock64() - l2;
  }
}

// Each epilogue thread owns one output row (its TMEM lane) and COLS = BN/2 columns
// (warps 2-5 take the first half of the tile's columns, warps 6-9 the second half).
// row0 = first row of the warp's 32-row block; n0 = first column of the warp's half.
template <int BN, bool LN>
__device__ __forceinline__ void epilogue_dense(const GemmDev& p, uint32_t taddr, int64_t row0, int rows_valid, int lane,
                                               int64_t n0, float* stg, float2* xch_grp0, int grp) {
  constexpr int COLS = BN / 2;
  const GemmEpilogue& ep = p.ep;
  if (ep.debug & 1) rows_valid = 0;  // timing experiment: no global traffic from the epilogue
  const bool row_ok = lane < rows_valid;
  const int64_t row = row0 + lane;
  int code = 0;
  if (row_ok && ep.row_code) code = ep.row_code[row];
  if constexpr (LN) {
    epilogue_ln_chunked<BN>(p, taddr, row0, rows_valid, lane, n0, stg, xch_grp0, grp);
  } else {
    const bool prof = (ep.debug & 2) && blockIdx.x == 0 && threadIdx.x == 64;
#pragma unroll 1
    for (int c = 0; c < COLS / 32; ++c) {
      float v[32];
      long long t0 = prof ? clock64() : 0;
      tmem_ld<32>(taddr + c * 32, v);
      long long t1 = prof ? clock64() : 0;
      const int64_t ncol0 = n0 + c * 32;
      const int64_t n_pad = (p.N + 63) / 64 * 64;  // planes are zero padded to a multiple of 64 columns
      if (ncol0 >= n_pad) continue;                // warp-uniform
      const int nvalid = (p.N - ncol0 >= 32) ? 32 : (p.N > ncol0 ? static_cast<int>(p.N - ncol0) : 0);
      if (ep.col_scale) {  // 2-unit product: undo the power-of-two row scales of both operands (exact)
        const float rs = row_ok ? ep.row_scale[row] : 1.f;
#pragma unroll
        for (int j = 0; j < 32; ++j)
          if (j < nvalid) v[j] *= rs * __ldg(ep.col_scale + ncol0 + j);
      }
      dense_chunk(v, ep, ncol0, code, nvalid);
      long long t2 = prof ? clock64() : 0;
      if (prof) { g_dbg_cycles[2] += t1 - t0; g_dbg_cycles[3] += t2 - t1; }
      if (ep.residual || ep.residual_planes) {
        float rs[32];
        if (ep.residual) warp_load_f32(stg, ep.residual + row0 * ep.ldr + ncol0, ep.ldr, rows_valid, lane, rs);
        else warp_load_planes(stg, ep.residual_planes + row0 * ep.ldrp + ncol0, ep.residual_plane_stride, ep.ldrp,
                              rows_valid, lane, rs);
#pragma unroll
        for (int j = 0; j < 32; ++j) v[j] += rs[j];
      }
      if (ep.out_f32 && nvalid > 0) {
        if ((ep.ldo & 3) == 0 && nvalid == 32) {
          warp_store_f32(stg, v, ep.out_scale, ep.out_f32 + row0 * ep.ldo + ncol0, ep.ldo, rows_valid, lane);
        } else if (row_ok) {
          float* dst = ep.out_f32 + row * ep.ldo + ncol0;
#pragma unroll
          for (int j = 0; j < 32; ++j)
            if (ncol0 + j < p.N) dst[j] = v[j] * ep.out_scale;
        }
      }
      long long t3 = prof ? clock64() : 0;
      if (ep.out_planes)
        warp_store_planes(stg, v, ep.out_planes + row0 * ep.ldpl + ncol0, ep.plane_stride, ep.ldpl, rows_valid, lane);
      if (prof) { long long t4 = clock64(); g_dbg_cycles[4] += t3 - t2; g_dbg_cycles[5] += t4 - t3; }
    }
  }
}

// head epilogue: per row, online log-sum-exp (base 2) over this thread's COLS classes
// of the tile, optional logQ bias / accidental-hit removal (sampled softmax), rank count.
template <int BN>
__device__ __forceinline__ void epilogue_head(const GemmDev& p, uint32_t taddr, int64_t row, bool row_ok, int64_t n0,
                                              int part_idx) {
  constexpr int COLS = BN / 2;
  const GemmEpilogue& ep = p.ep;
  constexpr float kLog2e = 1.4426950408889634f;
  const float scale2 = ep.inv_tau * kLog2e;
  float m_run = -INFINITY, s_run = 0.f, z_run = 0.f;
  const bool want_z = (ep.part_z != nullptr);
  int cnt = 0;
  int64_t label = -1;
  float tgt = 0.f;
  const bool want_rank = (ep.row_rank != nullptr);
  if (row_ok && ep.row_label) label = ep.row_label[row];
  if (row_ok && want_rank) tgt = ep.row_tgt[row];
  const int hit_c = (row_ok && ep.hit_col) ? ep.hit_col[row] : -1;
  const float row_scale = (row_ok && ep.row_scale) ? ep.row_scale[row] : 1.f;
  const bool full_tile = (n0 + COLS <= p.N);
#pragma unroll 1
  for (int c = 0; c < COLS / 32; ++c) {
    float v[32];
    tmem_ld<32>(taddr + c * 32, v);
    if (!row_ok) continue;
    const int64_t ncol0 = n0 + c * 32;
    if (ncol0 >= p.N) continue;
    if (ep.debug & 32) { m_run = fmaxf(m_run, v[c]); continue; }  // timing experiment: TMEM reads only
    if (ep.col_scale) {  // 2-unit product: undo the power-of-two row scales of both operands (exact)
      if (full_tile) {
        const float4* c4 = reinterpret_cast<const float4*>(ep.col_scale + ncol0);
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const float4 cs = __ldg(c4 + j);
          v[4 * j + 0] *= row_scale * cs.x; v[4 * j + 1] *= row_scale * cs.y;
          v[4 * j + 2] *= row_scale * cs.z; v[4 * j + 3] *= row_scale * cs.w;
        }
      } else {
#pragma unroll
        for (int j = 0; j < 32; ++j)
          if (ncol0 + j < p.N) v[j] *= row_scale * __ldg(ep.col_scale + ncol0 + j);
      }
    }
    if (ep.col_bias) {
      if (full_tile && (ncol0 & 3) == 0) {
        const float4* b4 = reinterpret_cast<const float4*>(ep.col_bias + ncol0);
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const float4 b = __ldg(b4 + j);
          v[4 * j + 0] += b.x; v[4 * j + 1] += b.y; v[4 * j + 2] += b.z; v[4 * j + 3] += b.w;
        }
      } else {
#pragma unroll
        for (int j = 0; j < 32; ++j)
          if (full_tile || ncol0 + j < p.N) v[j] += __ldg(ep.col_bias + ncol0 + j);
      }
    }
    if (ep.hit_col) {           // the row's accidental hit, found once per row (launch_hit_cols)
      const int64_t rel = static_cast<int64_t>(hit_c) - ncol0;
      if (rel >= 0 && rel < 32) {
#pragma unroll
        for (int j = 0; j < 32; ++j)
          if (j == rel) v[j] = ep.hit_value;
      }
    } else if (ep.col_ids) {
#pragma unroll
      for (int j = 0; j < 32; ++j)
        if ((full_tile || ncol0 + j < p.N) && __ldg(ep.col_ids + ncol0 + j) == label) v[j] = ep.hit_value;
    }
    if (!full_tile) {
#pragma unroll
      for (int j = 0; j < 32; ++j)
        if (ncol0 + j >= p.N) v[j] = -INFINITY;
    }
    if (want_rank) {
      // classes scoring above the label; ties resolved "lower id first" like a stable top-k
      const int64_t lab_col = label - ep.col_offset;
#pragma unroll
      for (int j = 0; j < 32; ++j) {
        const float x = v[j] * ep.inv_tau;
        const int64_t col = ncol0 + j;
        cnt += (col != lab_col) && ((x > tgt) || (x == tgt && col < lab_col));
      }
    }
    if (want_z) {
      // label smoothing needs sum_j z_j; masked columns are -inf and must not enter the sum
      float zs = 0.f;
#pragma unroll
      for (int j = 0; j < 32; ++j) zs += (v[j] == -INFINITY) ? 0.f : v[j];
      z_run = fmaf(zs, ep.inv_tau, z_run);
    }
    // four independent chains each for the max and the sum: with two epilogue warps per scheduler a single
    // 32-long dependent FMNMX / FADD chain (4 cycles per link) left this loop latency-bound at ~5k cycles per
    // 128x256 tile, 2.4x its SFU (ex2) floor
    float mx[4] = {v[0], v[1], v[2], v[3]};
#pragma unroll
    for (int j = 4; j < 32; j += 4) {
      mx[0] = fmaxf(mx[0], v[j]); mx[1] = fmaxf(mx[1], v[j + 1]);
      mx[2] = fmaxf(mx[2], v[j + 2]); mx[3] = fmaxf(mx[3], v[j + 3]);
    }
    const float cmax = fmaxf(fmaxf(mx[0], mx[1]), fmaxf(mx[2], mx[3])) * scale2;  // scale2 > 0
    const float m_new = fmaxf(m_run, cmax);
    if (ep.debug & 16) { m_run = m_new; continue; }  // timing experiment: no exponentials
    if (m_new > -INFINITY) {
      float acc[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
      for (int j = 0; j < 32; j += 4) {
        acc[0] += fast_exp2(fmaf(v[j], scale2, -m_new));
        acc[1] += fast_exp2(fmaf(v[j + 1], scale2, -m_new));
        acc[2] += fast_exp2(fmaf(v[j + 2], scale2, -m_new));
        acc[3] += fast_exp2(fmaf(v[j + 3], scale2, -m_new));
      }
      s_run = s_run * fast_exp2(m_run - m_new) + ((acc[0] + acc[1]) + (acc[2] + acc[3]));
      m_run = m_new;
    }
  }
  if (row_ok) {
    ep.part_m[static_cast<int64_t>(part_idx) * ep.part_ld + row] = m_run;
    ep.part_s[static_cast<int64_t>(part_idx) * ep.part_ld + row] = s_run;
    if (want_z) ep.part_z[static_cast<int64_t>(part_idx) * ep.part_ld + row] = z_run;
    if (want_rank && cnt) atomicAdd(ep.row_rank + row, cnt);
  }
}

template <int BN, bool LN, bool HEAD>
__global__ void __launch_bounds__(320, 1)
gemm_bf16x3_kernel(const __grid_constant__ CUtensorMap tmAh, const __grid_constant__ CUtensorMap tmAl,
                   const __grid_constant__ CUtensorMap tmBh, const __grid_constant__ CUtensorMap tmBl,
                   const GemmDev p) {
  using Cfg = GemmCfg<BN>;
  constexpr int A_PLANE_BYTES = Cfg::A_PLANE_BYTES;
  extern __shared__ uint8_t smem_raw[];
  // 1024-byte alignment for the 128B-swizzled tiles, done with pointer arithmetic on the
  // __shared__ array so the compiler keeps the shared address space (LDS/STS, not generic LD/ST)
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + Cfg::STAGES * Cfg::STAGE_BYTES);
  uint64_t* empty_bar = full_bar + Cfg::STAGES;
  uint64_t* tfull_bar = empty_bar + Cfg::STAGES;
  uint64_t* tempty_bar = tfull_bar + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty_bar + 2);
  float2* xch = reinterpret_cast<float2*>(smem + Cfg::STAGES * Cfg::STAGE_BYTES + 256);  // [2 parity][2 half][128]
  float* stg_all = reinterpret_cast<float*>(smem + Cfg::STAGES * Cfg::STAGE_BYTES + 256 + 4096);  // [8 warps][32][20]

  const int warp = warp_id();
  const int lane = lane_id();

  int M_eff = p.M;
  if (p.m_dev) M_eff = min(p.M, *p.m_dev);
  const int tiles_m = (M_eff + BM - 1) / BM;
  const int tiles_n = static_cast<int>((p.N + BN - 1) / BN);
  const int64_t num_tiles = static_cast<int64_t>(tiles_m) * tiles_n;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmAh);
    tma_prefetch_desc(&tmAl);
    tma_prefetch_desc(&tmBh);
    tma_prefetch_desc(&tmBl);
  }
  if (warp == 1 && lane == 0) {
    for (int i = 0; i < Cfg::STAGES; ++i) {
      mbar_init(&full_bar[i], 1);
      mbar_init(&empty_bar[i], 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&tfull_bar[i], 1);
      mbar_init(&tempty_bar[i], 8);
    }
    fence_barrier_init();
  }
  if (warp == 2) {
    tmem_alloc(tmem_slot, Cfg::TMEM_COLS);
    tmem_relinquish();
  }
  tc_fence_before_sync();
  __syncthreads();
  tc_fence_after_sync();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // ===================== TMA producer =====================
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      const uint32_t bytes = (p.nprod != 1) ? Cfg::STAGE_BYTES : (A_PLANE_BYTES + Cfg::B_PLANE_BYTES);
      for (int64_t tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
        const int m0 = static_cast<int>(tile % tiles_m) * BM;
        const int n0 = static_cast<int>(tile / tiles_m) * BN;
        for (int kb = 0; kb < p.nkb; ++kb) {
          mbar_wait(&empty_bar[stage], phase ^ 1);
          uint8_t* st = smem + stage * Cfg::STAGE_BYTES;
          mbar_arrive_expect_tx(&full_bar[stage], bytes);
          tma_load_2d(st, &tmAh, &full_bar[stage], kb * 64, m0);
          tma_load_2d(st + 2 * A_PLANE_BYTES, &tmBh, &full_bar[stage], kb * 64, n0);
          if (p.nprod != 1) {
            tma_load_2d(st + A_PLANE_BYTES, &tmAl, &full_bar[stage], kb * 64, m0);
            tma_load_2d(st + 2 * A_PLANE_BYTES + Cfg::B_PLANE_BYTES, &tmBl, &full_bar[stage], kb * 64, n0);
          }
          if (++stage == Cfg::STAGES) { stage = 0; phase ^= 1; }
        }
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    // ===================== MMA issuer =====================
    if (lane == 0) {
      constexpr uint32_t idesc = umma_idesc_bf16(BM, BN);
      int stage = 0;
      uint32_t phase = 0;
      int as = 0;
      uint32_t aph = 0;
      for (int64_t tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
        mbar_wait(&tempty_bar[as], aph ^ 1);
        tc_fence_after_sync();
        const uint32_t d_tmem = tmem_base + static_cast<uint32_t>(as * BN);
        for (int kb = 0; kb < p.nkb; ++kb) {
          mbar_wait(&full_bar[stage], phase);
          tc_fence_after_sync();
          const uint32_t a_hi = smem_u32(smem + stage * Cfg::STAGE_BYTES);
          const uint32_t a_lo = a_hi + A_PLANE_BYTES;
          const uint32_t b_hi = a_hi + 2 * A_PLANE_BYTES;
          const uint32_t b_lo = b_hi + Cfg::B_PLANE_BYTES;
          if (p.nprod == 2) {
            // 2-unit product (t4r_mixed_pack.cuh): plane 0 = fp16, plane 1 = [64 x hi8 | 64 x lo8] e4m3 per row.
            // Four K = 16 fp16 MMAs, then lo8(A) x hi8(B) and hi8(A) x lo8(B) as two K = 32 e4m3 MMAs each,
            // all into the same fp32 accumulator.
            constexpr uint32_t idesc_h = umma_idesc_f16(BM, BN);
            constexpr uint32_t idesc_8 = umma_idesc_e4m3(BM, BN);
            // bring-up switches (T4R_GEMM_DEBUG): 64 / 128 / 256 drop the main / first / second cross product
            const int dbg = p.ep.debug;
            uint32_t acc = (kb != 0) ? 1u : 0u;
            if (!(dbg & 64)) {
#pragma unroll
              for (int k4 = 0; k4 < 4; ++k4) {
                umma_bf16(d_tmem, umma_desc_sw128(a_hi + k4 * 32), umma_desc_sw128(b_hi + k4 * 32), idesc_h, acc);
                acc = 1u;
              }
            }
#pragma unroll
            for (int j = 0; j < 2; ++j) {
              if (!(dbg & 128)) { umma_f8(d_tmem, umma_desc_sw128(a_lo + 64 + j * 32), umma_desc_sw128(b_lo + j * 32), idesc_8, acc); acc = 1u; }
              if (!(dbg & 256)) { umma_f8(d_tmem, umma_desc_sw128(a_lo + j * 32), umma_desc_sw128(b_lo + 64 + j * 32), idesc_8, acc); acc = 1u; }
            }
          } else {
#pragma unroll
          for (int k4 = 0; k4 < Cfg::KSTEPS; ++k4) {
            const uint64_t da_hi = umma_desc_sw128(a_hi + k4 * 32);
            const uint64_t db_hi = umma_desc_sw128(b_hi + k4 * 32);
            if (p.nprod == 3) {
              const uint64_t da_lo = umma_desc_sw128(a_lo + k4 * 32);
              const uint64_t db_lo = umma_desc_sw128(b_lo + k4 * 32);
              umma_bf16(d_tmem, da_lo, db_hi, idesc, (kb | k4) != 0);
              umma_bf16(d_tmem, da_hi, db_lo, idesc, 1u);
              umma_bf16(d_tmem, da_hi, db_hi, idesc, 1u);
            } else {
              umma_bf16(d_tmem, da_hi, db_hi, idesc, (kb | k4) != 0);
            }
          }
          }
          umma_commit(&empty_bar[stage]);  // smem slot free once these MMAs retire
          if (++stage == Cfg::STAGES) { stage = 0; phase ^= 1; }
        }
        umma_commit(&tfull_bar[as]);  // accumulator ready for the epilogue
        as ^= 1;
        if (as == 0) aph ^= 1;
      }
    }
    __syncwarp();
  } else {
    // ===================== epilogue warps (2..9) =====================
    const int quad = warp & 3;          // TMEM lane quadrant this warp may access
    const int half = (warp - 2) >> 2;   // which half of the tile's columns
    constexpr int COLS = BN / 2;
    int as = 0;
    uint32_t aph = 0;
    uint32_t tile_parity = 0;
    for (int64_t tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
      const int tile_n = static_cast<int>(tile / tiles_m);
      const int64_t m0 = static_cast<int64_t>(tile % tiles_m) * BM;
      const int64_t n0 = static_cast<int64_t>(tile_n) * BN + half * COLS;
      const bool prof = (p.ep.debug & 2) && blockIdx.x == 0 && threadIdx.x == 64;
      const long long tw0 = prof ? clock64() : 0;
      mbar_wait(&tfull_bar[as], aph);
      tc_fence_after_sync();
      const long long tw1 = prof ? clock64() : 0;
      const uint32_t taddr = tmem_base + (static_cast<uint32_t>(quad * 32) << 16) +
                             static_cast<uint32_t>(as * BN + half * COLS);
      const int64_t row0 = m0 + quad * 32;
      const int64_t row = row0 + lane;
      const bool row_ok = row < M_eff;
      if (HEAD) {
        epilogue_head<BN>(p, taddr, row, row_ok, n0, tile_n * 2 + half);
      } else {
        float2* xg0 = xch + (tile_parity * 2) * 128 + quad * 32 + lane;   // [parity][group][row]
        const int64_t left = static_cast<int64_t>(M_eff) - row0;
        const int rows_valid = left < 0 ? 0 : (left > 32 ? 32 : static_cast<int>(left));
        epilogue_dense<BN, LN>(p, taddr, row0, rows_valid, lane, n0, stg_all + (warp - 2) * STG_WORDS, xg0, half);
      }
      if (prof) { g_dbg_cycles[0] += tw1 - tw0; g_dbg_cycles[1] += clock64() - tw1; g_dbg_cycles[6] += 1; }
      tile_parity ^= 1;
      tc_fence_before_sync();
      __syncwarp();
      if (lane == 0) mbar_arrive(&tempty_bar[as]);
      as ^= 1;
      if (as == 0) aph ^= 1;
    }
  }

  tc_fence_before_sync();
  __syncthreads();
  tc_fence_after_sync();
  if (warp == 2) tmem_dealloc(tmem_base, Cfg::TMEM_COLS);
}


// ============================================================================
// CTA-pair variant (tcgen05 cta_group::2): two SMs of a TPC share one 256 x BN tile.  Each CTA loads its own 128
// rows of A and HALF of the B tile (BN/2 rows), so per SM the L2->SM operand stream and the shared-memory operand
// reads of the tensor core drop by a third (BN = 256) -- the bound of every GEMM on this path except the K = 256 head
// (DESIGN.md section 5).  Protocol (leader = cluster rank 0):
//   * both TMA warps wait on their OWN empty[s]; the leader arms full[s] with the bytes of both CTAs and all eight
//     loads credit the leader's full[s];
//   * the leader's MMA warp issues M = 256 MMAs and commits with a 2-CTA multicast: empty[s] and tfull[as] fire in both;
//   * the 16 epilogue warps of both CTAs read their own TMEM and arrive on the LEADER's tempty[as].
// ============================================================================
template <int BN>
struct Gemm2Cfg {
  static constexpr int A_PLANE_BYTES = BM * 128;
  static constexpr int B_PLANE_BYTES = (BN / 2) * 128;  // this CTA's half of the B tile
  static constexpr int STAGE_BYTES = 2 * A_PLANE_BYTES + 2 * B_PLANE_BYTES;
  static constexpr int STAGES = (BN == 256) ? 3 : 4;
  static constexpr int TMEM_COLS = 2 * BN;
  static constexpr int SMEM_BYTES = STAGES * STAGE_BYTES + 1024 + 256 + 4096 + 8 * 32 * 20 * 4;
};

template <int BN, bool LN, bool HEAD>
__global__ void __launch_bounds__(320, 1)
gemm2_bf16x3_kernel(const __grid_constant__ CUtensorMap tmAh, const __grid_constant__ CUtensorMap tmAl,
                    const __grid_constant__ CUtensorMap tmBh, const __grid_constant__ CUtensorMap tmBl,
                    const GemmDev p) {
  using Cfg = Gemm2Cfg<BN>;
  constexpr int A_PLANE_BYTES = Cfg::A_PLANE_BYTES;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + Cfg::STAGES * Cfg::STAGE_BYTES);
  uint64_t* empty_bar = full_bar + Cfg::STAGES;
  uint64_t* tfull_bar = empty_bar + Cfg::STAGES;
  uint64_t* tempty_bar = tfull_bar + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty_bar + 2);
  float2* xch = reinterpret_cast<float2*>(smem + Cfg::STAGES * Cfg::STAGE_BYTES + 256);
  float* stg_all = reinterpret_cast<float*>(smem + Cfg::STAGES * Cfg::STAGE_BYTES + 256 + 4096);

  const int warp = warp_id();
  const int lane = lane_id();
  const int rank = static_cast<int>(cluster_ctarank());
  const bool leader = (rank == 0);
  const int pair = blockIdx.x >> 1;
  const int npairs = gridDim.x >> 1;

  int M_eff = p.M;
  if (p.m_dev) M_eff = min(p.M, *p.m_dev);
  const int tiles_m = (M_eff + 2 * BM - 1) / (2 * BM);
  const int tiles_n = static_cast<int>((p.N + BN - 1) / BN);
  const int64_t num_tiles = static_cast<int64_t>(tiles_m) * tiles_n;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmAh); tma_prefetch_desc(&tmAl); tma_prefetch_desc(&tmBh); tma_prefetch_desc(&tmBl);
  }
  if (warp == 1 && lane == 0) {
    for (int i = 0; i < Cfg::STAGES; ++i) {
      mbar_init(&full_bar[i], 1);
      mbar_init(&empty_bar[i], 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&tfull_bar[i], 1);
      mbar_init(&tempty_bar[i], 16);  // 8 epilogue warps of each CTA (only the leader's copy is used)
    }
    fence_barrier_init();
  }
  if (warp == 2) {
    tmem_alloc_pair(tmem_slot, Cfg::TMEM_COLS);
    tmem_relinquish_pair();
  }
  tc_fence_before_sync();
  __syncthreads();
  cluster_sync_all();  // both CTAs' barriers are initialised before any remote arrive / TMA credit
  tc_fence_after_sync();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // ===================== TMA producer (both CTAs) =====================
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      const uint32_t bytes = (p.nprod != 1) ? Cfg::STAGE_BYTES : (A_PLANE_BYTES + Cfg::B_PLANE_BYTES);
      for (int64_t tile = pair; tile < num_tiles; tile += npairs) {
        const int m0 = static_cast<int>(tile % tiles_m) * (2 * BM) + rank * BM;
        const int n0 = static_cast<int>(tile / tiles_m) * BN + rank * (BN / 2);
        for (int kb = 0; kb < p.nkb; ++kb) {
          mbar_wait(&empty_bar[stage], phase ^ 1);
          uint8_t* st = smem + stage * Cfg::STAGE_BYTES;
          if (leader) mbar_arrive_expect_tx(&full_bar[stage], 2 * bytes);
          tma_load_2d_pair(st, &tmAh, &full_bar[stage], kb * 64, m0);
          tma_load_2d_pair(st + 2 * A_PLANE_BYTES, &tmBh, &full_bar[stage], kb * 64, n0);
          if (p.nprod != 1) {
            tma_load_2d_pair(st + A_PLANE_BYTES, &tmAl, &full_bar[stage], kb * 64, m0);
            tma_load_2d_pair(st + 2 * A_PLANE_BYTES + Cfg::B_PLANE_BYTES, &tmBl, &full_bar[stage], kb * 64, n0);
          }
          if (++stage == Cfg::STAGES) { stage = 0; phase ^= 1; }
        }
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    // ===================== MMA issuer (leader only) =====================
    if (leader && lane == 0) {
      constexpr uint32_t idesc = umma_idesc_bf16(2 * BM, BN);
      int stage = 0;
      uint32_t phase = 0;
      int as = 0;
      uint32_t aph = 0;
      for (int64_t tile = pair; tile < num_tiles; tile += npairs) {
        mbar_wait(&tempty_bar[as], aph ^ 1);
        tc_fence_after_sync();
        const uint32_t d_tmem = tmem_base + static_cast<uint32_t>(as * BN);
        for (int kb = 0; kb < p.nkb; ++kb) {
          mbar_wait(&full_bar[stage], phase);
          tc_fence_after_sync();
          const uint32_t a_hi = smem_u32(smem + stage * Cfg::STAGE_BYTES);
          const uint32_t a_lo = a_hi + A_PLANE_BYTES;
          const uint32_t b_hi = a_hi + 2 * A_PLANE_BYTES;
          const uint32_t b_lo = b_hi + Cfg::B_PLANE_BYTES;
          if (p.nprod == 2) {  // 2-unit product: see the single-CTA kernel
            constexpr uint32_t idesc_h = umma_idesc_f16(2 * BM, BN);
            constexpr uint32_t idesc_8 = umma_idesc_e4m3(2 * BM, BN);
            const int dbg = p.ep.debug;  // bring-up switches: 64 / 128 / 256 drop the main / first / second cross product
            uint32_t acc = (kb != 0) ? 1u : 0u;
            if (!(dbg & 64)) {
#pragma unroll
              for (int k4 = 0; k4 < 4; ++k4) {
                umma_bf16_pair(d_tmem, umma_desc_sw128(a_hi + k4 * 32), umma_desc_sw128(b_hi + k4 * 32), idesc_h, acc);
                acc = 1u;
              }
            }
#pragma unroll
            for (int j = 0; j < 2; ++j) {
              if (!(dbg & 128)) { umma_f8_pair(d_tmem, umma_desc_sw128(a_lo + 64 + j * 32), umma_desc_sw128(b_lo + j * 32), idesc_8, acc); acc = 1u; }
              if (!(dbg & 256)) { umma_f8_pair(d_tmem, umma_desc_sw128(a_lo + j * 32), umma_desc_sw128(b_lo + 64 + j * 32), idesc_8, acc); acc = 1u; }
            }
          } else {
#pragma unroll
          for (int k4 = 0; k4 < 4; ++k4) {
            const uint64_t da_hi = umma_desc_sw128(a_hi + k4 * 32);
            const uint64_t db_hi = umma_desc_sw128(b_hi + k4 * 32);
            if (p.nprod == 3) {
              const uint64_t da_lo = umma_desc_sw128(a_lo + k4 * 32);
              const uint64_t db_lo = umma_desc_sw128(b_lo + k4 * 32);
              umma_bf16_pair(d_tmem, da_lo, db_hi, idesc, (kb | k4) != 0);
              umma_bf16_pair(d_tmem, da_hi, db_lo, idesc, 1u);
              umma_bf16_pair(d_tmem, da_hi, db_hi, idesc, 1u);
            } else {
              umma_bf16_pair(d_tmem, da_hi, db_hi, idesc, (kb | k4) != 0);
            }
          }
          }
          umma_commit_pair(&empty_bar[stage]);  // the stage is free in BOTH CTAs once these MMAs retire
          if (++stage == Cfg::STAGES) { stage = 0; phase ^= 1; }
        }
        umma_commit_pair(&tfull_bar[as]);  // both CTAs' halves of the accumulator are ready
        as ^= 1;
        if (as == 0) aph ^= 1;
      }
    }
    __syncwarp();
  } else {
    // ===================== epilogue warps (2..9) of both CTAs =====================
    const int quad = warp & 3;
    const int half = (warp - 2) >> 2;
    constexpr int COLS = BN / 2;
    int as = 0;
    uint32_t aph = 0;
    uint32_t tile_parity = 0;
    for (int64_t tile = pair; tile < num_tiles; tile += npairs) {
      const int tile_n = static_cast<int>(tile / tiles_m);
      const int64_t m0 = static_cast<int64_t>(tile % tiles_m) * (2 * BM) + rank * BM;
      const int64_t n0 = static_cast<int64_t>(tile_n) * BN + half * COLS;
      mbar_wait(&tfull_bar[as], aph);
      tc_fence_after_sync();
      const uint32_t taddr = tmem_base + (static_cast<uint32_t>(quad * 32) << 16) +
                             static_cast<uint32_t>(as * BN + half * COLS);
      const int64_t row0 = m0 + quad * 32;
      const int64_t row = row0 + lane;
      const bool row_ok = row < M_eff;
      if (HEAD) {
        epilogue_head<BN>(p, taddr, row, row_ok, n0, tile_n * 2 + half);
      } else {
        float2* xg0 = xch + (tile_parity * 2) * 128 + quad * 32 + lane;   // [parity][group][row]
        const int64_t left = static_cast<int64_t>(M_eff) - row0;
        const int rows_valid = left < 0 ? 0 : (left > 32 ? 32 : static_cast<int>(left));
        epilogue_dense<BN, LN>(p, taddr, row0, rows_valid, lane, n0, stg_all + (warp - 2) * STG_WORDS, xg0, half);
      }
      tile_parity ^= 1;
      tc_fence_before_sync();
      __syncwarp();
      if (lane == 0) mbar_arrive_leader(&tempty_bar[as]);
      as ^= 1;
      if (as == 0) aph ^= 1;
    }
  }

  tc_fence_before_sync();
  __syncthreads();
  cluster_sync_all();  // no CTA tears down its barriers / TMEM while the peer may still signal or read them
  tc_fence_after_sync();
  if (warp == 2) tmem_dealloc_pair(tmem_base, Cfg::TMEM_COLS);
}


// Per-row running state of the online log-sum-exp, carried ACROSS the column tiles of one unit by the resident-A
// kernel: one partial per (unit, column half, row) instead of one per (tile, half, row) -- 16x fewer partials to
// write, read back and reduce (config 2: 0.64 GB -> 40 MB of DRAM traffic per launch).  Same arithmetic per tile as
// epilogue_head (which the other kernels keep using).
struct HeadRowState {
  float m_run, s_run, z_run, tgt, row_scale;
  int cnt;
  int hit_col;
  int64_t label;
};
__device__ __forceinline__ void head_state_init(HeadRowState& st, const GemmEpilogue& ep, int64_t row, bool row_ok) {
  st.m_run = -INFINITY; st.s_run = 0.f; st.z_run = 0.f; st.cnt = 0; st.label = -1; st.tgt = 0.f;
  if (row_ok && ep.row_label) st.label = ep.row_label[row];
  if (row_ok && ep.row_rank) st.tgt = ep.row_tgt[row];
  st.row_scale = (row_ok && ep.row_scale) ? ep.row_scale[row] : 1.f;
  st.hit_col = (row_ok && ep.hit_col) ? ep.hit_col[row] : -1;
}
template <int BN>
__device__ __forceinline__ void head_state_tile(HeadRowState& st, const GemmDev& p, uint32_t taddr, bool row_ok, int64_t n0) {
  constexpr int COLS = BN / 2;
  const GemmEpilogue& ep = p.ep;
  constexpr float kLog2e = 1.4426950408889634f;
  const float scale2 = ep.inv_tau * kLog2e;
  const bool want_z = (ep.part_z != nullptr);
  const bool want_rank = (ep.row_rank != nullptr);
  const bool full_tile = (n0 + COLS <= p.N);
  // Fast path of the training full softmax (no logQ bias, no hit removal, no ranks, no label smoothing, whole tile
  // inside V): packed fp32 pairs (fmul2 / ffma2 / fadd2) halve the FMA-pipe instructions per logit and the row scale
  // of the 2-unit product rides in the exponent's scale factor instead of costing a multiply per logit.  With K = 64
  // (config 3) or nprod = 2 the main loop is short enough for this epilogue to be on the critical path.
  if (full_tile && !ep.col_bias && !ep.col_ids && !ep.hit_col && !want_rank && !want_z) {
    const float scale2r = scale2 * st.row_scale;  // > 0: power-of-two row scale
    // The column scales of the 2-unit product (one per table row) are the only global loads of this epilogue, and their
    // latency sat right in front of the multiply: 54 % of the kernel's stall samples (profiles/r2_head_lines.txt), with
    // the tensor pipe at 74 % -- the epilogue paces the kernel.  They are now fetched one chunk AHEAD, before the
    // TMEM load of the chunk they follow.
    const bool scaled = ep.col_scale != nullptr;
    float4 cs_cur[8], cs_nxt[8];
    if (scaled) {
      const float4* c4 = reinterpret_cast<const float4*>(ep.col_scale + n0);
#pragma unroll
      for (int j = 0; j < 8; ++j) cs_cur[j] = __ldg(c4 + j);
    }
#pragma unroll 1
    for (int c = 0; c < COLS / 32; ++c) {
      if (scaled && c + 1 < COLS / 32) {
        const float4* c4 = reinterpret_cast<const float4*>(ep.col_scale + n0 + (c + 1) * 32);
#pragma unroll
        for (int j = 0; j < 8; ++j) cs_nxt[j] = __ldg(c4 + j);
      }
      float v[32];
      tmem_ld<32>(taddr + c * 32, v);
      float2* v2 = reinterpret_cast<float2*>(v);
      if (scaled) {
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          v2[2 * j] = __fmul2_rn(v2[2 * j], make_float2(cs_cur[j].x, cs_cur[j].y));
          v2[2 * j + 1] = __fmul2_rn(v2[2 * j + 1], make_float2(cs_cur[j].z, cs_cur[j].w));
          cs_cur[j] = cs_nxt[j];
        }
      }
      if (!row_ok) continue;
      float mx[4] = {v[0], v[1], v[2], v[3]};
#pragma unroll
      for (int j = 4; j < 32; j += 4) {
        mx[0] = fmaxf(mx[0], v[j]); mx[1] = fmaxf(mx[1], v[j + 1]);
        mx[2] = fmaxf(mx[2], v[j + 2]); mx[3] = fmaxf(mx[3], v[j + 3]);
      }
      const float cmax = fmaxf(fmaxf(mx[0], mx[1]), fmaxf(mx[2], mx[3])) * scale2r;
      const float m_new = fmaxf(st.m_run, cmax);
      if (m_new > -INFINITY) {
        const float2 sc = make_float2(scale2r, scale2r), nm = make_float2(-m_new, -m_new);
        float2 acc2[2] = {make_float2(0.f, 0.f), make_float2(0.f, 0.f)};
#pragma unroll
        for (int j = 0; j < 16; j += 2) {
          const float2 a0 = __ffma2_rn(v2[j], sc, nm), a1 = __ffma2_rn(v2[j + 1], sc, nm);
          acc2[0] = __fadd2_rn(acc2[0], make_float2(fast_exp2(a0.x), fast_exp2(a0.y)));
          acc2[1] = __fadd2_rn(acc2[1], make_float2(fast_exp2(a1.x), fast_exp2(a1.y)));
        }
        st.s_run = st.s_run * fast_exp2(st.m_run - m_new) + ((acc2[0].x + acc2[0].y) + (acc2[1].x + acc2[1].y));
        st.m_run = m_new;
      }
    }
    return;
  }
#pragma unroll 1
  for (int c = 0; c < COLS / 32; ++c) {
    float v[32];
    tmem_ld<32>(taddr + c * 32, v);
    if (!row_ok) continue;
    const int64_t ncol0 = n0 + c * 32;
    if (ncol0 >= p.N) continue;
    if (ep.col_scale) {
      if (full_tile) {
        const float4* c4 = reinterpret_cast<const float4*>(ep.col_scale + ncol0);
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const float4 cs = __ldg(c4 + j);
          v[4 * j + 0] *= st.row_scale * cs.x; v[4 * j + 1] *= st.row_scale * cs.y;
          v[4 * j + 2] *= st.row_scale * cs.z; v[4 * j + 3] *= st.row_scale * cs.w;
        }
      } else {
#pragma unroll
        for (int j = 0; j < 32; ++j)
          if (ncol0 + j < p.N) v[j] *= st.row_scale * __ldg(ep.col_scale + ncol0 + j);
      }
    }
    if (ep.col_bias) {
      if (full_tile && (ncol0 & 3) == 0) {
        const float4* b4 = reinterpret_cast<const float4*>(ep.col_bias + ncol0);
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const float4 b = __ldg(b4 + j);
          v[4 * j + 0] += b.x; v[4 * j + 1] += b.y; v[4 * j + 2] += b.z; v[4 * j + 3] += b.w;
        }
      } else {
#pragma unroll
        for (int j = 0; j < 32; ++j)
          if (full_tile || ncol0 + j < p.N) v[j] += __ldg(ep.col_bias + ncol0 + j);
      }
    }
    if (ep.hit_col) {           // the row's accidental hit, found once per row (launch_hit_cols)
      const int64_t rel = static_cast<int64_t>(st.hit_col) - ncol0;
      if (rel >= 0 && rel < 32) {
#pragma unroll
        for (int j = 0; j < 32; ++j)
          if (j == rel) v[j] = ep.hit_value;
      }
    } else if (ep.col_ids) {
#pragma unroll
      for (int j = 0; j < 32; ++j)
        if ((full_tile || ncol0 + j < p.N) && __ldg(ep.col_ids + ncol0 + j) == st.label) v[j] = ep.hit_value;
    }
    if (!full_tile) {
#pragma unroll
      for (int j = 0; j < 32; ++j)
        if (ncol0 + j >= p.N) v[j] = -INFINITY;
    }
    if (want_rank) {
      const int64_t lab_col = st.label - ep.col_offset;
#pragma unroll
      for (int j = 0; j < 32; ++j) {
        const float x = v[j] * ep.inv_tau;
        const int64_t col = ncol0 + j;
        st.cnt += (col != lab_col) && ((x > st.tgt) || (x == st.tgt && col < lab_col));
      }
    }
    if (want_z) {
      float zs = 0.f;
#pragma unroll
      for (int j = 0; j < 32; ++j) zs += (v[j] == -INFINITY) ? 0.f : v[j];
      st.z_run = fmaf(zs, ep.inv_tau, st.z_run);
    }
    float mx[4] = {v[0], v[1], v[2], v[3]};
#pragma unroll
    for (int j = 4; j < 32; j += 4) {
      mx[0] = fmaxf(mx[0], v[j]); mx[1] = fmaxf(mx[1], v[j + 1]);
      mx[2] = fmaxf(mx[2], v[j + 2]); mx[3] = fmaxf(mx[3], v[j + 3]);
    }
    const float cmax = fmaxf(fmaxf(mx[0], mx[1]), fmaxf(mx[2], mx[3])) * scale2;
    const float m_new = fmaxf(st.m_run, cmax);
    if (m_new > -INFINITY) {
      float acc[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
      for (int j = 0; j < 32; j += 4) {
        acc[0] += fast_exp2(fmaf(v[j], scale2, -m_new));
        acc[1] += fast_exp2(fmaf(v[j + 1], scale2, -m_new));
        acc[2] += fast_exp2(fmaf(v[j + 2], scale2, -m_new));
        acc[3] += fast_exp2(fmaf(v[j + 3], scale2, -m_new));
      }
      st.s_run = st.s_run * fast_exp2(st.m_run - m_new) + ((acc[0] + acc[1]) + (acc[2] + acc[3]));
      st.m_run = m_new;
    }
  }
}
__device__ __forceinline__ void head_state_flush(const HeadRowState& st, const GemmEpilogue& ep, int64_t row, bool row_ok,
                                                 int part_idx) {
  if (!row_ok) return;
  ep.part_m[static_cast<int64_t>(part_idx) * ep.part_ld + row] = st.m_run;
  ep.part_s[static_cast<int64_t>(part_idx) * ep.part_ld + row] = st.s_run;
  if (ep.part_z) ep.part_z[static_cast<int64_t>(part_idx) * ep.part_ld + row] = st.z_run;
  if (ep.row_rank && st.cnt) atomicAdd(ep.row_rank + row, st.cnt);
}

// ============================================================================
// Head GEMM with a RESIDENT A tile (CTA pairs, K <= 256; the default head kernel since round 2, T4R_HEAD_RESIDENT=0 = streaming).
// The tied-logits GEMM multiplies a small A (T label rows) by a huge B (the item table).  In gemm2_bf16x3_kernel
// every 256 x 256 output tile re-streams both operands from L2: 64 KB per CTA and K block, half of it A -- the same
// A rows over and over.  Here a CTA pair works on UNITS of (one 256-row block of A) x (HEAD_CHUNK consecutive column
// tiles): A (all K blocks, 4 x 32 KB per CTA) is loaded once per unit and stays in shared memory, only the B half-tiles
// (32 KB per K block) stream through a 3-stage ring.  L2->SM traffic per launch drops from 2 x (A + B) to
// ~(1 + 1/HEAD_CHUNK) x ... half (config 2: 41 GB -> ~22 GB), which matters once the products get cheaper than the
// operand stream (nprod = 2: 1024 tensor cycles per 64 KB; nprod = 1: 512).  Units are numbered column-chunk-major,
// row-block-minor and dealt round-robin to the pairs, so the ~20 row blocks of one column chunk run at the same time
// on neighbouring pairs and share the chunk's B tiles in L2.  The A slot of K block kb is released by a commit after the
// LAST tile's MMAs on it, so the next unit's A[kb] load overlaps the tail of the current unit (no drain bubble).
// Barriers: a_full/a_empty[4] (per K block, one phase per unit), b_full/b_empty[3], tfull/tempty[2] as in gemm2.
// ============================================================================
constexpr int HEAD_CHUNK_DEFAULT = 16;
// column tiles per unit: T4R_HEAD_CHUNK (1..256) for tuning without a rebuild; read per call
static int head_chunk() {
  int c = HEAD_CHUNK_DEFAULT;
  if (const char* e = getenv("T4R_HEAD_CHUNK")) c = atoi(e);
  return c < 1 ? 1 : (c > 256 ? 256 : c);
}
struct HeadResCfg {
  static constexpr int BN = 256;
  static constexpr int A_PLANE_BYTES = BM * 128;             // 16 KB: 128 rows x 64 K elements, one plane
  static constexpr int A_SLOT_BYTES = 2 * A_PLANE_BYTES;     // both planes of one K block
  static constexpr int MAX_KB = 4;                           // K <= 256
  static constexpr int B_PLANE_BYTES = (BN / 2) * 128;       // this CTA's half of the B tile, one plane
  static constexpr int B_STAGE_BYTES = 2 * B_PLANE_BYTES;
  static constexpr int STAGES = 3;
  static constexpr int TMEM_COLS = 2 * BN;
  static constexpr int DATA_BYTES = MAX_KB * A_SLOT_BYTES + STAGES * B_STAGE_BYTES;  // 224 KB
  static constexpr int SMEM_BYTES = DATA_BYTES + 1024 /*align*/ + 256 /*barriers*/;
};

__global__ void __launch_bounds__(320, 1)
head_resident_kernel(const __grid_constant__ CUtensorMap tmAh, const __grid_constant__ CUtensorMap tmAl,
                     const __grid_constant__ CUtensorMap tmBh, const __grid_constant__ CUtensorMap tmBl,
                     const GemmDev p) {
  using Cfg = HeadResCfg;
  constexpr int BN = Cfg::BN;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  uint8_t* a_base = smem;
  uint8_t* b_base = smem + Cfg::MAX_KB * Cfg::A_SLOT_BYTES;
  uint64_t* a_full = reinterpret_cast<uint64_t*>(smem + Cfg::DATA_BYTES);
  uint64_t* a_empty = a_full + Cfg::MAX_KB;
  uint64_t* b_full = a_empty + Cfg::MAX_KB;
  uint64_t* b_empty = b_full + Cfg::STAGES;
  uint64_t* tfull_bar = b_empty + Cfg::STAGES;
  uint64_t* tempty_bar = tfull_bar + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty_bar + 2);

  const int warp = warp_id();
  const int lane = lane_id();
  const int rank = static_cast<int>(cluster_ctarank());
  const bool leader = (rank == 0);
  const int pair = blockIdx.x >> 1;
  const int npairs = gridDim.x >> 1;

  int M_eff = p.M;
  if (p.m_dev) M_eff = min(p.M, *p.m_dev);
  const int tiles_m = (M_eff + 2 * BM - 1) / (2 * BM);
  const int tiles_n = static_cast<int>((p.N + BN - 1) / BN);
  const int HEAD_CHUNK = p.head_chunk;
  const int chunks_n = (tiles_n + HEAD_CHUNK - 1) / HEAD_CHUNK;
  const int64_t num_units = static_cast<int64_t>(tiles_m) * chunks_n;
  const int nkb = p.nkb;  // <= MAX_KB (checked by the launcher)

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmAh); tma_prefetch_desc(&tmAl); tma_prefetch_desc(&tmBh); tma_prefetch_desc(&tmBl);
  }
  if (warp == 1 && lane == 0) {
    for (int i = 0; i < Cfg::MAX_KB; ++i) { mbar_init(&a_full[i], 1); mbar_init(&a_empty[i], 1); }
    for (int i = 0; i < Cfg::STAGES; ++i) { mbar_init(&b_full[i], 1); mbar_init(&b_empty[i], 1); }
    for (int i = 0; i < 2; ++i) { mbar_init(&tfull_bar[i], 1); mbar_init(&tempty_bar[i], 16); }
    fence_barrier_init();
  }
  if (warp == 2) {
    tmem_alloc_pair(tmem_slot, Cfg::TMEM_COLS);
    tmem_relinquish_pair();
  }
  tc_fence_before_sync();
  __syncthreads();
  cluster_sync_all();
  tc_fence_after_sync();
  const uint32_t tmem_base = *tmem_slot;
  const bool two_planes = (p.nprod != 1);

  if (warp == 0) {
    // ===================== TMA producer (both CTAs) =====================
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      uint32_t uphase = 0;  // parity of the unit count: one a_full / a_empty phase per unit and K block
      const uint32_t a_bytes = two_planes ? Cfg::A_SLOT_BYTES : Cfg::A_PLANE_BYTES;
      const uint32_t b_bytes = two_planes ? Cfg::B_STAGE_BYTES : Cfg::B_PLANE_BYTES;
      for (int64_t unit = pair; unit < num_units; unit += npairs) {
        const int tm = static_cast<int>(unit % tiles_m);
        const int chunk = static_cast<int>(unit / tiles_m);
        const int m0 = tm * (2 * BM) + rank * BM;
        const int t_begin = chunk * HEAD_CHUNK;
        const int t_end = min(t_begin + HEAD_CHUNK, tiles_n);
        for (int tn = t_begin; tn < t_end; ++tn) {
          const int n0 = tn * BN + rank * (BN / 2);
          for (int kb = 0; kb < nkb; ++kb) {
            if (tn == t_begin) {  // this unit's A, K block kb: wait until the previous unit's last MMAs on the slot retired
              mbar_wait(&a_empty[kb], uphase ^ 1);
              uint8_t* sa = a_base + kb * Cfg::A_SLOT_BYTES;
              if (leader) mbar_arrive_expect_tx(&a_full[kb], 2 * a_bytes);
              tma_load_2d_pair(sa, &tmAh, &a_full[kb], kb * 64, m0);
              if (two_planes) tma_load_2d_pair(sa + Cfg::A_PLANE_BYTES, &tmAl, &a_full[kb], kb * 64, m0);
            }
            mbar_wait(&b_empty[stage], phase ^ 1);
            uint8_t* sb = b_base + stage * Cfg::B_STAGE_BYTES;
            if (leader) mbar_arrive_expect_tx(&b_full[stage], 2 * b_bytes);
            tma_load_2d_pair(sb, &tmBh, &b_full[stage], kb * 64, n0);
            if (two_planes) tma_load_2d_pair(sb + Cfg::B_PLANE_BYTES, &tmBl, &b_full[stage], kb * 64, n0);
            if (++stage == Cfg::STAGES) { stage = 0; phase ^= 1; }
          }
        }
        uphase ^= 1;
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    // ===================== MMA issuer (leader only) =====================
    if (leader && lane == 0) {
      constexpr uint32_t idesc = umma_idesc_bf16(2 * BM, BN);
      constexpr uint32_t idesc_h = umma_idesc_f16(2 * BM, BN);
      constexpr uint32_t idesc_8 = umma_idesc_e4m3(2 * BM, BN);
      int stage = 0;
      uint32_t phase = 0;
      uint32_t uphase = 0;
      int as = 0;
      uint32_t aph = 0;
      for (int64_t unit = pair; unit < num_units; unit += npairs) {
        const int chunk = static_cast<int>(unit / tiles_m);
        const int t_begin = chunk * HEAD_CHUNK;
        const int t_end = min(t_begin + HEAD_CHUNK, tiles_n);
        for (int tn = t_begin; tn < t_end; ++tn) {
          mbar_wait(&tempty_bar[as], aph ^ 1);
          tc_fence_after_sync();
          const uint32_t d_tmem = tmem_base + static_cast<uint32_t>(as * BN);
          for (int kb = 0; kb < nkb; ++kb) {
            if (tn == t_begin) mbar_wait(&a_full[kb], uphase);
            mbar_wait(&b_full[stage], phase);
            tc_fence_after_sync();
            const uint32_t a_hi = smem_u32(a_base + kb * Cfg::A_SLOT_BYTES);
            const uint32_t a_lo = a_hi + Cfg::A_PLANE_BYTES;
            const uint32_t b_hi = smem_u32(b_base + stage * Cfg::B_STAGE_BYTES);
            const uint32_t b_lo = b_hi + Cfg::B_PLANE_BYTES;
            if (p.nprod == 2) {  // fp16 x fp16 + two e4m3 cross terms (t4r_mixed_pack.cuh)
              const int dbg = p.ep.debug;
              uint32_t acc = (kb != 0) ? 1u : 0u;
              if (!(dbg & 64)) {
#pragma unroll
                for (int k4 = 0; k4 < 4; ++k4) {
                  umma_bf16_pair(d_tmem, umma_desc_sw128(a_hi + k4 * 32), umma_desc_sw128(b_hi + k4 * 32), idesc_h, acc);
                  acc = 1u;
                }
              }
#pragma unroll
              for (int j = 0; j < 2; ++j) {
                if (!(dbg & 128)) { umma_f8_pair(d_tmem, umma_desc_sw128(a_lo + 64 + j * 32), umma_desc_sw128(b_lo + j * 32), idesc_8, acc); acc = 1u; }
                if (!(dbg & 256)) { umma_f8_pair(d_tmem, umma_desc_sw128(a_lo + j * 32), umma_desc_sw128(b_lo + 64 + j * 32), idesc_8, acc); acc = 1u; }
              }
            } else {
#pragma unroll
              for (int k4 = 0; k4 < 4; ++k4) {
                const uint64_t da_hi = umma_desc_sw128(a_hi + k4 * 32);
                const uint64_t db_hi = umma_desc_sw128(b_hi + k4 * 32);
                if (p.nprod == 3) {
                  umma_bf16_pair(d_tmem, umma_desc_sw128(a_lo + k4 * 32), db_hi, idesc, (kb | k4) != 0);
                  umma_bf16_pair(d_tmem, da_hi, umma_desc_sw128(b_lo + k4 * 32), idesc, 1u);
                  umma_bf16_pair(d_tmem, da_hi, db_hi, idesc, 1u);
                } else {
                  umma_bf16_pair(d_tmem, da_hi, db_hi, idesc, (kb | k4) != 0);
                }
              }
            }
            umma_commit_pair(&b_empty[stage]);                       // B stage free in both CTAs
            if (tn == t_end - 1) umma_commit_pair(&a_empty[kb]);      // last use of this unit's A[kb]
            if (++stage == Cfg::STAGES) { stage = 0; phase ^= 1; }
          }
          umma_commit_pair(&tfull_bar[as]);
          as ^= 1;
          if (as == 0) aph ^= 1;
        }
        uphase ^= 1;
      }
    }
    __syncwarp();
  } else {
    // ===================== epilogue warps (2..9) of both CTAs =====================
    const int quad = warp & 3;
    const int half = (warp - 2) >> 2;
    constexpr int COLS = BN / 2;
    int as = 0;
    uint32_t aph = 0;
    for (int64_t unit = pair; unit < num_units; unit += npairs) {
      const int tm = static_cast<int>(unit % tiles_m);
      const int chunk = static_cast<int>(unit / tiles_m);
      const int t_begin = chunk * HEAD_CHUNK;
      const int t_end = min(t_begin + HEAD_CHUNK, tiles_n);
      const int64_t m0 = static_cast<int64_t>(tm) * (2 * BM) + rank * BM;
      const int64_t row = m0 + quad * 32 + lane;
      const bool row_ok = row < M_eff;
      HeadRowState st;
      head_state_init(st, p.ep, row, row_ok);
      for (int tn = t_begin; tn < t_end; ++tn) {
        const int64_t n0 = static_cast<int64_t>(tn) * BN + half * COLS;
        mbar_wait(&tfull_bar[as], aph);
        tc_fence_after_sync();
        const uint32_t taddr = tmem_base + (static_cast<uint32_t>(quad * 32) << 16) +
                               static_cast<uint32_t>(as * BN + half * COLS);
        head_state_tile<BN>(st, p, taddr, row_ok, n0);
        tc_fence_before_sync();
        __syncwarp();
        if (lane == 0) mbar_arrive_leader(&tempty_bar[as]);
        as ^= 1;
        if (as == 0) aph ^= 1;
      }
      head_state_flush(st, p.ep, row, row_ok, chunk * 2 + half);  // ONE partial per (column chunk, half, row)
    }
  }

  tc_fence_before_sync();
  __syncthreads();
  cluster_sync_all();
  tc_fence_after_sync();
  if (warp == 2) tmem_dealloc_pair(tmem_base, Cfg::TMEM_COLS);
}

// ----------------------------------------------------------------------------
// host launcher
// ----------------------------------------------------------------------------
static int g_num_sms = 0;
static int num_sms() {
  if (g_num_sms == 0) {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return 148;
    int n = 0;
    if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) n = 148;
    g_num_sms = n;
  }
  return g_num_sms;
}

template <int BN, bool LN, bool HEAD>
static int launch_inst(const CUtensorMap& ah, const CUtensorMap& al, const CUtensorMap& bh, const CUtensorMap& bl,
                       const GemmDev& dp, int64_t max_tiles, cudaStream_t stream) {
  using Cfg = GemmCfg<BN>;
  auto kern = gemm_bf16x3_kernel<BN, LN, HEAD>;
  static bool attr_set = false;
  if (!attr_set) {
    T4R_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::SMEM_BYTES));
    attr_set = true;
  }
  int grid = static_cast<int>(max_tiles < num_sms() ? max_tiles : num_sms());
  if (grid < 1) grid = 1;
  kern<<<grid, 320, Cfg::SMEM_BYTES, stream>>>(ah, al, bh, bl, dp);
  T4R_LAUNCH_CHECK("gemm_bf16x3_kernel");
  return 0;
}


template <int BN, bool LN, bool HEAD>
static int launch_inst2(const CUtensorMap& ah, const CUtensorMap& al, const CUtensorMap& bh, const CUtensorMap& bl,
                        const GemmDev& dp, int64_t max_pair_tiles, cudaStream_t stream) {
  using Cfg = Gemm2Cfg<BN>;
  auto kern = gemm2_bf16x3_kernel<BN, LN, HEAD>;
  static bool attr_set = false;
  if (!attr_set) {
    T4R_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::SMEM_BYTES));
    attr_set = true;
  }
  const int max_pairs = num_sms() / 2;
  int pairs = static_cast<int>(max_pair_tiles < max_pairs ? max_pair_tiles : max_pairs);
  if (pairs < 1) pairs = 1;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(2 * pairs, 1, 1);
  cfg.blockDim = dim3(320, 1, 1);
  cfg.dynamicSmemBytes = Cfg::SMEM_BYTES;
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 2;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  T4R_CUDA(cudaLaunchKernelEx(&cfg, kern, ah, al, bh, bl, dp));
  T4R_LAUNCH_CHECK("gemm2_bf16x3_kernel");
  return 0;
}

static int launch_head_resident(const CUtensorMap& ah, const CUtensorMap& al, const CUtensorMap& bh, const CUtensorMap& bl,
                                const GemmDev& dp, int64_t units, cudaStream_t stream) {
  using Cfg = HeadResCfg;
  static bool attr_set = false;
  if (!attr_set) {
    T4R_CUDA(cudaFuncSetAttribute(head_resident_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::SMEM_BYTES));
    attr_set = true;
  }
  const int max_pairs = num_sms() / 2;
  int pairs = static_cast<int>(units < max_pairs ? units : max_pairs);
  if (pairs < 1) pairs = 1;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(2 * pairs, 1, 1);
  cfg.blockDim = dim3(320, 1, 1);
  cfg.dynamicSmemBytes = Cfg::SMEM_BYTES;
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 2;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  T4R_CUDA(cudaLaunchKernelEx(&cfg, head_resident_kernel, ah, al, bh, bl, dp));
  T4R_LAUNCH_CHECK("head_resident_kernel");
  return 0;
}

}  // namespace t4r
extern "C" int t4r_debug_ffn_cycles(unsigned long long* out16, int reset) {
  if (out16) cudaMemcpyFromSymbol(out16, t4r::g_dbg_ffn, sizeof(unsigned long long) * 16);
  if (reset) { unsigned long long z[16] = {0}; cudaMemcpyToSymbol(t4r::g_dbg_ffn, z, sizeof(z)); }
  return 0;
}
extern "C" int t4r_debug_gemm_cycles(unsigned long long* out8, int reset) {
  if (out8) cudaMemcpyFromSymbol(out8, t4r::g_dbg_cycles, sizeof(unsigned long long) * 8);
  if (reset) { unsigned long long z[8] = {0}; cudaMemcpyToSymbol(t4r::g_dbg_cycles, z, sizeof(z)); }
  return 0;
}
namespace t4r {
// T4R_HEAD_RESIDENT != 0 (the default) and a shape the resident-A head kernel covers: K <= 256, more than one 128-row
// block, CTA pairs enabled.  Returns the number of LSE partials per row the head call must size
// for (2 per column CHUNK), or 0 when the regular kernels run (2 per column TILE).
int head_resident_partials(int64_t M, int64_t V, int Kp) {
  int resident = T4R_HEAD_RESIDENT_DEFAULT;
  if (const char* e = getenv("T4R_HEAD_RESIDENT")) resident = atoi(e);
  int two_cta = T4R_GEMM_2CTA_DEFAULT;
  if (const char* e = getenv("T4R_GEMM_2CTA")) two_cta = atoi(e);
  if (!resident || !two_cta || M <= BM || Kp > 64 * HeadResCfg::MAX_KB) return 0;
  const int64_t tiles_n = (V + HeadResCfg::BN - 1) / HeadResCfg::BN;
  const int hc = head_chunk();
  return 2 * static_cast<int>((tiles_n + hc - 1) / hc);
}

int launch_gemm(const GemmProblem& pb, const GemmEpilogue& ep, cudaStream_t stream) {
  T4R_REQUIRE(pb.M > 0 && pb.N > 0 && pb.Kp > 0 && pb.Kp % 64 == 0, "gemm: bad shape M=%lld N=%lld Kp=%d",
              (long long)pb.M, (long long)pb.N, pb.Kp);
  T4R_REQUIRE(pb.M < (1ll << 31), "gemm: M too large");
  T4R_REQUIRE(pb.nprod == 1 || pb.nprod == 3 || pb.nprod == 2, "gemm: nprod must be 1, 2 or 3");
  T4R_REQUIRE(pb.nprod != 2 || (ep.row_scale && ep.col_scale && ep.ln_gamma == nullptr),
              "gemm: nprod = 2 (fp16 + e4m3 cross terms) needs both row-scale vectors and has no LayerNorm epilogue");
  const bool ln = ep.ln_gamma != nullptr;
  int bn = pb.bn;
  if (ln) {
    T4R_REQUIRE(pb.N == 64 || pb.N == 128 || pb.N == 256,
                "fused LayerNorm epilogue supports N in {64,128,256}, got %lld", (long long)pb.N);
    bn = static_cast<int>(pb.N);
  } else if (ep.head) {
    if (bn == 0) bn = 256;
  } else {
    if (bn == 0) {
      const int64_t np = (pb.N + 63) / 64 * 64;
      bn = (np % 256 == 0) ? 256 : ((np % 128 == 0) ? 128 : 64);
    }
    T4R_REQUIRE((ep.residual == nullptr && ep.residual_planes == nullptr) || pb.N % 32 == 0,
                "gemm: a residual needs N %% 32 == 0");
  }
  T4R_REQUIRE(bn == 64 || bn == 128 || bn == 256, "gemm: bad BN %d", bn);

  CUtensorMap ah, al, bh, bl;
  T4R_TRY(make_tmap(&ah, pb.a_planes, pb.M, pb.Kp, BM));
  T4R_TRY(make_tmap(&al, pb.a_planes + pb.a_rows * pb.Kp, pb.M, pb.Kp, BM));
  T4R_TRY(make_tmap(&bh, pb.b_planes, pb.N, pb.Kp, bn));
  T4R_TRY(make_tmap(&bl, pb.b_planes + pb.b_rows * pb.Kp, pb.N, pb.Kp, bn));

  GemmDev dp;
  dp.M = static_cast<int>(pb.M);
  dp.N = pb.N;
  dp.nkb = pb.Kp / 64;
  dp.nprod = pb.nprod;
  dp.head_chunk = head_chunk();
  dp.m_dev = pb.m_dev;
  dp.ep = ep;
  {
    const char* e = getenv("T4R_GEMM_DEBUG");  // read per call: tests flip the bring-up switches within one process
    dp.ep.debug = e ? atoi(e) : 0;
  }
  const int64_t max_tiles = ((pb.M + BM - 1) / BM) * ((pb.N + bn - 1) / bn);

  // T4R_GEMM_2CTA=1: CTA-pair kernel (cta_group::2, 256-row tiles).  Needs more than one 128-row tile.
  int two_cta = T4R_GEMM_2CTA_DEFAULT;  // read per call so that tests can exercise both kernels in one process
  if (const char* e = getenv("T4R_GEMM_2CTA")) two_cta = atoi(e);
  if (two_cta && pb.M > BM) {
    CUtensorMap bh2, bl2;
    T4R_TRY(make_tmap(&bh2, pb.b_planes, pb.N, pb.Kp, bn / 2));
    T4R_TRY(make_tmap(&bl2, pb.b_planes + pb.b_rows * pb.Kp, pb.N, pb.Kp, bn / 2));
    const int64_t pair_tiles = ((pb.M + 2 * BM - 1) / (2 * BM)) * ((pb.N + bn - 1) / bn);
    // the head kernel that keeps the A tile in shared memory (the head entry point decided it: head_resident_partials)
    T4R_REQUIRE(!ep.head_resident || (ep.head && bn == 256 && dp.nkb <= HeadResCfg::MAX_KB),
                "gemm: resident head requested for an unsupported shape");
    if (ep.head_resident) {
      const int64_t tiles_n = (pb.N + bn - 1) / bn;
      const int64_t units = ((pb.M + 2 * BM - 1) / (2 * BM)) * ((tiles_n + dp.head_chunk - 1) / dp.head_chunk);
      return launch_head_resident(ah, al, bh2, bl2, dp, units, stream);
    }
    if (ep.head) {
      if (bn == 256) return launch_inst2<256, false, true>(ah, al, bh2, bl2, dp, pair_tiles, stream);
      if (bn == 128) return launch_inst2<128, false, true>(ah, al, bh2, bl2, dp, pair_tiles, stream);
      return launch_inst2<64, false, true>(ah, al, bh2, bl2, dp, pair_tiles, stream);
    }
    if (ln) {
      if (bn == 256) return launch_inst2<256, true, false>(ah, al, bh2, bl2, dp, pair_tiles, stream);
      if (bn == 128) return launch_inst2<128, true, false>(ah, al, bh2, bl2, dp, pair_tiles, stream);
      return launch_inst2<64, true, false>(ah, al, bh2, bl2, dp, pair_tiles, stream);
    }
    if (bn == 256) return launch_inst2<256, false, false>(ah, al, bh2, bl2, dp, pair_tiles, stream);
    if (bn == 128) return launch_inst2<128, false, false>(ah, al, bh2, bl2, dp, pair_tiles, stream);
    return launch_inst2<64, false, false>(ah, al, bh2, bl2, dp, pair_tiles, stream);
  }

  T4R_REQUIRE(!ep.head_resident, "gemm: resident head needs the CTA-pair path (T4R_GEMM_2CTA=1, M > 128)");
  if (ep.head) {
    if (bn == 256) return launch_inst<256, false, true>(ah, al, bh, bl, dp, max_tiles, stream);
    if (bn == 128) return launch_inst<128, false, true>(ah, al, bh, bl, dp, max_tiles, stream);
    return launch_inst<64, false, true>(ah, al, bh, bl, dp, max_tiles, stream);
  }
  if (ln) {
    if (bn == 256) return launch_inst<256, true, false>(ah, al, bh, bl, dp, max_tiles, stream);
    if (bn == 128) return launch_inst<128, true, false>(ah, al, bh, bl, dp, max_tiles, stream);
    return launch_inst<64, true, false>(ah, al, bh, bl, dp, max_tiles, stream);
  }
  if (bn == 256) return launch_inst<256, false, false>(ah, al, bh, bl, dp, max_tiles, stream);
  if (bn == 128) return launch_inst<128, false, false>(ah, al, bh, bl, dp, max_tiles, stream);
  return launch_inst<64, false, false>(ah, al, bh, bl, dp, max_tiles, stream);
}


// ============================================================================
// K7: fused feed-forward block
//     Y = epilogue( gelu(X W1^T + b1) W2^T )          epilogue = + b2 + residual -> LayerNorm -> stores
//     (HF:xlnet:297-305 XLNetFeedForward; HF:gpt2:229-243 GPT2MLP + the residual / next LayerNorm)
// The 4d-wide intermediate never leaves the SM: per 128-row tile the hidden units are processed in
// chunks of 128.  GEMM1 (SS form: X and W1 chunk from shared memory via TMA) accumulates the chunk in
// TMEM; the epilogue warps apply bias + GELU, split to bf16 hi/lo and write the result back to TMEM
// as the A operand of GEMM2 (TS form: A from TMEM, W2 chunk from shared memory), which accumulates
// the d-wide output in TMEM across all chunks.  The MMA warp issues GEMM1(c+1) before GEMM2(c), so
// the GELU of chunk c runs under GEMM1(c+1).  All products are issued three times (split bf16).
// TMEM columns: Y [0,256)  S [256,384)  G_hi [384,448)  G_lo [448,512).
// ============================================================================
__device__ __forceinline__ void umma_bf16_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t bdesc, uint32_t idesc,
                                             uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}"
      ::"r"(tmem_d), "r"(tmem_a), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}

struct FfnDev {
  int M;
  int n_chunks;          // hidden / 128
  const float* b1;       // [hidden]
  GemmEpilogue ep;       // final epilogue (bias = b2, residual, LayerNorm, outputs)
};

constexpr int FFN_HC = 128;                 // hidden units per chunk
constexpr int FFN_STAGE_BYTES = 64 * 1024;  // one ring stage (see below)
constexpr int FFN_STAGES = 3;
constexpr int FFN_SMEM_BYTES = FFN_STAGES * FFN_STAGE_BYTES + 1024 + 256 + 4096 + 8 * 32 * 20 * 4;

template <int D>
__global__ void __launch_bounds__(320, 1)
ffn_fused_kernel(const __grid_constant__ CUtensorMap tmXh, const __grid_constant__ CUtensorMap tmXl,
                 const __grid_constant__ CUtensorMap tmW1h, const __grid_constant__ CUtensorMap tmW1l,
                 const __grid_constant__ CUtensorMap tmW2h, const __grid_constant__ CUtensorMap tmW2l, const FfnDev p) {
  constexpr int STAGES = FFN_STAGES;
  constexpr int HCW = FFN_HC / 2;                   // hidden units of a chunk per epilogue warp
  constexpr int KB1 = D / 64;                       // k blocks of GEMM1 (K = d)
  constexpr int KB2 = FFN_HC / 64;                  // k blocks of GEMM2 per chunk (K = 128)
  constexpr int XP = BM * 128;                      // X plane bytes per k block
  constexpr int W1P = FFN_HC * 128;                 // W1 chunk plane bytes per k block
  constexpr int W2P = D * 128;                      // W2 chunk plane bytes per k block
  constexpr uint32_t Y_COL = 0, S_COL = 256, GH_COL = 384, GL_COL = 448;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + STAGES * FFN_STAGE_BYTES);
  uint64_t* empty_bar = full_bar + STAGES;
  uint64_t* s_full = empty_bar + STAGES;
  uint64_t* s_empty = s_full + 1;
  uint64_t* g_full = s_empty + 1;
  uint64_t* g_empty = g_full + 1;
  uint64_t* y_full = g_empty + 1;
  uint64_t* y_empty = y_full + 1;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(y_empty + 1);
  float2* xch = reinterpret_cast<float2*>(smem + STAGES * FFN_STAGE_BYTES + 256);
  float* stg_all = reinterpret_cast<float*>(smem + STAGES * FFN_STAGE_BYTES + 256 + 4096);

  const int warp = warp_id();
  const int lane = lane_id();
  const int tiles_m = (p.M + BM - 1) / BM;
  const int NC = p.n_chunks;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmXh); tma_prefetch_desc(&tmXl);
    tma_prefetch_desc(&tmW1h); tma_prefetch_desc(&tmW1l);
    tma_prefetch_desc(&tmW2h); tma_prefetch_desc(&tmW2l);
  }
  if (warp == 1 && lane == 0) {
    for (int i = 0; i < STAGES; ++i) { mbar_init(&full_bar[i], 1); mbar_init(&empty_bar[i], 1); }
    mbar_init(s_full, 1); mbar_init(s_empty, 8);
    mbar_init(g_full, 8); mbar_init(g_empty, 1);
    mbar_init(y_full, 1); mbar_init(y_empty, 8);
    fence_barrier_init();
  }
  if (warp == 2) {
    tmem_alloc(tmem_slot, 512);
    tmem_relinquish();
  }
  tc_fence_before_sync();
  __syncthreads();
  tc_fence_after_sync();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // ===================== TMA producer: stages in the exact order the MMA warp consumes them =====
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      auto load_g1 = [&](int m0, int c, int kb) {
        mbar_wait(&empty_bar[stage], phase ^ 1);
        uint8_t* st = smem + stage * FFN_STAGE_BYTES;
        mbar_arrive_expect_tx(&full_bar[stage], 2 * XP + 2 * W1P);
        tma_load_2d(st, &tmXh, &full_bar[stage], kb * 64, m0);
        tma_load_2d(st + XP, &tmXl, &full_bar[stage], kb * 64, m0);
        tma_load_2d(st + 2 * XP, &tmW1h, &full_bar[stage], kb * 64, c * FFN_HC);
        tma_load_2d(st + 2 * XP + W1P, &tmW1l, &full_bar[stage], kb * 64, c * FFN_HC);
        if (++stage == STAGES) { stage = 0; phase ^= 1; }
      };
      auto load_g2 = [&](int c, int kb) {
        mbar_wait(&empty_bar[stage], phase ^ 1);
        uint8_t* st = smem + stage * FFN_STAGE_BYTES;
        mbar_arrive_expect_tx(&full_bar[stage], 2 * W2P);
        tma_load_2d(st, &tmW2h, &full_bar[stage], c * FFN_HC + kb * 64, 0);
        tma_load_2d(st + W2P, &tmW2l, &full_bar[stage], c * FFN_HC + kb * 64, 0);
        if (++stage == STAGES) { stage = 0; phase ^= 1; }
      };
      for (int tile = blockIdx.x; tile < tiles_m; tile += gridDim.x) {
        const int m0 = tile * BM;
        for (int kb = 0; kb < KB1; ++kb) load_g1(m0, 0, kb);
        for (int c = 0; c < NC; ++c) {
          if (c + 1 < NC)
            for (int kb = 0; kb < KB1; ++kb) load_g1(m0, c + 1, kb);
          for (int kb = 0; kb < KB2; ++kb) load_g2(c, kb);
        }
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    // ===================== MMA issuer =====================
    if (lane == 0) {
      constexpr uint32_t idesc1 = umma_idesc_bf16(BM, FFN_HC);
      constexpr uint32_t idesc2 = umma_idesc_bf16(BM, D);
      int stage = 0;
      uint32_t phase = 0;
      uint32_t ph_s_empty = 0, ph_g_full = 0, ph_y_empty = 0;
      const bool mprof = (p.ep.debug & 2) && blockIdx.x == 0;
      auto gemm1 = [&]() {  // S = X W1c^T
        const long long q0 = mprof ? clock64() : 0;
        mbar_wait(s_empty, ph_s_empty ^ 1);
        const long long q1 = mprof ? clock64() : 0;
        ph_s_empty ^= 1;
        tc_fence_after_sync();
        for (int kb = 0; kb < KB1; ++kb) {
          mbar_wait(&full_bar[stage], phase);
          tc_fence_after_sync();
          const uint32_t a_hi = smem_u32(smem + stage * FFN_STAGE_BYTES);
          const uint32_t a_lo = a_hi + XP, b_hi = a_hi + 2 * XP, b_lo = b_hi + W1P;
          if (!(p.ep.debug & 4))  // timing experiment: no GEMM1 MMAs
#pragma unroll
          for (int k4 = 0; k4 < 4; ++k4) {
            umma_bf16(tmem_base + S_COL, umma_desc_sw128(a_lo + k4 * 32), umma_desc_sw128(b_hi + k4 * 32), idesc1, (kb | k4) != 0);
            umma_bf16(tmem_base + S_COL, umma_desc_sw128(a_hi + k4 * 32), umma_desc_sw128(b_lo + k4 * 32), idesc1, 1u);
            umma_bf16(tmem_base + S_COL, umma_desc_sw128(a_hi + k4 * 32), umma_desc_sw128(b_hi + k4 * 32), idesc1, 1u);
          }
          umma_commit(&empty_bar[stage]);
          if (++stage == STAGES) { stage = 0; phase ^= 1; }
        }
        umma_commit(s_full);
        if (mprof) { g_dbg_ffn[8] += q1 - q0; g_dbg_ffn[9] += clock64() - q1; }
      };
      for (int tile = blockIdx.x; tile < tiles_m; tile += gridDim.x) {
        gemm1();
        for (int c = 0; c < NC; ++c) {
          if (c + 1 < NC) gemm1();  // runs on the tensor pipe while the epilogue warps GELU chunk c
          const long long r0 = mprof ? clock64() : 0;
          mbar_wait(g_full, ph_g_full);
          const long long r1 = mprof ? clock64() : 0;
          ph_g_full ^= 1;
          if (c == 0) {  // Y of the previous tile must have been drained
            mbar_wait(y_empty, ph_y_empty ^ 1);
            ph_y_empty ^= 1;
          }
          const long long r2 = mprof ? clock64() : 0;
          tc_fence_after_sync();
          for (int kb = 0; kb < KB2; ++kb) {  // Y += G_c W2c^T, A (= G) from TMEM
            mbar_wait(&full_bar[stage], phase);
            tc_fence_after_sync();
            const uint32_t b_hi = smem_u32(smem + stage * FFN_STAGE_BYTES);
            const uint32_t b_lo = b_hi + W2P;
            if (!(p.ep.debug & 8))  // timing experiment: no GEMM2 MMAs
#pragma unroll
            for (int k4 = 0; k4 < 4; ++k4) {
              const uint32_t acol = static_cast<uint32_t>(kb * 32 + k4 * 8);
              umma_bf16_ts(tmem_base + Y_COL, tmem_base + GL_COL + acol, umma_desc_sw128(b_hi + k4 * 32), idesc2, (c | kb | k4) != 0);
              umma_bf16_ts(tmem_base + Y_COL, tmem_base + GH_COL + acol, umma_desc_sw128(b_lo + k4 * 32), idesc2, 1u);
              umma_bf16_ts(tmem_base + Y_COL, tmem_base + GH_COL + acol, umma_desc_sw128(b_hi + k4 * 32), idesc2, 1u);
            }
            umma_commit(&empty_bar[stage]);
            if (++stage == STAGES) { stage = 0; phase ^= 1; }
          }
          umma_commit(g_empty);
          if (c == NC - 1) umma_commit(y_full);
          if (mprof) { g_dbg_ffn[10] += r1 - r0; g_dbg_ffn[11] += r2 - r1; g_dbg_ffn[12] += clock64() - r2; g_dbg_ffn[13] += (c == NC - 1); }
        }
      }
    }
    __syncwarp();
  } else {
    // ===================== epilogue warps (2..9) =====================
    const int quad = warp & 3;
    const int half = (warp - 2) >> 2;   // which half of the hidden chunk and of the output columns
    const uint32_t lane_base = static_cast<uint32_t>(quad * 32) << 16;
    uint32_t ph_s_full = 0, ph_g_empty = 0, ph_y_full = 0, tile_parity = 0;
    GemmDev gp;  // view of the final epilogue for epilogue_dense
    gp.M = p.M; gp.N = D; gp.nkb = 0; gp.nprod = 3; gp.m_dev = nullptr; gp.ep = p.ep;
    const bool eprof = (p.ep.debug & 2) && blockIdx.x == 0 && threadIdx.x == 64;
    for (int tile = blockIdx.x; tile < tiles_m; tile += gridDim.x) {
      const int64_t row0 = static_cast<int64_t>(tile) * BM + quad * 32;
      for (int c = 0; c < NC; ++c) {
        // ---- S chunk -> bias + GELU -> split -> G (A operand of GEMM2) in TMEM
        const long long e0 = eprof ? clock64() : 0;
        mbar_wait(s_full, ph_s_full);
        const long long e1 = eprof ? clock64() : 0;
        ph_s_full ^= 1;
        tc_fence_after_sync();
        float v[HCW];
        tmem_ld<HCW>(tmem_base + lane_base + S_COL + half * HCW, v);
        tc_fence_before_sync();
        __syncwarp();
        if (lane == 0) mbar_arrive(s_empty);  // S may be overwritten by GEMM1(c+1)
        const long long e2 = eprof ? clock64() : 0;
        const float* b1 = p.b1 + c * FFN_HC + half * HCW;
        uint32_t gh[HCW / 2], gl[HCW / 2];
#pragma unroll
        for (int j = 0; j < HCW / 4; ++j) {  // bias + GELU + hi/lo split on packed fp32 pairs (fma.rn.f32x2)
          const float4 b = __ldg(reinterpret_cast<const float4*>(b1) + j);
          const float2 g0 = gelu_erf2(__fadd2_rn(make_float2(v[4 * j + 0], v[4 * j + 1]), make_float2(b.x, b.y)));
          const float2 g1 = gelu_erf2(__fadd2_rn(make_float2(v[4 * j + 2], v[4 * j + 3]), make_float2(b.z, b.w)));
          split_bf16x2(g0, gh[2 * j], gl[2 * j]);
          split_bf16x2(g1, gh[2 * j + 1], gl[2 * j + 1]);
        }
        const long long e3 = eprof ? clock64() : 0;
        mbar_wait(g_empty, ph_g_empty ^ 1);  // GEMM2(c-1) has finished reading G
        const long long e4 = eprof ? clock64() : 0;
        ph_g_empty ^= 1;
        tc_fence_after_sync();
#pragma unroll
        for (int q = 0; q < HCW / 16; ++q) {
          uint32_t r[8];
#pragma unroll
          for (int j = 0; j < 8; ++j) r[j] = gh[q * 8 + j];
          tmem_st8(tmem_base + lane_base + GH_COL + half * (HCW / 2) + q * 8, r);
#pragma unroll
          for (int j = 0; j < 8; ++j) r[j] = gl[q * 8 + j];
          tmem_st8(tmem_base + lane_base + GL_COL + half * (HCW / 2) + q * 8, r);
        }
        tmem_st_wait();
        tc_fence_before_sync();
        __syncwarp();
        if (lane == 0) mbar_arrive(g_full);
        if (eprof) {
          g_dbg_ffn[0] += e1 - e0; g_dbg_ffn[1] += e2 - e1; g_dbg_ffn[2] += e3 - e2; g_dbg_ffn[3] += e4 - e3;
          g_dbg_ffn[4] += clock64() - e4; g_dbg_ffn[7] += 1;
        }
      }
      // ---- final epilogue of the tile: Y + b2 + residual -> LayerNorm -> stores
      const long long f0 = eprof ? clock64() : 0;
      mbar_wait(y_full, ph_y_full);
      const long long f1 = eprof ? clock64() : 0;
      ph_y_full ^= 1;
      tc_fence_after_sync();
      {
        const int64_t left = static_cast<int64_t>(p.M) - row0;
        const int rows_valid = left < 0 ? 0 : (left > 32 ? 32 : static_cast<int>(left));
        float2* xg0 = xch + (tile_parity * 2) * 128 + quad * 32 + lane;   // [parity][group][row]
        epilogue_dense<D, true>(gp, tmem_base + lane_base + Y_COL + half * (D / 2), row0, rows_valid, lane,
                                static_cast<int64_t>(half) * (D / 2), stg_all + (warp - 2) * STG_WORDS, xg0, half);
        tile_parity ^= 1;
      }
      tc_fence_before_sync();
      __syncwarp();
      if (lane == 0) mbar_arrive(y_empty);
      if (eprof) { g_dbg_ffn[5] += f1 - f0; g_dbg_ffn[6] += clock64() - f1; }
    }
  }

  tc_fence_before_sync();
  __syncthreads();
  tc_fence_after_sync();
  if (warp == 2) tmem_dealloc(tmem_base, 512);
}

template <int D>
static int launch_ffn_inst(const CUtensorMap (&tm)[6], const FfnDev& dp, cudaStream_t stream) {
  auto kern = ffn_fused_kernel<D>;
  static bool attr_set = false;
  if (!attr_set) {
    T4R_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, FFN_SMEM_BYTES));
    attr_set = true;
  }
  const int tiles = (dp.M + BM - 1) / BM;
  const int grid = tiles < num_sms() ? tiles : num_sms();
  kern<<<grid, 320, FFN_SMEM_BYTES, stream>>>(tm[0], tm[1], tm[2], tm[3], tm[4], tm[5], dp);
  T4R_LAUNCH_CHECK("ffn_fused_kernel");
  return 0;
}


bool ffn_fused_supported(int d, int hidden) { return (d == 64 || d == 128 || d == 256) && hidden % FFN_HC == 0; }

// x_planes [2, M, d], w1_planes [2, hidden, d], w2_planes [2, d, hidden]; `ep` = final epilogue (bias = b2,
// residual / residual_planes, ln_gamma/beta/eps, out_f32 / out_pre / out_planes, all with row length d).
int launch_ffn_fused(const __nv_bfloat16* x_planes, int64_t M, int d, int hidden, const __nv_bfloat16* w1_planes,
                     const float* b1, const __nv_bfloat16* w2_planes, const GemmEpilogue& ep, cudaStream_t stream) {
  T4R_REQUIRE(ffn_fused_supported(d, hidden), "ffn_fused: unsupported d=%d hidden=%d", d, hidden);
  T4R_REQUIRE(ep.ln_gamma && ep.ln_beta && b1, "ffn_fused: needs b1 and a LayerNorm epilogue");
  T4R_REQUIRE(M > 0 && M < (1ll << 31), "ffn_fused: bad M");
  CUtensorMap tm[6];
  T4R_TRY(make_tmap(&tm[0], x_planes, M, d, BM));
  T4R_TRY(make_tmap(&tm[1], x_planes + M * d, M, d, BM));
  T4R_TRY(make_tmap(&tm[2], w1_planes, hidden, d, FFN_HC));
  T4R_TRY(make_tmap(&tm[3], w1_planes + static_cast<int64_t>(hidden) * d, hidden, d, FFN_HC));
  T4R_TRY(make_tmap(&tm[4], w2_planes, d, hidden, d));
  T4R_TRY(make_tmap(&tm[5], w2_planes + static_cast<int64_t>(d) * hidden, d, hidden, d));
  FfnDev dp;
  dp.M = static_cast<int>(M);
  dp.n_chunks = hidden / FFN_HC;
  dp.b1 = b1;
  dp.ep = ep;
  {
    static int dbg = -1;
    if (dbg < 0) { const char* e = getenv("T4R_GEMM_DEBUG"); dbg = e ? atoi(e) : 0; }
    dp.ep.debug = dbg & (1 | 2 | 4 | 8 | 64);
  }
  if (d == 256) return launch_ffn_inst<256>(tm, dp, stream);
  if (d == 128) return launch_ffn_inst<128>(tm, dp, stream);
  return launch_ffn_inst<64>(tm, dp, stream);
}

}  // namespace t4r
