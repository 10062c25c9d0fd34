// t4r_internal.h -- host-side declarations shared by the translation units of
// libt4r_b200.so (not part of the public C ABI).
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdint.h>
#include <stddef.h>
#include <atomic>

#include "../../include/t4r_b200.h"

namespace t4r {

void set_error(const char* fmt, ...);
int cuda_fail(cudaError_t e, const char* what);  // records message, returns T4R_ERR_CUDA
extern std::atomic<long long> g_launches;

#define T4R_CUDA(expr)                                           \
  do {                                                           \
    cudaError_t _e = (expr);                                     \
    if (_e != cudaSuccess) return ::t4r::cuda_fail(_e, #expr);   \
  } while (0)
#define T4R_LAUNCH_CHECK(name)                                   \
  do {                                                           \
    ::t4r::g_launches.fetch_add(1, std::memory_order_relaxed);   \
    cudaError_t _e = cudaGetLastError();                         \
    if (_e != cudaSuccess) return ::t4r::cuda_fail(_e, name);    \
  } while (0)
#define T4R_REQUIRE(cond, ...)                                   \
  do {                                                           \
    if (!(cond)) {                                               \
      ::t4r::set_error(__VA_ARGS__);                             \
      return T4R_ERR_INVALID;                                    \
    }                                                            \
  } while (0)
#define T4R_TRY(expr)                                            \
  do {                                                           \
    int _rc = (expr);                                            \
    if (_rc != 0) return _rc;                                    \
  } while (0)

inline int round_up(int x, int m) { return (x + m - 1) / m * m; }
inline int64_t round_up64i(int64_t x, int64_t m) { return (x + m - 1) / m * m; }

// ---------------------------------------------------------------------------
// tcgen05 GEMM  C[M,N] = epilogue(A[M,Kp] * B[N,Kp]^T), A/B in split-bf16 planes
// ---------------------------------------------------------------------------
struct GemmEpilogue {
  // dense epilogue
  const float* bias = nullptr;         // [N]
  int act = 0;                         // T4R_ACT_*
  const uint8_t* row_code = nullptr;   // [M]
  const float* mask_vec = nullptr;     // [N]
  const float* residual = nullptr;     // [M, ldr]
  int ldr = 0;
  const __nv_bfloat16* residual_planes = nullptr;  // alternative residual as split planes [2, rows, ldrp] (hi + lo)
  int ldrp = 0;
  int64_t residual_plane_stride = 0;
  const float* ln_gamma = nullptr;     // LayerNorm over N (requires BN == N)
  const float* ln_beta = nullptr;
  float ln_eps = 0.f;
  float* out_pre = nullptr;            // [M, ldp]
  int ldp = 0;
  float* out_f32 = nullptr;            // [M, ldo]
  int64_t ldo = 0;
  float out_scale = 1.f;               // applied to out_f32 (logit materialisation)
  __nv_bfloat16* out_planes = nullptr; // [2, plane_rows, ldpl]
  int ldpl = 0;
  int64_t plane_stride = 0;            // elements between hi and lo plane
  // head epilogue (online log-sum-exp partials per (column tile, row))
  bool head = false;
  float* part_m = nullptr;             // [n_tiles, part_ld]   running max  (log2 domain)
  float* part_s = nullptr;             // [n_tiles, part_ld]   sum of 2^(x - max)
  float* part_z = nullptr;             // [n_tiles, part_ld]   plain sum of the scaled logits (label smoothing) or null
  int part_ld = 0;
  float inv_tau = 1.f;
  const float* col_bias = nullptr;     // [N]
  const int64_t* col_ids = nullptr;    // [N]
  const int32_t* hit_col = nullptr;    // [M] column holding the row's own label (accidental hit) or -1; replaces col_ids
  const int64_t* row_label = nullptr;  // [M]
  float hit_value = 0.f;
  const float* row_tgt = nullptr;      // [M] label logit (already scaled), for ranks
  int* row_rank = nullptr;             // [M] atomically accumulated
  int64_t col_offset = 0;              // global class id of column 0 (shards)
  bool head_resident = false;          // run head_resident_kernel: ONE partial per (column chunk of 16 tiles, half, row)
  const float* row_scale = nullptr;    // [M] nprod = 2: 1 / (power-of-two scale of A's row)
  const float* col_scale = nullptr;    // [N] nprod = 2: 1 / (power-of-two scale of B's row)
  int debug = 0;                       // T4R_GEMM_DEBUG: 1 = epilogue skips all global loads/stores (timing experiments)
};

struct GemmProblem {
  int64_t M = 0;          // rows of A (capacity)
  int64_t N = 0;          // rows of B / output columns
  int Kp = 0;             // padded K, multiple of 64
  const __nv_bfloat16* a_planes = nullptr;  // [2, a_rows, Kp]
  int64_t a_rows = 0;                       // rows per plane of A (plane stride = a_rows*Kp)
  const __nv_bfloat16* b_planes = nullptr;  // [2, b_rows, Kp]
  int64_t b_rows = 0;
  const int32_t* m_dev = nullptr;
  int nprod = 3;
  int bn = 0;             // 0 = choose
};

int launch_gemm(const GemmProblem& pb, const GemmEpilogue& ep, cudaStream_t stream);
int head_resident_partials(int64_t M, int64_t V, int Kp);  // > 0: the resident-A head kernel will run (t4r_gemm.cu)

// fused feed-forward block (t4r_gemm.cu): Y = epilogue(gelu(X W1^T + b1) W2^T), intermediate kept in TMEM
bool ffn_fused_supported(int d, int hidden);
int launch_ffn_fused(const __nv_bfloat16* x_planes, int64_t M, int d, int hidden, const __nv_bfloat16* w1_planes,
                     const float* b1, const __nv_bfloat16* w2_planes, const GemmEpilogue& ep, cudaStream_t stream);

// ---------------------------------------------------------------------------
// SIMT kernels (t4r_kernels.cu)
// ---------------------------------------------------------------------------
int launch_split_planes(const float* x, int64_t rows, int K, int64_t ld, const uint8_t* row_code,
                        const float* mask_vec, float* out_f32, __nv_bfloat16* planes, cudaStream_t s);
// all layers in one launch: r_out [n_layer, 2L, d] fp32, r_planes [n_layer, 2, 2L, d] bf16 (or null)
int launch_rel_pos_proj(const float* const* wr_layers, int n_layer, int L, int d, float* r_out,
                        __nv_bfloat16* r_planes, cudaStream_t s);
// tensor-path attention (t4r_attn_mma.cu): operands as split planes
bool attn_mma_supported(int L, int d, int H, bool rel);
int launch_attn_mma(bool rel, const __nv_bfloat16* qkv_planes, int64_t qkv_plane_stride, const __nv_bfloat16* r_planes,
                    int64_t r_plane_stride, const float* rw, const float* rr, int B, int L, int d, int H,
                    __nv_bfloat16* out_planes, int64_t out_plane_stride, cudaStream_t s);
int launch_attn_mma_plm(const __nv_bfloat16* qkv_planes, int64_t qkv_plane_stride, const __nv_bfloat16* r_planes,
                        int64_t r_plane_stride, const float* rw, const float* rr, int B, int L, int d, int H,
                        __nv_bfloat16* out_planes, int64_t out_plane_stride, const uint8_t* plm_mask, cudaStream_t s);
int launch_xlnet_attn(const float* qkv /*[M, 3d]*/, const float* r /*[2L, d]*/, const float* rw, const float* rr,
                      int B, int L, int d, int H, __nv_bfloat16* out_planes, int64_t plane_stride, cudaStream_t s);
int launch_causal_attn(const float* qkv, int B, int L, int d, int H, __nv_bfloat16* out_planes,
                       int64_t plane_stride, cudaStream_t s);
int launch_addpos_ln(const float* x, const float* wpe, int B, int L, int d, const float* g, const float* b,
                     float eps, float* h_out, __nv_bfloat16* planes, int64_t plane_stride, cudaStream_t s);
int launch_head_reduce(const float* part_m, const float* part_s, const float* part_z, int n_tiles, int part_ld,
                       int T_cap, const int32_t* t_dev, const float* pos_logit, const float* row_tgt_in,
                       float label_smoothing, int64_t n_classes, float* row_lse, float* row_loss, float* loss,
                       float* scratch, cudaStream_t s);
int launch_hit_cols(const int64_t* col_ids, int64_t S, const int64_t* labels, int T_cap, const int32_t* t_dev,
                    int32_t* hit_col, cudaStream_t s);
int launch_target_logit(const float* xt, const float* w, const int64_t* labels, int T_cap, const int32_t* t_dev,
                        int De, int64_t v_offset, int64_t V, const float* class_bias, float inv_tau, float* out,
                        cudaStream_t s);

}  // namespace t4r
