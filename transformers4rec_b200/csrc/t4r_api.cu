// t4r_api.cu -- C-ABI entry points that compose the kernels: error reporting,
// dense layer, XLNet / GPT-2 encoders, next-item head.  Host orchestration only;
// every launch goes to the caller's stream, nothing synchronises.
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include "t4r_common.cuh"
#include <stddef.h>

#include "t4r_internal.h"

namespace t4r {

static thread_local char g_err[1024] = "";
std::atomic<long long> g_launches{0};

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}
int cuda_fail(cudaError_t e, const char* what) {
  set_error("CUDA error %d (%s) at %s", static_cast<int>(e), cudaGetErrorString(e), what);
  return T4R_ERR_CUDA;
}

// bump allocator over the caller's workspace
struct Arena {
  uint8_t* base;
  size_t size;
  size_t off = 0;
  bool ok = true;
  Arena(void* p, size_t n) : base(static_cast<uint8_t*>(p)), size(n) {}
  template <typename T>
  T* take(size_t count) {
    const size_t bytes = (count * sizeof(T) + 255) / 256 * 256;
    if (off + bytes > size) {
      ok = false;
      return nullptr;
    }
    T* r = reinterpret_cast<T*>(base + off);
    off += bytes;
    return r;
  }
};
static size_t pad256(size_t b) { return (b + 255) / 256 * 256; }

// plain fp32 reference GEMM (debug / tests): C[M,N] = A[M,K] * B[N,K]^T + bias
__global__ void __launch_bounds__(256)
sgemm_nt_kernel(const float* __restrict__ A, const float* __restrict__ B, const float* __restrict__ bias,
                float* __restrict__ C, int64_t M, int N, int K) {
  __shared__ float As[16][17];
  __shared__ float Bs[16][17];
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
  const int64_t row = static_cast<int64_t>(blockIdx.y) * 16 + ty;
  const int col = blockIdx.x * 16 + tx;
  float acc = 0.f;
  for (int k0 = 0; k0 < K; k0 += 16) {
    As[ty][tx] = (row < M && k0 + tx < K) ? A[row * K + k0 + tx] : 0.f;
    const int brow = blockIdx.x * 16 + ty;
    Bs[ty][tx] = (brow < N && k0 + tx < K) ? B[static_cast<int64_t>(brow) * K + k0 + tx] : 0.f;
    __syncthreads();
#pragma unroll
    for (int k = 0; k < 16; ++k) acc = fmaf(As[ty][k], Bs[tx][k], acc);
    __syncthreads();
  }
  if (row < M && col < N) C[row * N + col] = acc + (bias ? bias[col] : 0.f);
}

}  // namespace t4r

using namespace t4r;

extern "C" const char* t4r_last_error(void) { return t4r::g_err; }
extern "C" int t4r_version(void) { return 100; }
extern "C" long long t4r_launch_count(void) { return t4r::g_launches.load(); }

extern "C" int t4r_debug_sgemm_nt(const float* A, const float* B, const float* bias, float* C, int64_t M, int N, int K,
                                  void* stream) {
  T4R_REQUIRE(A && B && C && M > 0 && N > 0 && K > 0, "debug_sgemm_nt: bad arguments");
  dim3 grid((N + 15) / 16, static_cast<unsigned>((M + 15) / 16));
  sgemm_nt_kernel<<<grid, 256, 0, static_cast<cudaStream_t>(stream)>>>(A, B, bias, C, M, N, K);
  T4R_LAUNCH_CHECK("sgemm_nt_kernel");
  return 0;
}

// ----------------------------------------------------------------------------
// K2 dense layer
// ----------------------------------------------------------------------------
extern "C" int t4r_linear_fwd(const t4r_linear_args* a, void* stream) {
  T4R_REQUIRE(a != nullptr, "linear_fwd: null args");
  T4R_REQUIRE(a->M > 0 && a->N > 0 && a->K > 0 && a->x_planes && a->w_planes, "linear_fwd: bad shape/pointers");
  T4R_REQUIRE(a->ln_gamma == nullptr || a->N % 64 == 0, "linear_fwd: LayerNorm needs N in {64,128,256} (got %d)", a->N);
  T4R_REQUIRE(a->out_f32 || a->out_planes || a->out_pre_ln, "linear_fwd: no output requested");
  T4R_REQUIRE(a->row_code == nullptr || a->mask_vec != nullptr, "linear_fwd: row_code needs mask_vec");
  T4R_REQUIRE((a->ln_gamma == nullptr) == (a->ln_beta == nullptr), "linear_fwd: ln_gamma and ln_beta go together");
  T4R_REQUIRE(a->out_pre_ln == nullptr || a->ln_gamma != nullptr, "linear_fwd: out_pre_ln needs LayerNorm");
  const int Kp = t4r_round_up64(a->K);
  GemmProblem pb;
  pb.M = a->M;
  pb.N = a->N;
  pb.Kp = Kp;
  pb.a_planes = static_cast<const __nv_bfloat16*>(a->x_planes);
  pb.a_rows = a->M;
  pb.b_planes = static_cast<const __nv_bfloat16*>(a->w_planes);
  pb.b_rows = a->N;
  pb.m_dev = a->m_dev;
  pb.nprod = a->nprod ? a->nprod : 3;
  GemmEpilogue ep;
  ep.bias = a->bias;
  ep.act = a->act;
  ep.row_code = a->row_code;
  ep.mask_vec = a->mask_vec;
  ep.residual = a->residual;
  ep.ldr = a->N;
  ep.ln_gamma = a->ln_gamma;
  ep.ln_beta = a->ln_beta;
  ep.ln_eps = a->ln_eps;
  ep.out_pre = a->out_pre_ln;
  ep.ldp = a->N;
  ep.out_f32 = a->out_f32;
  ep.ldo = a->N;
  ep.out_planes = static_cast<__nv_bfloat16*>(a->out_planes);
  ep.ldpl = t4r_round_up64(a->N);
  ep.plane_stride = a->M * static_cast<int64_t>(ep.ldpl);
  return launch_gemm(pb, ep, static_cast<cudaStream_t>(stream));
}

extern "C" int t4r_ffn_fwd(const void* x_planes, int64_t M, int d, int hidden, const void* w1_planes, const float* b1,
                           const void* w2_planes, const float* b2, const float* residual, const float* ln_gamma,
                           const float* ln_beta, float ln_eps, float* out_pre_ln, float* out_f32, void* out_planes,
                           void* stream) {
  T4R_REQUIRE(x_planes && w1_planes && w2_planes && b1 && ln_gamma && ln_beta && M > 0, "ffn_fwd: bad arguments");
  T4R_REQUIRE(out_f32 || out_planes || out_pre_ln, "ffn_fwd: no output requested");
  T4R_REQUIRE(ffn_fused_supported(d, hidden), "ffn_fwd: d must be 64, 128 or 256 and hidden a multiple of 128 (got %d, %d)",
              d, hidden);
  GemmEpilogue ep;
  ep.bias = b2;
  if (residual) { ep.residual = residual; ep.ldr = d; }
  else { ep.residual_planes = static_cast<const __nv_bfloat16*>(x_planes); ep.ldrp = d; ep.residual_plane_stride = M * d; }
  ep.ln_gamma = ln_gamma; ep.ln_beta = ln_beta; ep.ln_eps = ln_eps;
  ep.out_pre = out_pre_ln; ep.ldp = d;
  ep.out_f32 = out_f32; ep.ldo = d;
  ep.out_planes = static_cast<__nv_bfloat16*>(out_planes); ep.ldpl = d; ep.plane_stride = M * d;
  return launch_ffn_fused(static_cast<const __nv_bfloat16*>(x_planes), M, d, hidden,
                          static_cast<const __nv_bfloat16*>(w1_planes), b1, static_cast<const __nv_bfloat16*>(w2_planes), ep,
                          static_cast<cudaStream_t>(stream));
}

// ----------------------------------------------------------------------------
// XLNet encoder
// ----------------------------------------------------------------------------
extern "C" size_t t4r_xlnet_encoder_workspace_bytes(int B, int L, int d, int n_head) {
  (void)n_head;
  const size_t M = static_cast<size_t>(B) * L;
  size_t b = 0;
  b += pad256(M * 3 * d * 4);        // qkv fp32
  b += pad256(static_cast<size_t>(T4R_MAX_FEATURES) * 2 * L * d * 4);      // r, all layers
  b += pad256(static_cast<size_t>(T4R_MAX_FEATURES) * 2 * 2 * L * d * 2);  // r planes, all layers
  b += pad256(2 * M * d * 2);        // attention output planes
  b += pad256(M * d * 4);            // h1 fp32
  b += pad256(2 * M * d * 2);        // h1 planes
  b += pad256(2 * M * d * 2);        // x planes (when split internally)
  b += 2 * (pad256(M * d * 4) + pad256(2 * M * d * 2));  // layer io ping-pong
  return b + 1024;
}

// plm_mask != nullptr: the two-stream PLM forward -- B counts the stacked row sessions (2 x the real batch: h rows, then
// g rows) and only the attention step knows about the streams (everything else is row-wise).
static int xlnet_encoder_impl(const t4r_xlnet_layer* layers, int n_layer, int B, int L, int d, int n_head,
                              float ln_eps, const float* x_f32, const void* x_planes, float* out_f32,
                              void* out_planes, void* workspace, size_t workspace_bytes, void* stream,
                              const uint8_t* plm_mask);
extern "C" int t4r_xlnet_encoder_fwd(const t4r_xlnet_layer* layers, int n_layer, int B, int L, int d, int n_head,
                                     float ln_eps, const float* x_f32, const void* x_planes, float* out_f32,
                                     void* out_planes, void* workspace, size_t workspace_bytes, void* stream) {
  return xlnet_encoder_impl(layers, n_layer, B, L, d, n_head, ln_eps, x_f32, x_planes, out_f32, out_planes, workspace,
                            workspace_bytes, stream, nullptr);
}
extern "C" int t4r_xlnet_encoder_plm_fwd(const t4r_xlnet_layer* layers, int n_layer, int B, int L, int d, int n_head,
                                         float ln_eps, const float* x_f32, const uint8_t* perm_mask, float* out_f32,
                                         void* workspace, size_t workspace_bytes, void* stream) {
  T4R_REQUIRE(perm_mask != nullptr, "xlnet_encoder_plm: perm_mask is required");
  T4R_REQUIRE(attn_mma_supported(L, d, n_head, true),
              "xlnet_encoder_plm: needs the tensor-path attention (L + 2 <= 32, or <= 64 with T4R_ATTN_MMA64=1); L=%d", L);
  return xlnet_encoder_impl(layers, n_layer, 2 * B, L, d, n_head, ln_eps, x_f32, nullptr, out_f32, nullptr, workspace,
                            workspace_bytes, stream, perm_mask);
}
static int xlnet_encoder_impl(const t4r_xlnet_layer* layers, int n_layer, int B, int L, int d, int n_head,
                              float ln_eps, const float* x_f32, const void* x_planes, float* out_f32,
                              void* out_planes, void* workspace, size_t workspace_bytes, void* stream,
                              const uint8_t* plm_mask) {
  T4R_REQUIRE(layers && n_layer >= 1 && B > 0 && L > 0 && x_f32 && out_f32 && workspace, "xlnet_encoder: bad arguments");
  T4R_REQUIRE(d == 64 || d == 128 || d == 256, "xlnet_encoder: d_model must be 64, 128 or 256 (got %d)", d);
  T4R_REQUIRE(workspace_bytes >= t4r_xlnet_encoder_workspace_bytes(B, L, d, n_head), "xlnet_encoder: workspace too small");
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const int64_t M = static_cast<int64_t>(B) * L;
  Arena ar(workspace, workspace_bytes);
  float* qkv = ar.take<float>(M * 3 * d);
  float* rbuf = ar.take<float>(static_cast<size_t>(T4R_MAX_FEATURES) * 2 * L * d);
  __nv_bfloat16* r_p = ar.take<__nv_bfloat16>(static_cast<size_t>(T4R_MAX_FEATURES) * 2 * 2 * L * d);
  __nv_bfloat16* attn_p = ar.take<__nv_bfloat16>(2 * M * d);
  float* h1 = ar.take<float>(M * d);
  // tensor-path attention (mma.sync) consumes q|k|v as split planes; the SIMT kernel (L > 30) fp32
  static int force_simt = -1;
  if (force_simt < 0) { const char* e = getenv("T4R_ATTN_SIMT"); force_simt = (e && atoi(e)) ? 1 : 0; }
  const bool tc_attn = !force_simt && attn_mma_supported(L, d, n_head, true);
  __nv_bfloat16* qkv_p = reinterpret_cast<__nv_bfloat16*>(qkv);  // same bytes: [2, M, 3d] bf16
  __nv_bfloat16* h1_p = ar.take<__nv_bfloat16>(2 * M * d);
  __nv_bfloat16* x_p_own = ar.take<__nv_bfloat16>(2 * M * d);
  float* io_f[2];
  __nv_bfloat16* io_p[2];
  for (int i = 0; i < 2; ++i) {
    io_f[i] = ar.take<float>(M * d);
    io_p[i] = ar.take<__nv_bfloat16>(2 * M * d);
  }
  T4R_REQUIRE(ar.ok, "xlnet_encoder: workspace carve-up failed");

  const float* cur_f = x_f32;
  const __nv_bfloat16* cur_p = static_cast<const __nv_bfloat16*>(x_planes);
  if (!cur_p) {
    T4R_TRY(launch_split_planes(x_f32, M, d, d, nullptr, nullptr, nullptr, x_p_own, s));
    cur_p = x_p_own;
  }
  // R_l = pos_emb @ Wr_l (HF:xlnet:262) depends on the weights only: all layers in one launch, once
  // per forward for the whole batch (the reference recomputes it per batch element and layer)
  T4R_REQUIRE(n_layer <= T4R_MAX_FEATURES, "xlnet_encoder: at most %d layers", T4R_MAX_FEATURES);
  {
    const float* wrs[T4R_MAX_FEATURES];
    for (int li = 0; li < n_layer; ++li) wrs[li] = layers[li].wr;
    T4R_TRY(launch_rel_pos_proj(wrs, n_layer, L, d, rbuf, tc_attn ? r_p : nullptr, s));
  }
  const float* in_f = x_f32;
  const __nv_bfloat16* in_p = cur_p;
  for (int li = 0; li < n_layer; ++li) {
    const t4r_xlnet_layer& w = layers[li];
    const bool last = (li == n_layer - 1);
    const float* rbuf_l = rbuf + static_cast<size_t>(li) * 2 * L * d;
    const __nv_bfloat16* r_p_l = r_p + static_cast<size_t>(li) * 4 * L * d;
    float* dst_f = last ? out_f32 : nullptr;
    __nv_bfloat16* dst_p = last ? static_cast<__nv_bfloat16*>(out_planes) : io_p[li & 1];
    // Q | K | V projections (HF:xlnet:253-259), one GEMM over the fused [3d, d] weight
    {
      GemmProblem pb;
      pb.M = M; pb.N = 3 * d; pb.Kp = d;
      pb.a_planes = in_p; pb.a_rows = M;
      pb.b_planes = static_cast<const __nv_bfloat16*>(w.wqkv_planes); pb.b_rows = 3 * d;
      GemmEpilogue ep;
      if (tc_attn) { ep.out_planes = qkv_p; ep.ldpl = 3 * d; ep.plane_stride = M * 3 * d; }
      else { ep.out_f32 = qkv; ep.ldo = 3 * d; }
      T4R_TRY(launch_gemm(pb, ep, s));
    }
    // relative attention core (HF:xlnet:95-140)
    if (plm_mask) {
      T4R_REQUIRE(tc_attn, "xlnet_encoder_plm: the FFMA attention fallback has no two-stream form (unset T4R_ATTN_SIMT)");
      T4R_TRY(launch_attn_mma_plm(qkv_p, M * 3 * d, r_p_l, static_cast<int64_t>(2) * L * d, w.r_w_bias, w.r_r_bias, B / 2,
                                  L, d, n_head, attn_p, M * d, plm_mask, s));
    } else if (tc_attn)
      T4R_TRY(launch_attn_mma(true, qkv_p, M * 3 * d, r_p_l, static_cast<int64_t>(2) * L * d, w.r_w_bias, w.r_r_bias, B,
                              L, d, n_head, attn_p, M * d, s));
    else
      T4R_TRY(launch_xlnet_attn(qkv, rbuf_l, w.r_w_bias, w.r_r_bias, B, L, d, n_head, attn_p, M * d, s));
    // post_attention: h1 = LN(x + attn @ Wo^T) (HF:xlnet:142-152)
    {
      GemmProblem pb;
      pb.M = M; pb.N = d; pb.Kp = d;
      pb.a_planes = attn_p; pb.a_rows = M;
      pb.b_planes = static_cast<const __nv_bfloat16*>(w.wo_planes); pb.b_rows = d;
      GemmEpilogue ep;
      // residual: the caller's fp32 x for the first layer, afterwards the split planes of the
      // previous layer's output (hi + lo, exact to 16 mantissa bits) -- no fp32 copy of the
      // residual stream is written between layers (the store path bounds these epilogues)
      if (in_f) { ep.residual = in_f; ep.ldr = d; }
      else { ep.residual_planes = in_p; ep.ldrp = d; ep.residual_plane_stride = M * d; }
      ep.ln_gamma = w.ln1_gamma; ep.ln_beta = w.ln1_beta; ep.ln_eps = ln_eps;
      ep.out_planes = h1_p; ep.ldpl = d; ep.plane_stride = M * d;
      T4R_TRY(launch_gemm(pb, ep, s));
    }
    // feed-forward (HF:xlnet:297-305): out = LN(h1 + gelu(h1 W1^T + b1) W2^T + b2)
    {
      GemmEpilogue ep;
      ep.bias = w.b2;
      ep.residual_planes = h1_p; ep.ldrp = d; ep.residual_plane_stride = M * d;
      ep.ln_gamma = w.ln2_gamma; ep.ln_beta = w.ln2_beta; ep.ln_eps = ln_eps;
      ep.out_f32 = dst_f; ep.ldo = d;
      ep.out_planes = dst_p; ep.ldpl = d; ep.plane_stride = M * d;
      T4R_TRY(launch_ffn_fused(h1_p, M, d, 4 * d, static_cast<const __nv_bfloat16*>(w.w1_planes), w.b1,
                               static_cast<const __nv_bfloat16*>(w.w2_planes), ep, s));
    }
    in_f = dst_f;
    in_p = dst_p;
  }
  return 0;
}

// ----------------------------------------------------------------------------
// GPT-2 encoder
// ----------------------------------------------------------------------------
extern "C" size_t t4r_gpt2_encoder_workspace_bytes(int B, int L, int d, int n_head) {
  (void)n_head;
  const size_t M = static_cast<size_t>(B) * L;
  size_t b = 0;
  b += pad256(M * 3 * d * 4);      // qkv
  b += pad256(2 * M * d * 2);      // attention planes
  b += 2 * pad256(M * d * 4);      // residual stream ping-pong
  b += 2 * pad256(2 * M * d * 2);  // LN output planes ping-pong
  return b + 1024;
}

extern "C" int t4r_gpt2_encoder_fwd(const t4r_gpt2_layer* layers, int n_layer, int B, int L, int d, int n_head,
                                    float ln_eps, const float* wpe, const float* lnf_gamma, const float* lnf_beta,
                                    const float* x_f32, float* out_f32, void* out_planes, void* workspace,
                                    size_t workspace_bytes, void* stream) {
  T4R_REQUIRE(layers && n_layer >= 1 && B > 0 && L > 0 && x_f32 && out_f32 && workspace && wpe && lnf_gamma && lnf_beta,
              "gpt2_encoder: bad arguments");
  T4R_REQUIRE(d == 64 || d == 128 || d == 256, "gpt2_encoder: d_model must be 64, 128 or 256 (got %d)", d);
  T4R_REQUIRE(workspace_bytes >= t4r_gpt2_encoder_workspace_bytes(B, L, d, n_head), "gpt2_encoder: workspace too small");
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const int64_t M = static_cast<int64_t>(B) * L;
  Arena ar(workspace, workspace_bytes);
  float* qkv = ar.take<float>(M * 3 * d);
  __nv_bfloat16* attn_p = ar.take<__nv_bfloat16>(2 * M * d);
  float* hbuf[2] = {ar.take<float>(M * d), ar.take<float>(M * d)};
  __nv_bfloat16* lnp[2] = {ar.take<__nv_bfloat16>(2 * M * d), ar.take<__nv_bfloat16>(2 * M * d)};
  T4R_REQUIRE(ar.ok, "gpt2_encoder: workspace carve-up failed");
  static int force_simt = -1;
  if (force_simt < 0) { const char* e = getenv("T4R_ATTN_SIMT"); force_simt = (e && atoi(e)) ? 1 : 0; }
  const bool tc_attn = !force_simt && attn_mma_supported(L, d, n_head, false);
  __nv_bfloat16* qkv_p = reinterpret_cast<__nv_bfloat16*>(qkv);

  // h = x + wpe[0:L]; a = ln_1^{(0)}(h)   (HF:gpt2:579-585, :272)
  int hc = 0, pc = 0;
  T4R_TRY(launch_addpos_ln(x_f32, wpe, B, L, d, layers[0].ln1_gamma, layers[0].ln1_beta, ln_eps, hbuf[hc], lnp[pc],
                           M * d, s));
  for (int li = 0; li < n_layer; ++li) {
    const t4r_gpt2_layer& w = layers[li];
    const bool last = (li == n_layer - 1);
    {  // c_attn (HF:gpt2:188)
      GemmProblem pb;
      pb.M = M; pb.N = 3 * d; pb.Kp = d;
      pb.a_planes = lnp[pc]; pb.a_rows = M;
      pb.b_planes = static_cast<const __nv_bfloat16*>(w.wqkv_planes); pb.b_rows = 3 * d;
      GemmEpilogue ep;
      ep.bias = w.bqkv;
      if (tc_attn) { ep.out_planes = qkv_p; ep.ldpl = 3 * d; ep.plane_stride = M * 3 * d; }
      else { ep.out_f32 = qkv; ep.ldo = 3 * d; }
      T4R_TRY(launch_gemm(pb, ep, s));
    }
    if (tc_attn)
      T4R_TRY(launch_attn_mma(false, qkv_p, M * 3 * d, nullptr, 0, nullptr, nullptr, B, L, d, n_head, attn_p, M * d, s));
    else
      T4R_TRY(launch_causal_attn(qkv, B, L, d, n_head, attn_p, M * d, s));
    {  // h = h + attn c_proj + b; m = ln_2(h)   (HF:gpt2:284-290)
      GemmProblem pb;
      pb.M = M; pb.N = d; pb.Kp = d;
      pb.a_planes = attn_p; pb.a_rows = M;
      pb.b_planes = static_cast<const __nv_bfloat16*>(w.wo_planes); pb.b_rows = d;
      GemmEpilogue ep;
      ep.bias = w.bo;
      ep.residual = hbuf[hc]; ep.ldr = d;
      ep.ln_gamma = w.ln2_gamma; ep.ln_beta = w.ln2_beta; ep.ln_eps = ln_eps;
      ep.out_pre = hbuf[hc ^ 1]; ep.ldp = d;
      ep.out_planes = lnp[pc ^ 1]; ep.ldpl = d; ep.plane_stride = M * d;
      T4R_TRY(launch_gemm(pb, ep, s));
      hc ^= 1; pc ^= 1;
    }
    {  // c_fc + gelu (HF:gpt2:237-239); h = h + ff c_proj + b; next = ln_1^{(i+1)}(h) or ln_f(h)  (HF:gpt2:305-309, :617)
      GemmEpilogue ep;
      ep.bias = w.b2;
      ep.residual = hbuf[hc]; ep.ldr = d;
      ep.ln_eps = ln_eps;
      if (last) {
        ep.ln_gamma = lnf_gamma; ep.ln_beta = lnf_beta;
        ep.out_f32 = out_f32; ep.ldo = d;
        if (out_planes) { ep.out_planes = static_cast<__nv_bfloat16*>(out_planes); ep.ldpl = d; ep.plane_stride = M * d; }
      } else {
        ep.ln_gamma = layers[li + 1].ln1_gamma; ep.ln_beta = layers[li + 1].ln1_beta;
        ep.out_pre = hbuf[hc ^ 1]; ep.ldp = d;
        ep.out_planes = lnp[pc ^ 1]; ep.ldpl = d; ep.plane_stride = M * d;
      }
      T4R_TRY(launch_ffn_fused(lnp[pc], M, d, 4 * d, static_cast<const __nv_bfloat16*>(w.w1_planes), w.b1,
                               static_cast<const __nv_bfloat16*>(w.w2_planes), ep, s));
      hc ^= 1; pc ^= 1;
    }
  }
  return 0;
}

// ----------------------------------------------------------------------------
// head
// ----------------------------------------------------------------------------
static const int kHeadBN = 256;

extern "C" size_t t4r_head_workspace_bytes(int T_cap, int64_t V, int De) {
  (void)De;
  const size_t part_ld = static_cast<size_t>((T_cap + 127) / 128) * 128;
  const size_t n_tiles = 2 * static_cast<size_t>((V + kHeadBN - 1) / kHeadBN);  // two column halves per tile
  return 3 * pad256(n_tiles * part_ld * 4) + pad256(3 * 64 * part_ld * 4) + pad256(part_ld * 4) + 1024;
}

extern "C" size_t t4r_sizeof_struct(int which) {
  switch (which) {
    case 0: return sizeof(t4r_head_args);
    case 1: return sizeof(t4r_linear_args);
    case 2: return sizeof(t4r_feature_list);
    case 3: return sizeof(t4r_feature);
    case 4: return sizeof(t4r_xlnet_layer);
    case 5: return sizeof(t4r_gpt2_layer);
    default: return 0;
  }
}
extern "C" size_t t4r_head_args_last_offset(void) { return offsetof(t4r_head_args, col_ids_sorted_unique); }

extern "C" int t4r_head_softmax_ce_fwd(const t4r_head_args* a, void* stream) {
  T4R_REQUIRE(a != nullptr, "head: null args");
  T4R_REQUIRE(a->T_cap > 0 && a->V > 0 && a->De > 0 && a->xt_planes && a->w_planes && a->workspace,
              "head: bad shape/pointers");
  T4R_REQUIRE(a->row_loss != nullptr, "head: row_loss output is required");
  T4R_REQUIRE(a->pos_logit != nullptr || (a->xt_f32 && a->w_f32 && a->labels && a->row_tgt),
              "head: full softmax needs xt_f32, w_f32, labels and row_tgt");
  T4R_REQUIRE(a->row_rank == nullptr || a->labels != nullptr, "head: ranks need labels");
  T4R_REQUIRE(a->workspace_bytes >= t4r_head_workspace_bytes(a->T_cap, a->V, a->De), "head: workspace too small");
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const int part_ld = (a->T_cap + 127) / 128 * 128;
  int n_tiles = 2 * static_cast<int>((a->V + kHeadBN - 1) / kHeadBN);  // partials per (tile, column half)
  const int res_parts = head_resident_partials(a->T_cap, a->V, t4r_round_up64(a->De));
  if (res_parts > 0) n_tiles = res_parts;  // resident-A kernel: one partial per (16-tile column chunk, half)
  Arena ar(a->workspace, a->workspace_bytes);
  float* part_m = ar.take<float>(static_cast<size_t>(n_tiles) * part_ld);
  float* part_s = ar.take<float>(static_cast<size_t>(n_tiles) * part_ld);
  float* scratch = ar.take<float>(static_cast<size_t>(3) * 64 * part_ld);
  int32_t* hit_col = reinterpret_cast<int32_t*>(ar.take<float>(part_ld));
  float* part_z = nullptr;
  if (a->label_smoothing != 0.f) {
    T4R_REQUIRE(a->pos_logit == nullptr && a->v_offset == 0, "head: label smoothing needs the unsharded full softmax");
    part_z = ar.take<float>(static_cast<size_t>(n_tiles) * part_ld);
  }
  T4R_REQUIRE(ar.ok, "head: workspace carve-up failed");
  const float inv_tau = a->inv_temperature != 0.f ? a->inv_temperature : 1.f;

  if (!a->pos_logit) {
    // exact fp32 label logit (0 when the label lives in another shard)
    T4R_TRY(launch_target_logit(a->xt_f32, a->w_f32, a->labels, a->T_cap, a->t_dev, a->De, a->v_offset, a->V, nullptr,
                                inv_tau, a->row_tgt, s));
  }
  if (a->row_rank) T4R_CUDA(cudaMemsetAsync(a->row_rank, 0, sizeof(int32_t) * a->T_cap, s));

  GemmProblem pb;
  pb.M = a->T_cap;
  pb.N = a->V;
  pb.Kp = t4r_round_up64(a->De);
  pb.a_planes = static_cast<const __nv_bfloat16*>(a->xt_planes);
  pb.a_rows = a->T_cap;
  pb.b_planes = static_cast<const __nv_bfloat16*>(a->w_planes);
  pb.b_rows = a->V;
  pb.m_dev = a->t_dev;
  pb.nprod = a->nprod ? a->nprod : 3;
  pb.bn = kHeadBN;
  GemmEpilogue ep;
  ep.head = true;
  ep.part_m = part_m;
  ep.part_s = part_s;
  ep.part_z = part_z;
  ep.part_ld = part_ld;
  ep.inv_tau = inv_tau;
  ep.col_bias = a->col_bias;
  ep.col_ids = a->col_ids;
  if (a->col_ids && a->col_ids_sorted_unique && a->labels && a->V < (1ll << 31)) {
    // one binary search per row instead of one 8-byte id comparison per logit
    T4R_TRY(launch_hit_cols(a->col_ids, a->V, a->labels, a->T_cap, a->t_dev, hit_col, s));
    ep.hit_col = hit_col;
    ep.col_ids = nullptr;
  }
  ep.row_label = a->labels;
  ep.hit_value = a->hit_value;
  ep.row_tgt = a->rank_tgt ? a->rank_tgt : a->row_tgt;
  ep.row_rank = a->row_rank;
  ep.col_offset = a->v_offset;
  ep.head_resident = res_parts > 0;
  if (pb.nprod == 2) {
    T4R_REQUIRE(a->xt_inv_scale && a->w_inv_scale, "head: nprod = 2 needs xt_inv_scale and w_inv_scale");
    ep.row_scale = a->xt_inv_scale;
    ep.col_scale = a->w_inv_scale;
  }
  if (a->ev_gemm_start) T4R_CUDA(cudaEventRecord(static_cast<cudaEvent_t>(a->ev_gemm_start), s));
  T4R_TRY(launch_gemm(pb, ep, s));
  if (a->ev_gemm_stop) T4R_CUDA(cudaEventRecord(static_cast<cudaEvent_t>(a->ev_gemm_stop), s));
  return launch_head_reduce(part_m, part_s, part_z, n_tiles, part_ld, a->T_cap, a->t_dev, a->pos_logit, a->row_tgt,
                            a->label_smoothing, a->V, a->row_lse, a->row_loss, a->loss, scratch, s);
}

static int head_logits_impl(const void* xt_planes, const void* w_planes, int T_cap, const int32_t* t_dev, int64_t V,
                            int De, float inv_temperature, float* out, int64_t ldo, int nprod, const float* xt_inv_scale,
                            const float* w_inv_scale, void* stream);
extern "C" int t4r_head_logits(const void* xt_planes, const void* w_planes, int T_cap, const int32_t* t_dev, int64_t V,
                               int De, float inv_temperature, float* out, int64_t ldo, int nprod, void* stream) {
  T4R_REQUIRE(nprod != 2, "head_logits: nprod = 2 operands go through t4r_head_logits_mixed");
  return head_logits_impl(xt_planes, w_planes, T_cap, t_dev, V, De, inv_temperature, out, ldo, nprod, nullptr, nullptr,
                          stream);
}
extern "C" int t4r_head_logits_mixed(const void* xt_planes, const void* w_planes, int T_cap, const int32_t* t_dev,
                                     int64_t V, int De, float inv_temperature, float* out, int64_t ldo,
                                     const float* xt_inv_scale, const float* w_inv_scale, void* stream) {
  T4R_REQUIRE(xt_inv_scale && w_inv_scale, "head_logits_mixed: the inverse row scales of both operands are required");
  return head_logits_impl(xt_planes, w_planes, T_cap, t_dev, V, De, inv_temperature, out, ldo, 2, xt_inv_scale,
                          w_inv_scale, stream);
}
static int head_logits_impl(const void* xt_planes, const void* w_planes, int T_cap, const int32_t* t_dev, int64_t V,
                            int De, float inv_temperature, float* out, int64_t ldo, int nprod, const float* xt_inv_scale,
                            const float* w_inv_scale, void* stream) {
  T4R_REQUIRE(xt_planes && w_planes && out && T_cap > 0 && V > 0 && De > 0 && ldo >= V, "head_logits: bad arguments");
  GemmProblem pb;
  pb.M = T_cap;
  pb.N = V;
  pb.Kp = t4r_round_up64(De);
  pb.a_planes = static_cast<const __nv_bfloat16*>(xt_planes);
  pb.a_rows = T_cap;
  pb.b_planes = static_cast<const __nv_bfloat16*>(w_planes);
  pb.b_rows = V;
  pb.m_dev = t_dev;
  pb.nprod = nprod ? nprod : 3;
  pb.bn = 256;
  GemmEpilogue ep;
  ep.out_f32 = out;
  ep.ldo = ldo;
  ep.out_scale = inv_temperature != 0.f ? inv_temperature : 1.f;
  ep.row_scale = xt_inv_scale;
  ep.col_scale = w_inv_scale;
  return launch_gemm(pb, ep, static_cast<cudaStream_t>(stream));
}

