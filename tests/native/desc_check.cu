// Host-side cross-check of the hand-written tcgen05 descriptor encodings (csrc/t4r_common.cuh) against CUTLASS / CuTe.
// Test infrastructure: compiled and run by tests/test_abi_and_host.py; nothing from CUTLASS is linked into the product.
// Every line prints our encoding; when the CuTe headers are on the include path (e.g. as vendored by flashinfer under
// flashinfer/data/cutlass/include) it also prints CuTe's and compares.  The test holds our encodings to CuTe's values
// as stored in tests/golden/umma_descriptors.json, so the check does not need the headers.
//   instruction descriptor: cute::UMMA::make_instr_desc<A, B, float, M, N, K-major, K-major>()
//   shared-memory descriptor: the bit fields of cute::UMMA::SmemDescriptor filled with the K-major SWIZZLE_128B
//   canonical values (start address >> 4, LBO = 1 unit, SBO = 8 rows * row bytes, version 1)
#include <cstdio>
#include "t4r_common.cuh"

#if __has_include(<cute/arch/mma_sm100_desc.hpp>)
#define T4R_HAVE_CUTE 1
#include <cute/arch/mma_sm100_desc.hpp>
#include <cute/numeric/numeric_types.hpp>
using namespace cute;

template <class A, class B, int M, int N>
constexpr uint32_t cute_idesc() {
  return uint32_t(UMMA::make_instr_desc<A, B, float, M, N, UMMA::Major::K, UMMA::Major::K>());
}
static uint64_t cute_sw(uint32_t addr, int sbo_bytes, UMMA::LayoutType lt) {
  UMMA::SmemDescriptor d;
  d.start_address_ = (addr >> 4) & 0x3FFF;
  d.leading_byte_offset_ = 1;
  d.stride_byte_offset_ = sbo_bytes >> 4;
  d.version_ = 1;
  d.base_offset_ = 0;
  d.lbo_mode_ = 0;
  d.layout_type_ = uint8_t(lt);
  return uint64_t(d);
}
#define CUTE(expr) (expr)
#else
#define T4R_HAVE_CUTE 0
#define CUTE(expr) 0
#endif

// the device helper restated for the host (same arithmetic as umma_desc_sw128)
static uint64_t ours_sw(uint32_t addr, int sbo_bytes, int layout) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((addr >> 4) & 0x3FFFu);
  d |= static_cast<uint64_t>(1) << 16;
  d |= static_cast<uint64_t>(sbo_bytes >> 4) << 32;
  d |= static_cast<uint64_t>(1) << 46;
  d |= static_cast<uint64_t>(layout) << 61;
  return d;
}

int main() {
  int bad = 0;
  char what[64];
#define CHECK32(mine, theirs, label) do { uint32_t a = (mine); printf("%-32s ours %08x", label, a); \
    if (T4R_HAVE_CUTE) { uint32_t b = CUTE(theirs); printf(" cute %08x %s", b, a == b ? "ok" : "MISMATCH"); bad += a != b; } \
    printf("\n"); } while (0)
#define CHECK64(mine, theirs, label) do { uint64_t a = (mine); printf("%-32s ours %016llx", label, (unsigned long long)a); \
    if (T4R_HAVE_CUTE) { uint64_t b = CUTE(theirs); printf(" cute %016llx %s", (unsigned long long)b, a == b ? "ok" : "MISMATCH"); \
                         bad += a != b; } \
    printf("\n"); } while (0)
  CHECK32(t4r::umma_idesc_bf16(128, 256), (cute_idesc<bfloat16_t, bfloat16_t, 128, 256>()), "idesc bf16 M128 N256");
  CHECK32(t4r::umma_idesc_bf16(256, 256), (cute_idesc<bfloat16_t, bfloat16_t, 256, 256>()), "idesc bf16 M256 N256");
  CHECK32(t4r::umma_idesc_bf16(128, 128), (cute_idesc<bfloat16_t, bfloat16_t, 128, 128>()), "idesc bf16 M128 N128");
  CHECK32(t4r::umma_idesc_bf16(128, 64), (cute_idesc<bfloat16_t, bfloat16_t, 128, 64>()), "idesc bf16 M128 N64");
  CHECK32(t4r::umma_idesc_f16(128, 256), (cute_idesc<half_t, half_t, 128, 256>()), "idesc fp16 M128 N256");
  CHECK32(t4r::umma_idesc_f16(256, 256), (cute_idesc<half_t, half_t, 256, 256>()), "idesc fp16 M256 N256");
  CHECK32(t4r::umma_idesc_e4m3(128, 256), (cute_idesc<float_e4m3_t, float_e4m3_t, 128, 256>()), "idesc e4m3 M128 N256");
  CHECK32(t4r::umma_idesc_e4m3(256, 256), (cute_idesc<float_e4m3_t, float_e4m3_t, 256, 256>()), "idesc e4m3 M256 N256");
  CHECK32(t4r::umma_idesc_e4m3(128, 128), (cute_idesc<float_e4m3_t, float_e4m3_t, 128, 128>()), "idesc e4m3 M128 N128");
  for (uint32_t addr : {0x0u, 0x400u, 0x8460u, 0x3fc20u}) {
    snprintf(what, sizeof what, "smem desc K-major SW128 @%05x", addr);
    CHECK64(ours_sw(addr, 1024, 2), cute_sw(addr, 1024, UMMA::LayoutType::SWIZZLE_128B), what);
  }
  return bad;
}
