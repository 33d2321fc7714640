// TMA (cp.async.bulk.tensor) + swizzled UMMA shared-memory descriptors for sm_100a, inline PTX.
//
// The image-resident conv kernels (conv_img.cuh) move whole operand tiles global -> shared with one TMA
// instruction issued by one thread and hand them to tcgen05.mma through SWIZZLE_128B / SWIZZLE_64B descriptors.
// Facts this relies on, measured on a B200 with tools/tma_probe.cu (60 configurations):
//   * a TMA box with inner extent 128 B (64 B) and CU_TENSOR_MAP_SWIZZLE_128B (64B), landing on a 1024-byte
//     aligned address, is exactly the UMMA canonical K-major (rows = M/N, 8-row groups at SBO = 8 * row bytes)
//     and MN-major (rows = K, 8-row groups at SBO, 64/32-element MN groups at LBO) layout;
//   * the swizzle is a function of the absolute shared-memory address, so a descriptor may start at ANY whole
//     row of the tile with base_offset = 0 (tap shifts of an image kept resident in shared memory);
//   * LBO may be smaller than a tile (two MN groups that alias the same image one row apart).
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "tc_core.cuh"

namespace tma {
using tc::smem_u32;

__device__ __forceinline__ void prefetch_desc(const CUtensorMap* m) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(m) : "memory");
}
__device__ __forceinline__ void expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void load_2d(uint32_t dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(dst),
      "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void load_3d(uint32_t dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1, int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];" ::"r"(
          dst),
      "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}
__device__ __forceinline__ void load_4d(uint32_t dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1, int c2,
                                        int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];" ::
          "r"(dst),
      "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
      : "memory");
}

// L2 eviction-priority policies for the cache_hint operand (the pre-encoded descriptors createpolicy would return)
constexpr uint64_t L2_EVICT_NORMAL = 0x1000000000000000ull, L2_EVICT_FIRST = 0x12F0000000000000ull,
                   L2_EVICT_LAST = 0x14F0000000000000ull;
__device__ __forceinline__ void load_3d_hint(uint32_t dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1, int c2,
                                             uint64_t policy) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1, {%3, %4, %5}], "
      "[%2], %6;" ::"r"(dst),
      "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "l"(policy)
      : "memory");
}
__device__ __forceinline__ void store_3d_hint(const CUtensorMap* map, uint32_t src, int c0, int c1, int c2, uint64_t policy) {
  asm volatile("cp.async.bulk.tensor.3d.global.shared::cta.bulk_group.L2::cache_hint [%0, {%2, %3, %4}], [%1], %5;" ::"l"(map),
               "r"(src), "r"(c0), "r"(c1), "r"(c2), "l"(policy)
               : "memory");
}
// bf16 hi/lo planes of one value, stored with an L2 eviction priority
__device__ __forceinline__ void st1_planes_hint(__nv_bfloat16* hi, __nv_bfloat16* lo, float v, uint64_t policy) {
  const __nv_bfloat16 h = __float2bfloat16_rn(v);
  const __nv_bfloat16 l = __float2bfloat16_rn(v - __bfloat162float(h));
  asm volatile("st.global.L2::cache_hint.b16 [%0], %1, %2;" ::"l"(hi), "h"(*reinterpret_cast<const unsigned short*>(&h)), "l"(policy) : "memory");
  asm volatile("st.global.L2::cache_hint.b16 [%0], %1, %2;" ::"l"(lo), "h"(*reinterpret_cast<const unsigned short*>(&l)), "l"(policy) : "memory");
}

// UMMA layout types (cute/arch/mma_sm100_desc.hpp: UMMA::LayoutType)
constexpr uint32_t LT_SW128 = 2, LT_SW64 = 4, LT_SW32 = 6;
// swizzled shared-memory matrix descriptor; saddr may be any 16-byte aligned address inside a 1024-byte aligned tile
__device__ __forceinline__ uint64_t make_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes, uint32_t layout_type) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr >> 4) & 0x3FFFu);
  d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFFu) << 16;
  d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFFu) << 32;
  d |= (uint64_t)1 << 46;  // descriptor version (Blackwell)
  d |= (uint64_t)(layout_type & 7u) << 61;
  return d;
}

// The MMA-issuing thread is a single instruction stream: rebuilding 64-bit descriptors for every MMA costs more
// than the MMA itself (32 cycles at N = 64).  Split form: the high word (SBO, version, layout) is loop-invariant and
// the low word (start address >> 4 | LBO >> 4 << 16) advances by plain 32-bit adds of (byte offset >> 4).
__device__ __forceinline__ uint32_t desc_hi32(uint32_t sbo_bytes, uint32_t layout_type) {
  return ((sbo_bytes >> 4) & 0x3FFFu) | (1u << 14) | ((layout_type & 7u) << 29);
}
__device__ __forceinline__ uint32_t desc_lo32(uint32_t saddr, uint32_t lbo_bytes) {
  return ((saddr >> 4) & 0x3FFFu) | (((lbo_bytes >> 4) & 0x3FFFu) << 16);
}
template <bool ACC>
__device__ __forceinline__ void mma_bf16_split(uint32_t d_tmem, uint32_t a_lo, uint32_t a_hi, uint32_t b_lo, uint32_t b_hi,
                                               uint32_t idesc) {
  if (ACC) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        ".reg .b64 da, db;\n"
        "setp.eq.u32 p, 1, 1;\n"
        "mov.b64 da, {%1, %2};\n"
        "mov.b64 db, {%3, %4};\n"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %5, p;\n"
        "}\n" ::"r"(d_tmem),
        "r"(a_lo), "r"(a_hi), "r"(b_lo), "r"(b_hi), "r"(idesc)
        : "memory");
  } else {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        ".reg .b64 da, db;\n"
        "setp.ne.u32 p, 1, 1;\n"
        "mov.b64 da, {%1, %2};\n"
        "mov.b64 db, {%3, %4};\n"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %5, p;\n"
        "}\n" ::"r"(d_tmem),
        "r"(a_lo), "r"(a_hi), "r"(b_lo), "r"(b_hi), "r"(idesc)
        : "memory");
  }
}
// The same with the A operand in tensor memory: M = 128 lanes (row m = lane m), K-major, two bf16 per 32-bit column
// (element k in the low half of column k / 2), so one K = 16 step reads 8 columns from a_tmem.  idesc: a_major = K.
template <bool ACC>
__device__ __forceinline__ void mma_bf16_tmem_a(uint32_t d_tmem, uint32_t a_tmem, uint32_t b_lo, uint32_t b_hi, uint32_t idesc) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      ".reg .b64 db;\n"
      "setp.ne.u32 p, %5, 0;\n"
      "mov.b64 db, {%2, %3};\n"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], db, %4, p;\n"
      "}\n" ::"r"(d_tmem),
      "r"(a_tmem), "r"(b_lo), "r"(b_hi), "r"(idesc), "n"(ACC ? 1 : 0)
      : "memory");
}

// ---- host: tensor-map encoding through the driver entry point (no link-time dependency on libcuda) ----------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static inline EncodeTiledFn encode_fn() {
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess) fn = (EncodeTiledFn)p;
  }
  return fn;
}
// fp32 tensor, no swizzle (row-major box in shared memory), rank <= 4, dims/box innermost first
static inline bool encode_f32(CUtensorMap* map, const void* base, int rank, const uint64_t* dims, const uint64_t* strides,
                              const uint32_t* box) {
  EncodeTiledFn fn = encode_fn();
  if (!fn) return false;
  cuuint64_t gd[5], gs[5];
  cuuint32_t bx[5], es[5];
  for (int i = 0; i < rank; ++i) gd[i] = dims[i], bx[i] = box[i], es[i] = 1;
  for (int i = 0; i + 1 < rank; ++i) gs[i] = strides[i];
  return fn(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, (cuuint32_t)rank, const_cast<void*>(base), gd, gs, bx, es,
            CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
            CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}
// bf16 tensor, rank <= 4, dims/box innermost first, strides (bytes) for dims 1..rank-1; sw_bytes = 128, 64 or 32
static inline bool encode_bf16(CUtensorMap* map, const void* base, int rank, const uint64_t* dims, const uint64_t* strides,
                               const uint32_t* box, int sw_bytes) {
  EncodeTiledFn fn = encode_fn();
  if (!fn) return false;
  cuuint64_t gd[5], gs[5];
  cuuint32_t bx[5], es[5];
  for (int i = 0; i < rank; ++i) gd[i] = dims[i], bx[i] = box[i], es[i] = 1;
  for (int i = 0; i + 1 < rank; ++i) gs[i] = strides[i];
  const CUtensorMapSwizzle sw = sw_bytes == 128 ? CU_TENSOR_MAP_SWIZZLE_128B
                                : sw_bytes == 64 ? CU_TENSOR_MAP_SWIZZLE_64B
                                                 : CU_TENSOR_MAP_SWIZZLE_32B;
  return fn(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, (cuuint32_t)rank, const_cast<void*>(base), gd, gs, bx, es,
            CU_TENSOR_MAP_INTERLEAVE_NONE, sw, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
            CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

}  // namespace tma
