// tcgen05 / TMEM / mbarrier primitives for sm_100a (inline PTX) and the shared-memory operand layouts used by
// the tensor-core implicit-GEMM kernels.
//
// Operand tiles are written by the CTA's own threads (global fp32/u8 -> bf16 hi/lo split -> st.shared) in the
// UMMA canonical *no-swizzle* layouts, so no TMA descriptor is involved: the im2col gather, the /255 dequant,
// the relu' masks and the fp32 -> 2 x bf16 split all happen on the way into shared memory.
//
// Layouts (16-byte "units" of 8 bf16; a core matrix = 8 units = 128 contiguous bytes):
//   K-major tile  [ROWS x 32]:  unit(row r, kunit u) at  u*(ROWS*16) + r*16          LBO = ROWS*16, SBO = 128
//   MN-major tile [32 x COLS]:  unit(k, mn-group g)  at  (k/8)*(COLS*16) + g*128 + (k%8)*16   LBO = COLS*16, SBO = 128
// In both, LBO is the byte stride between core matrices adjacent in K and SBO between core matrices adjacent in
// M/N, which is how the sm_100 matrix descriptor interprets them for SWIZZLE_NONE (cute/atom/mma_traits_sm100.hpp).
#pragma once
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace tc {

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// ---- mbarrier ------------------------------------------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_mbar_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
      "selp.u32 %0, 1, 0, p;\n"
      "}\n"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
// bounded wait: a protocol bug traps (kernel error) instead of hanging the GPU
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  uint32_t spins = 0;
  while (!mbar_try_wait(bar, parity)) {
    if (++spins > (1u << 24)) __trap();
  }
}

// one lane of a converged warp (elect.sync): code under `if (elect_one())` lets ptxas issue the uniform-datapath
// instructions (UTCHMMA, UTMALDG, UTCBAR) directly; under `if (lane == 0)` it wraps each of them in an ELECT /
// BRA.U.ANY waterfall loop
__device__ __forceinline__ bool elect_one() {
  uint32_t pred = 0, laneid = 0;
  asm volatile(
      "{\n"
      ".reg .b32 %%rx;\n"
      ".reg .pred %%px;\n"
      "     elect.sync %%rx|%%px, %2;\n"
      "@%%px mov.s32 %1, 1;\n"
      "     mov.s32 %0, %%rx;\n"
      "}\n"
      : "+r"(laneid), "+r"(pred)
      : "r"(0xFFFFFFFF));
  return pred != 0;
}

// ---- fences ---------------------------------------------------------------------------------------------
__device__ __forceinline__ void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tcgen05_before_sync() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tcgen05_after_sync() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// ---- TMEM -----------------------------------------------------------------------------------------------
// one full warp executes alloc/dealloc; ncols is a power of two in [32, 512]
__device__ __forceinline__ void tmem_alloc(uint32_t* smem_dst, uint32_t ncols) {
  __syncwarp();
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_dst)), "r"(ncols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  __syncwarp();
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
// 32 lanes x 16 consecutive fp32 columns: thread i of warp w receives row (32*(w%4) + i)
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, float* v) {
  uint32_t r[16];
  __syncwarp();  // .sync.aligned: the warp must be converged (callers branch per lane between loads)
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
  for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(r[i]);
}

// the same load without the wait: issue several, then tmem_ld_wait() once
__device__ __forceinline__ void tmem_ld16_nowait(uint32_t taddr, float* v) {
  uint32_t r[16];
  __syncwarp();
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
#pragma unroll
  for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(r[i]);
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
// 32 lanes x 16 consecutive 32-bit columns: thread i of warp w writes row (32*(w%4) + i); complete after tmem_st_wait()
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const uint32_t* r) {
  __syncwarp();
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16};" ::"r"(taddr),
      "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]), "r"(r[9]), "r"(r[10]),
      "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15])
      : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// ---- descriptors ------------------------------------------------------------------------------------------
// sm_100 shared-memory matrix descriptor, SWIZZLE_NONE (cute/arch/mma_sm100_desc.hpp: SmemDescriptor)
__device__ __forceinline__ uint64_t make_smem_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr >> 4) & 0x3FFFu);            // bits [0,14)  start address >> 4
  d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFFu) << 16;  // bits [16,30) leading-dimension byte offset >> 4
  d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFFu) << 32;  // bits [32,46) stride-dimension byte offset >> 4
  d |= (uint64_t)1 << 46;                             // bits [46,48) descriptor version = 1 (Blackwell)
  return d;                                           // base_offset 0, lbo_mode 0, layout_type 0 (no swizzle)
}
// instruction descriptor for kind::f16, bf16 x bf16 -> fp32 (InstrDescriptor in the same header)
__host__ __device__ constexpr uint32_t make_idesc_bf16(int M, int N, bool a_mn_major, bool b_mn_major) {
  return (1u << 4)                          // c_format  = F32
         | (1u << 7)                        // a_format  = BF16
         | (1u << 10)                       // b_format  = BF16
         | ((a_mn_major ? 1u : 0u) << 15)   // a_major   (0 = K-major)
         | ((b_mn_major ? 1u : 0u) << 16)   // b_major
         | ((uint32_t)(N >> 3) << 17)       // n_dim
         | ((uint32_t)(M >> 4) << 24);      // m_dim
}

// D[tmem] (+)= A[smem] * B[smem]; issued by ONE thread
__device__ __forceinline__ void mma_bf16(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                         uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n"
      "}\n" ::"r"(d_tmem),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// arrive on `bar` once every MMA issued so far by this thread has completed (implies fence::before_thread_sync)
__device__ __forceinline__ void mma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
               : "memory");
}

// ---- fp32 -> bf16 hi/lo split -------------------------------------------------------------------------------
// x = hi + lo + O(2^-18 |x|): hi = bf16(x), lo = bf16(x - hi).  hi*hi' + hi*lo' + lo*hi' reproduces the fp32
// product to ~2^-17 relative (SURVEY §7.2 "bf16x3").
__device__ __forceinline__ void split8(const float* x, uint4& hi, uint4& lo) {
  uint32_t h[4], l[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    // cvt.rn.bf16x2.f32 packs two conversions in one instruction; hi as fp32 is just its bits << 16
    const __nv_bfloat162 hp = __floats2bfloat162_rn(x[2 * i], x[2 * i + 1]);
    const uint32_t hb = *reinterpret_cast<const uint32_t*>(&hp);
    const float r0 = x[2 * i] - __uint_as_float(hb << 16);
    const float r1 = x[2 * i + 1] - __uint_as_float(hb & 0xffff0000u);
    const __nv_bfloat162 lp = __floats2bfloat162_rn(r0, r1);
    h[i] = hb;
    l[i] = *reinterpret_cast<const uint32_t*>(&lp);
  }
  hi = make_uint4(h[0], h[1], h[2], h[3]);
  lo = make_uint4(l[0], l[1], l[2], l[3]);
}
__device__ __forceinline__ uint4 pack8_exact(const float* x) {  // values exactly representable in bf16 (u8 pixels)
  uint32_t h[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const __nv_bfloat162 hp = __floats2bfloat162_rn(x[2 * i], x[2 * i + 1]);
    h[i] = *reinterpret_cast<const uint32_t*>(&hp);
  }
  return make_uint4(h[0], h[1], h[2], h[3]);
}

__device__ __forceinline__ void split4(const float4& x, uint2& hi, uint2& lo) {
  const __nv_bfloat162 h0 = __floats2bfloat162_rn(x.x, x.y), h1 = __floats2bfloat162_rn(x.z, x.w);
  const uint32_t b0 = *reinterpret_cast<const uint32_t*>(&h0), b1 = *reinterpret_cast<const uint32_t*>(&h1);
  const __nv_bfloat162 l0 = __floats2bfloat162_rn(x.x - __uint_as_float(b0 << 16), x.y - __uint_as_float(b0 & 0xffff0000u));
  const __nv_bfloat162 l1 = __floats2bfloat162_rn(x.z - __uint_as_float(b1 << 16), x.w - __uint_as_float(b1 & 0xffff0000u));
  hi = make_uint2(b0, b1);
  lo = make_uint2(*reinterpret_cast<const uint32_t*>(&l0), *reinterpret_cast<const uint32_t*>(&l1));
}
__device__ __forceinline__ void st1_planes(__nv_bfloat16* hi, __nv_bfloat16* lo, float v) {
  const __nv_bfloat16 h = __float2bfloat16_rn(v);
  *hi = h;
  *lo = __float2bfloat16_rn(v - __bfloat162float(h));
}

// optax.scale_by_adam + scale(-lr) on one element with MUFU-approximate sqrt/divide (relative error ~2^-22,
// far inside the 1e-4 parity bar; the IEEE versions cost >100 instructions per element)
struct AdamCoef {
  float b1, b2, omb1, omb2, rbc1, rbc2, lr, eps;
};
__device__ __forceinline__ AdamCoef adam_coef(float b1, float b2, float lr, float eps, int count) {
  AdamCoef c;
  const float t = (float)count;
  c.b1 = b1, c.b2 = b2, c.omb1 = 1.f - b1, c.omb2 = 1.f - b2;
  c.rbc1 = 1.f / (1.f - powf(b1, t));
  c.rbc2 = 1.f / (1.f - powf(b2, t));
  c.lr = lr, c.eps = eps;
  return c;
}
__device__ __forceinline__ void adam_elem(const AdamCoef& c, float g, float& p, float& m, float& v) {
  m = fmaf(c.b1, m, c.omb1 * g);
  v = fmaf(c.b2, v, c.omb2 * (g * g));
  float sq;
  asm("sqrt.approx.f32 %0, %1;" : "=f"(sq) : "f"(v * c.rbc2));
  p = fmaf(-c.lr, __fdividef(m * c.rbc1, sq + c.eps), p);
}

// ---- operand tile addressing (BK = 32 elements = 4 k-units per stage) ------------------------------------------
constexpr int BK = 32;
template <int ROWS>
struct KMajorTile {  // [ROWS x 32] bf16
  static constexpr uint32_t BYTES = ROWS * BK * 2, LBO = ROWS * 16, SBO = 128;
  __device__ static __forceinline__ uint32_t unit_off(int row, int kunit) { return kunit * (ROWS * 16) + row * 16; }
  __device__ static __forceinline__ uint32_t k16_off(int j) { return (2 * j) * LBO; }
};
template <int COLS>
struct MNMajorTile {  // [32 x COLS] bf16
  static constexpr uint32_t BYTES = COLS * BK * 2, LBO = COLS * 16, SBO = 128;
  __device__ static __forceinline__ uint32_t unit_off(int k, int group) {
    return (k >> 3) * (COLS * 16) + group * 128 + (k & 7) * 16;
  }
  __device__ static __forceinline__ uint32_t k16_off(int j) { return (2 * j) * LBO; }
};

}  // namespace tc
