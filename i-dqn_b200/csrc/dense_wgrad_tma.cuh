// Weight gradient of the big Dense layer (Dense_0: 7744 x 512) fused with optax.adam (idqn.py:52,106-107 of the
// reference), as a persistent TMA pipeline (sm_100a).  This is the HBM-bound kernel of the step: per parameter it
// reads W, mu, nu (12 B) and writes W, mu, nu (12 B) -- nothing else: the layer has no bf16 copies in HBM (its forward
// and data-gradient kernels split the fp32 master in shared memory, dense_stream.cuh); the gradient
//     dW[i][o] = sum_b x[b][i] dy[b][o]         (contraction over the batch only, K = 32)
// is produced on the tensor core straight into TMEM and never goes to memory.
//
// Tile = 8 FULL rows of the kernel (8 x 512 floats = 16 KB contiguous per array): the DRAM sees long contiguous
// runs (measured: 128-byte pieces per row -> 41% of peak, 512-byte pieces -> 59%).  The accumulator is the
// TRANSPOSE, D^T[o][i] = sum_b dy[b][o] x[b][i]: M = 128 columns o (TMEM lanes) per column block, four column blocks,
// N = 16 rows i per x plane of which the first 8 belong to the tile (the MMAs are far off the critical path).  Per tile one stage:
//   TMA loads (un-swizzled fp32 boxes {256 o, 8 i}, two per array) W, mu, nu + the [32 b][16 i] x planes   (warp 0)
//   tcgen05.mma per column block: D^T[128 o][32] = dy_hi^T [x_hi | x_lo], D^T[:, 0:16] += dy_lo^T x_hi     (warp 1)
//   epilogue, thread = (column o of one column block, 8 rows): g from TMEM, W/mu/nu from the stage (lanes =
//   consecutive floats, conflict free), Adam in registers, results written back IN PLACE             (warps 2..17)
//   TMA stores of the three updated tiles from the same stage; the stage returns to the producer when the bulk
//   stores have read it (cp.async.bulk.wait_group.read).
// The dy^T operand of the current head ([128 o][32 b] hi/lo per column block) is the MMAs' A operand in TMEM, next to
// the accumulators: the epilogue threads write it (tcgen05.st, each its own lane o) when the CTA's contiguous range of
// (head, row tile) items crosses a head.  Shared memory holds only the load ring: four stages of 50 KB.  One SM keeps
// about as many bytes in flight as it has stages, and the update's per-SM HBM rate rises with them.  The bias gradient
// of the layer is not computed here (head_bwd_kernel sums dL/dhidden over the batch; the final Adam launch covers the bias).
#pragma once
#include "common.cuh"
#include "tc_core.cuh"
#include "tma_core.cuh"

namespace dwt {
using namespace tc;
typedef __nv_bfloat16 bf16;

constexpr int NTHREADS = 608;   // warp 0: TMA loads, warp 1: MMA, warps 2..17: epilogue, warp 18: TMA stores
constexpr int STAGES = 4;
constexpr int TM = 8;           // rows (i) per tile
constexpr int TN = 16;          // N per x plane (rows i, the first TM are the tile's): one SWIZZLE_32B atom
constexpr int TO = 128;         // columns (o) per column block = TMEM lanes
constexpr int CB = 4;           // column blocks: O = CB * TO
constexpr int NB = 32;          // batch = K of the MMAs
constexpr uint32_t TILE_F32 = TM * CB * TO * 4;                  // 16 KB per array
constexpr uint32_t X_PLANE = NB * TN * 2;                        // [32 b][16 i] bf16: 1 KB
constexpr uint32_t STAGE_BYTES = 3 * TILE_F32 + 2 * X_PLANE;     // 50 KB
constexpr uint32_t BAR_OFF = STAGES * STAGE_BYTES;
constexpr uint32_t SMEM_TOTAL = BAR_OFF + 256 + 1024;
// TMEM columns: two accumulator buffers of CB x [hi*hi + lo*hi (16) | hi*lo (16)] fp32, then the dy^T operand,
// CB x [hi (16) | lo (16)] columns of bf16 pairs; 384 used, the allocation is a power of two
constexpr uint32_t ACC_COLS = CB * 2 * TN;
constexpr uint32_t A_COL = 2 * ACC_COLS;
constexpr uint32_t TMEM_COLS = 512;
static_assert(A_COL + CB * NB <= TMEM_COLS, "TMEM budget");

struct Args {
  int heads, tile0, ntiles;   // 8-row tiles [tile0, tile0 + ntiles) of every head
  int I, O;
  const int32_t* count;
  float lr, b1, b2, eps;
  float* grad;                // optional: materialised gradient (IDQN_F_KEEP_GRADS)
  const bf16 *dyh, *dyl;      // dL/dy planes [head][NB b][O o], head stride dystride
  int64_t dystride;
  unsigned long long stream_policy;  // L2 policy of the W / mu / nu loads and stores
  int64_t stride, w_off;
  int tl_id;
};

__device__ __forceinline__ void tma_store_3d(const CUtensorMap* map, uint32_t src, int c0, int c1, int c2) {
  asm volatile("cp.async.bulk.tensor.3d.global.shared::cta.bulk_group [%0, {%2, %3, %4}], [%1];" ::"l"(map), "r"(src),
               "r"(c0), "r"(c1), "r"(c2)
               : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void bulk_wait_read() {
  asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory");
}
__device__ __forceinline__ void bulk_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
__device__ __forceinline__ void epi_bar_sync() { asm volatile("bar.sync 1, 512;" ::: "memory"); }

__global__ void __launch_bounds__(NTHREADS, 1)
dense_wgrad_adam_kernel(const __grid_constant__ CUtensorMap mapX_hi, const __grid_constant__ CUtensorMap mapX_lo,
                        const __grid_constant__ CUtensorMap mapW, const __grid_constant__ CUtensorMap mapM,
                        const __grid_constant__ CUtensorMap mapV, const Args p) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* smem = smem_raw + (base - smem_u32(smem_raw));
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + BAR_OFF);
  uint64_t* full = bars;                 // [STAGES] TMA loads landed
  uint64_t* empty = bars + STAGES;       // [STAGES] bulk stores have read the stage
  uint64_t* ready = bars + 2 * STAGES;   // [STAGES] Adam results written into the stage (epilogue -> store warp)
  uint64_t* acc_full = bars + 3 * STAGES;       // [2]
  uint64_t* acc_empty = bars + 3 * STAGES + 2;  // [2]
  uint64_t* a_full = bars + 3 * STAGES + 4;     // dy^T operand of the current head written into TMEM
  __shared__ uint32_t tmem_base_s;

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  ktl_begin(p.tl_id);
  if (tid == 0) {
    for (int i = 0; i < STAGES; ++i) mbar_init(&full[i], 1), mbar_init(&empty[i], 1), mbar_init(&ready[i], 1);
    for (int i = 0; i < 2; ++i) mbar_init(&acc_full[i], 1), mbar_init(&acc_empty[i], 16);
    mbar_init(a_full, 16);
    fence_mbar_init();
  }
  if (warp == 1) tmem_alloc(&tmem_base_s, TMEM_COLS);
  fence_proxy_async_smem();
  tcgen05_before_sync();
  __syncthreads();
  tcgen05_after_sync();
  const uint32_t tmem = tmem_base_s;

  const int n_items = p.heads * p.ntiles;
  const int i0 = (int)((int64_t)blockIdx.x * n_items / gridDim.x), i1 = (int)((int64_t)(blockIdx.x + 1) * n_items / gridDim.x);

  if (warp == 0) {
    if (elect_one()) {
      int st = 0;
      uint32_t ph = 0;
      for (int it = i0; it < i1; ++it) {
        const int z = it / p.ntiles, row0 = (p.tile0 + it % p.ntiles) * TM;
        mbar_wait(&empty[st], ph ^ 1);
        tma::expect_tx(&full[st], STAGE_BYTES);
        const uint32_t s0 = base + st * STAGE_BYTES;
        tma::load_3d(s0 + 3 * TILE_F32, &mapX_hi, &full[st], row0, 0, z);
        tma::load_3d(s0 + 3 * TILE_F32 + X_PLANE, &mapX_lo, &full[st], row0, 0, z);
        for (int hb = 0; hb < 2; ++hb) {  // two boxes of 256 columns per array
          tma::load_3d_hint(s0 + hb * (TILE_F32 / 2), &mapW, &full[st], hb * 256, row0, z, p.stream_policy);
          tma::load_3d_hint(s0 + TILE_F32 + hb * (TILE_F32 / 2), &mapM, &full[st], hb * 256, row0, z, p.stream_policy);
          tma::load_3d_hint(s0 + 2 * TILE_F32 + hb * (TILE_F32 / 2), &mapV, &full[st], hb * 256, row0, z, p.stream_policy);
        }
        if (++st == STAGES) st = 0, ph ^= 1;
      }
    }
  } else if (warp == 1) {
    if (elect_one()) {
      const uint32_t idesc2 = make_idesc_bf16(128, 2 * TN, false, true);  // dy_hi^T [x_hi | x_lo]
      const uint32_t idesc1 = make_idesc_bf16(128, TN, false, true);      // dy_lo^T x_hi
      const uint32_t b_hi32 = tma::desc_hi32(256, tma::LT_SW32);          // SBO: 8 rows b of 32 bytes
      int st = 0, ai = 0, ti = 0, last_z = -1;
      uint32_t ph = 0;
      for (int it = i0; it < i1; ++it, ++ti) {
        const int z = it / p.ntiles;
        if (z != last_z) {
          last_z = z;
          mbar_wait(a_full, ai & 1);
          ++ai;
        }
        const int ab = ti & 1;
        mbar_wait(&acc_empty[ab], ((ti >> 1) & 1) ^ 1);
        mbar_wait(&full[st], ph);
        tcgen05_after_sync();
        const uint32_t xh = tma::desc_lo32(base + st * STAGE_BYTES + 3 * TILE_F32, X_PLANE);  // LBO: the lo plane
#pragma unroll
        for (int cbk = 0; cbk < CB; ++cbk) {
          const uint32_t d = tmem + (uint32_t)ab * ACC_COLS + cbk * 2 * TN;
          const uint32_t ah = tmem + A_COL + cbk * 2 * TN, al = ah + TN;
          tma::mma_bf16_tmem_a<false>(d, ah, xh, b_hi32, idesc2);
          tma::mma_bf16_tmem_a<true>(d, al, xh, b_hi32, idesc1);
          // k = 16..31: 8 TMEM columns further in A, 16 rows (512 bytes) further in the x planes
          tma::mma_bf16_tmem_a<true>(d, ah + 8, xh + 32, b_hi32, idesc2);
          tma::mma_bf16_tmem_a<true>(d, al + 8, xh + 32, b_hi32, idesc1);
        }
        mma_commit(&acc_full[ab]);
        if (++st == STAGES) st = 0, ph ^= 1;
      }
    }
  } else if (warp == 18) {
    // ===== store warp: a stage goes back to the loader as soon as ITS OWN bulk stores have read it.  (Bulk groups are
    // per thread: when an epilogue thread issued the stores it could only wait for the previous tile's group without
    // stalling the next tile's Adam, so every stage was held one tile period longer: 3 stages, ~1 load in flight.)
    if (elect_one()) {
      int st = 0;
      uint32_t ph = 0;
      for (int it = i0; it < i1; ++it) {
        const int z = it / p.ntiles, row0 = (p.tile0 + it % p.ntiles) * TM;
        mbar_wait(&ready[st], ph);
        const uint32_t src = base + st * STAGE_BYTES;
        for (int hb = 0; hb < 2; ++hb) {
          tma::store_3d_hint(&mapW, src + hb * (TILE_F32 / 2), hb * 256, row0, z, p.stream_policy);
          tma::store_3d_hint(&mapM, src + TILE_F32 + hb * (TILE_F32 / 2), hb * 256, row0, z, p.stream_policy);
          tma::store_3d_hint(&mapV, src + 2 * TILE_F32 + hb * (TILE_F32 / 2), hb * 256, row0, z, p.stream_policy);
        }
        bulk_commit();
        bulk_wait_read<0>();
        tma::arrive(&empty[st]);
        if (++st == STAGES) st = 0, ph ^= 1;
      }
      bulk_wait_all();
    }
  } else {
    // ===== epilogue: warps 2..17; TMEM lane quadrant = warp % 4 (column o), column block = (warp - 2) / 4 =====
    const int q = warp & 3, o = q * 32 + lane, cbk = (warp - 2) >> 2;
    int st = 0, ti = 0, last_z = -1;
    uint32_t ph = 0;
    AdamCoef ac;
    for (int it = i0; it < i1; ++it, ++ti) {
      const int z = it / p.ntiles, row0 = (p.tile0 + it % p.ntiles) * TM;
      if (z != last_z) {
        last_z = z;
        ac = adam_coef(p.b1, p.b2, p.lr, p.eps, p.count[z]);  // count already incremented for this step
        // dy^T of head z into this thread's TMEM lane, as bf16 pairs (b even in the low half).  The MMAs that read the
        // previous head's operand have completed: this warp waited for their commit (acc_full) in the previous item.
        const unsigned short* yh = reinterpret_cast<const unsigned short*>(p.dyh + z * p.dystride) + cbk * TO + o;
        const unsigned short* yl = reinterpret_cast<const unsigned short*>(p.dyl + z * p.dystride) + cbk * TO + o;
        uint32_t rh[NB / 2], rl[NB / 2];
#pragma unroll
        for (int j = 0; j < NB / 2; ++j) {
          rh[j] = (uint32_t)__ldg(yh + 2 * j * p.O) | (uint32_t)__ldg(yh + (2 * j + 1) * p.O) << 16;
          rl[j] = (uint32_t)__ldg(yl + 2 * j * p.O) | (uint32_t)__ldg(yl + (2 * j + 1) * p.O) << 16;
        }
        const uint32_t ta = tmem + ((uint32_t)(q * 32) << 16) + A_COL + cbk * 2 * TN;
        tmem_st16(ta, rh);
        tmem_st16(ta + TN, rl);
        tmem_st_wait();
        tcgen05_before_sync();
        __syncwarp();
        if (lane == 0) tma::arrive(a_full);
      }
      const int ab = ti & 1;
      mbar_wait(&acc_full[ab], (ti >> 1) & 1);
      mbar_wait(&full[st], ph);  // the stage's W / mu / nu tiles (async-proxy writes) are visible after this wait
      tcgen05_after_sync();
      float g[16];
      {
        const uint32_t taddr = tmem + ((uint32_t)(q * 32) << 16) + (uint32_t)ab * ACC_COLS + cbk * 2 * TN;
        float g2[16];
        tmem_ld16_nowait(taddr, g);
        tmem_ld16_nowait(taddr + TN, g2);
        tmem_ld_wait();
#pragma unroll
        for (int e = 0; e < TM; ++e) g[e] += g2[e];
      }
      tcgen05_before_sync();
      __syncwarp();
      if (lane == 0) tma::arrive(&acc_empty[ab]);
      // stage layout per array: [box][8 rows][256 columns]; this thread: column cbk * 128 + o
      float* sW = reinterpret_cast<float*>(smem + st * STAGE_BYTES + (cbk >> 1) * (TILE_F32 / 2)) + (cbk & 1) * 128 + o;
      float* sM = sW + TILE_F32 / 4;
      float* sV = sM + TILE_F32 / 4;
      const int64_t gb = (int64_t)z * p.stride + p.w_off + (int64_t)row0 * p.O + cbk * 128 + o;
      float P[TM], M[TM], V[TM];
#pragma unroll
      for (int e = 0; e < TM; ++e) P[e] = sW[e * 256], M[e] = sM[e * 256], V[e] = sV[e * 256];
#pragma unroll
      for (int e = 0; e < TM; ++e) {
        adam_elem(ac, g[e], P[e], M[e], V[e]);
        sW[e * 256] = P[e], sM[e * 256] = M[e], sV[e * 256] = V[e];
      }
      fence_proxy_async_smem();  // generic-proxy writes of this thread -> visible to the bulk stores
      epi_bar_sync();
      if (tid == 64) tma::arrive(&ready[st]);
      if (p.grad) {  // the optional gradient after the barrier: off the stores' critical path
#pragma unroll
        for (int e = 0; e < TM; ++e) p.grad[gb + (int64_t)e * p.O] = g[e];
      }
      if (++st == STAGES) st = 0, ph ^= 1;
    }
  }
  tcgen05_before_sync();
  __syncthreads();
  ktl_end(p.tl_id);
  if (warp == 1) tmem_dealloc(tmem, TMEM_COLS);
}

}  // namespace dwt
