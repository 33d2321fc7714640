// Image-resident tcgen05 convolution kernels (sm_100a): forward, data gradient and weight gradient of the
// NatureCNN conv stack (architectures/dqn.py:42-52 of the reference) for batch-32 i-DQN steps.
//
// Formulation.  A conv with kernel k, stride s (k % s == 0) and SAME low padding p is a stride-1 T x T conv
// (T = k/s) over the space-to-depth image X2[by][bx][(ry,rx,c)] = x[s*by+ry-p][s*bx+rx-p][c] with C2 = s*s*IC
// channels.  X2 is stored with a row pitch P = OW + 2(T-1) >= BW, so for the pitched output index m = oy*P + ox
//        y[m] = sum_{ty,tx} X2row[m + ty*P + tx] . W2[ty,tx]            (a pure row shift per tap)
// and one image is a [rows x C2] bf16 matrix that TMA drops into shared memory ONCE (SWIZZLE_128B, 64 channels
// per 128-byte row); the A operand of every tap is the same shared-memory image read through a UMMA descriptor
// whose start address is shifted by (ty*P+tx) rows (tma_core.cuh).  Outputs with ox >= OW are wrap-around garbage
// and are dropped in the epilogue.  The same trick gives
//   dgrad:  dX2[q] = sum_t dyZ[q + (T-1-ty)*P + (T-1-tx)] . W2[t]^T   with dyZ = dy zero-embedded at (T-1, T-1),
//   wgrad:  dW2[t] = sum_m X2row[m + shift(t)]^T dyZ[m + (T-1)(P+1)]    (both images resident, K = pixels).
// Weights are never re-laid out: a 4-D TMA box {OC, s*IC, s, 1} over the flax [KH][KW*IC][OC] kernel IS W2[ty,tx].
//
// Precision: bf16 hi/lo planes, three MMAs per product (hi*hi + hi*lo + lo*hi), fp32 accumulation in TMEM
// ("bf16x3", fp32-faithful to ~2^-17, SURVEY §7.2); uint8 frames are exact in bf16 (two MMAs).
//
// conv_taps_kernel (fwd, dgrad): persistent CTAs walk (net, image) units.  Warp roles: 0 = TMA of the image
// (double-buffered), 1 = TMA of the per-tap weight tiles (ring), 2 = MMA issue, 3..10 = epilogue (TMEM -> bias/relu
// or relu' -> fp32 + the bf16 planes of the consumer's layout); accumulators double-buffered in TMEM so the
// epilogue of unit u overlaps the MMAs of unit u+1.
// conv_wgrad_kernel: CTA = (head, image range); M tiles = tap pairs (the second 64-row group aliases the image at
// a different row shift through LBO) plus a ones tile for the bias gradient; partial dW per CTA, reduced in a
// fixed order by the Adam kernel (deterministic).
#pragma once
#include "common.cuh"
#include "gemm_simt.cuh"
#include "tc_core.cuh"
#include "tma_core.cuh"

namespace img {
using namespace tc;
typedef __nv_bfloat16 bf16;

constexpr int MAX_TAPS = 16;
constexpr int WG_THREADS = 320;  // wgrad: warp 0 TMA, warp 1 MMA, warps 2..9 epilogue
constexpr int NTHREADS = 352;  // 11 warps: TMA image, TMA weights, MMA issue, 8 epilogue warps

// debug timeline (IDQN_TL=<kernel tag> in the environment): lane 0 of every role of CTA 0 stamps clock64 at its
// pipeline events; read back with idqn_debug_timeline.  Costs one predictable branch when off.
constexpr int TL_MAX = 4096;
__device__ unsigned long long g_tl[TL_MAX];
__device__ int g_tl_n;
// fire-and-forget store (no atomic: a returning atomic would stall the role ~0.5 us per stamp); slot = tag
__device__ __forceinline__ void tl_stamp(int on, int tag) {
  if (on && blockIdx.x == 0 && tag < TL_MAX) g_tl[tag] = ((unsigned long long)clock64() << 16) | (unsigned)tag;
}

// one conv layer in space-to-depth form
struct Geom {
  int s, T, ph, pw;
  int IC, OC, C2, halves;
  int IH, IW, OH, OW;
  int BH, BW, P;
  int XR, XRa, x_chunks, x_chunk_rows;  // X2 rows per image, allocated rows (multiple of the TMA box), boxes per image
  int ZH, ZR, ZRa, z_chunks, z_chunk_rows;
  int Kd;
};

// where the epilogue writes bf16 planes: a consumer's X2 / dyZ / plain layout, all of the form
//   row = (img * H2 + (y + off) / s) * P + (x + off) / s ;  col = (((y+off) % s) * s + (x+off) % s) * C + c
struct PlaneDst {
  bf16 *hi, *lo;
  int64_t net_stride;   // elements between nets
  int64_t img_rows;     // allocated rows per image
  int s, off_y, off_x, P, C, C2;
};
__device__ __forceinline__ int64_t plane_index(const PlaneDst& d, int net, int im, int y, int x) {
  const int yy = y + d.off_y, xx = x + d.off_x;
  const int by = yy / d.s, ry = yy - by * d.s, bx = xx / d.s, rx = xx - bx * d.s;
  return (int64_t)net * d.net_stride + ((int64_t)im * d.img_rows + (int64_t)by * d.P + bx) * d.C2 + (ry * d.s + rx) * d.C;
}

struct TapsArgs {
  int n_units, imgs, nets_per_g, hpg, n_hg;
  int n_units_total;  // units of the whole layer (n_units may be a window of them)
  int unit0;  // first unit of this launch (best_action runs a single (net, image) unit of the training layout)
  // A image
  int a_rows_alloc, a_chunks, a_chunk_rows, a_halves, a_buf_rows;
  // M
  int tiles, tpp, P, M_valid, W_valid;  // tiles per image, tiles per pass, pitch, valid rows, valid columns (ox < W_valid)
  // taps
  int n_taps, kt, tap_group;             // kt = K=16 steps per tap; taps per ring slot
  int pair;                              // forward: the two M tiles of a unit share every weight group (one pass)
  int resident;                          // every tap group of a net has its own ring slot: weights are loaded when the net changes, not per pass
  int hg_major;                          // unit order: head group slowest (consecutive units share their weights) instead of fastest
  int a_shift[MAX_TAPS];                 // rows
  int w_c1[MAX_TAPS], w_c2[MAX_TAPS];    // TMA coordinates (dims 1, 2) of the tap's weight box
  // B tile
  uint32_t b_box_bytes, b_row_bytes;     // bytes of one box (one net), bytes per row (128 or 64)
  int N, ring;
  // epilogue
  int OH, OW, OC;                        // fwd: output geometry; dgrad: OC = IC of the layer (channels per pixel)
  int s, ph, pw, IH, IW;                 // dgrad: block -> pixel mapping
  float scale;
  NetPtr w;                              // fp32 arenas (bias), fwd
  int64_t b_off;
  float* out;                            // fwd: act (+act_off); dgrad: dact of the previous layer (+act_off)
  const bf16* mask_hi;                   // dgrad: X2 hi plane of this layer = its input (relu' mask), [net][img][rows][C2]
  int64_t mask_net_stride, mask_img_rows;
  int64_t out_net_stride;
  PlaneDst dst;
  int debug;
  int tl_id;  // kernel timeline slot (IDQN_F_TIMELINE) or -1
};

__host__ __device__ inline uint32_t round_up(uint32_t x, uint32_t m) { return (x + m - 1) / m * m; }
// unit -> (head group, (input, image) index)
__device__ __forceinline__ void unit_decode(const TapsArgs& p, int u, int& hg, int& gi) {
  if (p.hg_major) {
    const int per = p.n_units_total / p.n_hg;
    hg = u / per, gi = u - hg * per;
  } else {
    hg = u % p.n_hg, gi = u / p.n_hg;
  }
}

struct TapsSmem {
  uint32_t a_plane_bytes, a_buf_bytes, ring_off, slot_bytes, bar_off, total;
};
__host__ __device__ inline TapsSmem taps_smem(const TapsArgs& p, int a_planes) {
  TapsSmem s;
  s.a_plane_bytes = (uint32_t)p.a_halves * p.a_buf_rows * 128;
  s.a_buf_bytes = a_planes * s.a_plane_bytes;
  s.ring_off = 2 * s.a_buf_bytes;
  s.slot_bytes = round_up(2 * p.hpg * p.b_box_bytes * p.tap_group, 1024);
  s.bar_off = s.ring_off + p.ring * s.slot_bytes;
  s.total = s.bar_off + 256 + 1024;  // barriers + alignment slack
  return s;
}

// KIND 0: forward (B = weights MN-major, epilogue bias/relu); KIND 1: dgrad (B = weights K-major, epilogue relu').
// Work is cut into jobs = (unit, M tile); every CTA takes a contiguous, balanced range of jobs, so consecutive jobs
// reuse the image already resident in shared memory.  Weight tiles arrive in groups of `tap_group` taps per ring
// slot (one barrier round trip per group).
// PASSES.  With p.pair (forward layers whose image has two M tiles and whose accumulators fit twice: conv1, conv2) the two
// tiles of a unit that fall into the CTA's job range are processed as ONE pass: every weight group is loaded once and
// multiplied into both tiles' accumulators, which halves the weight traffic -- with two ring slots next to the two
// resident images the MMA thread was waiting ~0.3 us for the next tap's weights after every ~0.5 us of MMAs.
// Split products: the hi and lo weight tiles of a tap sit next to each other in the ring slot, so ONE MMA of width
// 2N computes A_hi*[B_hi | B_lo] (the A tile, the larger operand, is read from shared memory once for both), a
// second MMA of width N adds A_lo*B_hi into the first N columns; the epilogue sums the two column sets.
template <int KIND, int A_PLANES>
__global__ void __launch_bounds__(NTHREADS, 1)
conv_taps_kernel(const __grid_constant__ CUtensorMap mapA_hi, const __grid_constant__ CUtensorMap mapA_lo,
                 const __grid_constant__ CUtensorMap mapW_hi, const __grid_constant__ CUtensorMap mapW_lo,
                 const TapsArgs p) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* smem = smem_raw + (base - smem_u32(smem_raw));
  const TapsSmem L = taps_smem(p, A_PLANES);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + L.bar_off);
  uint64_t* x_full = bars;            // [2]
  uint64_t* x_empty = bars + 2;       // [2]
  uint64_t* acc_full = bars + 4;      // [2]
  uint64_t* acc_empty = bars + 6;     // [2]
  uint64_t* w_full = bars + 8;        // [ring]
  uint64_t* w_empty = bars + 8 + 8;   // [ring]  (ring <= 8)
  __shared__ uint32_t tmem_base_s;

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int N = p.N, N2 = 2 * p.N;   // accumulator columns per tile: [0,N) hi*hi + lo*hi, [N,2N) hi*lo
  const bool pair = p.pair != 0;  // forward conv1 / conv2 and the conv2 data gradient (N = 64: two tiles x 2N columns, twice)
  const int ACCW = (pair ? 2 : 1) * N2;  // columns of one accumulator buffer (one pass)
  uint32_t tmem_cols = 32;
  while ((int)tmem_cols < 2 * ACCW) tmem_cols <<= 1;
  const int n_groups = (p.n_taps + p.tap_group - 1) / p.tap_group;
  const uint32_t tap_bytes = 2u * p.hpg * p.b_box_bytes;  // hi boxes then lo boxes of one tap
  // this CTA's jobs
  const int J = p.n_units * p.tiles;
  const int j0 = (int)((int64_t)blockIdx.x * J / gridDim.x), j1 = (int)((int64_t)(blockIdx.x + 1) * J / gridDim.x);
  // tiles of the pass that starts at job j (pair mode: both tiles of a unit when both are ours)
#define PASS_TILES(j) ((pair && ((j) & 1) == 0 && (j) + 1 < j1) ? 2 : 1)

  // rows of an M tile past the image read whatever follows in shared memory (the other buffer, the ring): they only
  // produce accumulator rows that the epilogue drops
  if (tid == 0) {
    for (int i = 0; i < 2; ++i) {
      mbar_init(&x_full[i], 1), mbar_init(&x_empty[i], 1);
      mbar_init(&acc_full[i], 1), mbar_init(&acc_empty[i], 8);
    }
    for (int i = 0; i < p.ring; ++i) mbar_init(&w_full[i], 1), mbar_init(&w_empty[i], 1);
    fence_mbar_init();
  }
  if (warp == 2) tmem_alloc(&tmem_base_s, tmem_cols);
  fence_proxy_async_smem();
  tcgen05_before_sync();
  __syncthreads();
  tcgen05_after_sync();
  const uint32_t tmem = tmem_base_s;
  if (tid == 0) tl_stamp(p.debug, 1);
  ktl_begin(p.tl_id);
  if (tid == 0) ctl_stamp(p.tl_id, 0);

  if (warp == 0) {
    // ===== image producer: one load per unit this CTA touches =====
    if (elect_one()) {
      pdl_wait();  // the image is produced by the preceding kernels (the weight tiles of warp 1 are not)
      int xi = 0;
      for (int j = j0; j < j1; ++j) {
        if (j != j0 && j % p.tiles != 0) continue;
        const int u = p.unit0 + j / p.tiles, xb = xi & 1;
        mbar_wait(&x_empty[xb], ((xi >> 1) & 1) ^ 1);
        tl_stamp(p.debug, 1000 + xi);
        int hg_, gi;
        unit_decode(p, u, hg_, gi);  // gi = (g, img) linear
        const uint32_t bytes = (uint32_t)A_PLANES * p.a_halves * p.a_chunks * p.a_chunk_rows * 128;
        tma::expect_tx(&x_full[xb], bytes);
        const int row0 = gi * p.a_rows_alloc;
        for (int pl = 0; pl < A_PLANES; ++pl)
          for (int hf = 0; hf < p.a_halves; ++hf)
            for (int ch = 0; ch < p.a_chunks; ++ch) {
              const uint32_t dst = base + xb * L.a_buf_bytes + pl * L.a_plane_bytes + (uint32_t)hf * p.a_buf_rows * 128 +
                                   (uint32_t)ch * p.a_chunk_rows * 128;
              tma::load_3d(dst, pl ? &mapA_lo : &mapA_hi, &x_full[xb], 0, hf, row0 + ch * p.a_chunk_rows);
            }
        ++xi;
      }
    }
  } else if (warp == 1) {
    // ===== weight producer: groups of taps per ring slot, once per pass =====
    if (elect_one()) {
      int ws = 0, pi = 0, last_net0 = -1;
      uint32_t wphase = 0;
      for (int j = j0; j < j1; j += PASS_TILES(j), ++pi) {
        const int u = p.unit0 + j / p.tiles;
        int hg, gi;
        unit_decode(p, u, hg, gi);
        const int g = gi / p.imgs;
        const int net0 = g * p.nets_per_g + hg * p.hpg;
        const int nb = min(p.hpg, p.nets_per_g - hg * p.hpg);
        if (p.resident) {
          // slot = tap group; (re)loaded only when the net changes: the slots' barriers count reloads
          if (net0 == last_net0) continue;
          last_net0 = net0;
        }
        for (int grp = 0; grp < n_groups; ++grp) {
          if (p.resident) ws = grp;
          mbar_wait(&w_empty[ws], wphase ^ 1);
          tl_stamp(p.debug, 2000 + pi * 16 + grp);
          const int tg0 = grp * p.tap_group, tg1 = min(p.n_taps, tg0 + p.tap_group);
          tma::expect_tx(&w_full[ws], 2u * nb * p.b_box_bytes * (tg1 - tg0));
          for (int t = tg0; t < tg1; ++t) {
            const uint32_t slot = base + L.ring_off + ws * L.slot_bytes + (uint32_t)(t - tg0) * tap_bytes;
            for (int jn = 0; jn < nb; ++jn) {
              tma::load_4d(slot + jn * p.b_box_bytes, &mapW_hi, &w_full[ws], 0, p.w_c1[t], p.w_c2[t], net0 + jn);
              tma::load_4d(slot + (p.hpg + jn) * p.b_box_bytes, &mapW_lo, &w_full[ws], 0, p.w_c1[t], p.w_c2[t], net0 + jn);
            }
          }
          if (!p.resident && ++ws == p.ring) ws = 0, wphase ^= 1;
        }
        if (p.resident) wphase ^= 1;
      }
    }
  } else if (warp == 2) {
    // ===== MMA issuer: one elected lane walks the whole pipeline =====
    if (elect_one() && j0 < j1) {
      const uint32_t idesc2 = make_idesc_bf16(128, N2, false, KIND == 0);  // A_hi * [B_hi | B_lo]
      const uint32_t idesc1 = make_idesc_bf16(128, N, false, KIND == 0);   // A_lo * B_hi
      const uint32_t b_lt = p.b_row_bytes == 128 ? tma::LT_SW128 : tma::LT_SW64;
      const uint32_t a_hi32 = tma::desc_hi32(1024, tma::LT_SW128), b_hi32 = tma::desc_hi32(8 * p.b_row_bytes, b_lt);
      const uint32_t half16 = (uint32_t)p.a_buf_rows * 8;                 // next 64-channel half of the image
      const uint32_t bstep = KIND == 0 ? p.b_row_bytes : 2u;              // K = 16 step of B: 16 rows (MN-major) or 32 bytes
      int xi = 0, ws = 0, ai = 0, last_net0 = -1;
      uint32_t wphase = 0;
      bool new_unit = true;
      for (int j = j0; j < j1; ++ai) {
        const int npt = PASS_TILES(j);
        const int tile = j % p.tiles, xb = xi & 1, ab = ai & 1;
        const bool last_job = j + npt >= j1, unit_ends = last_job || tile + npt == p.tiles;
        const uint32_t a_hi = base + xb * L.a_buf_bytes, a_lo = a_hi + L.a_plane_bytes;
        // resident weights: this pass waits for its slots only if its net differs from the previous pass's, and hands them
        // back only if the next pass's does
        bool reload = true, release = true;
        if (p.resident) {
          int hg, gi;
          unit_decode(p, p.unit0 + j / p.tiles, hg, gi);
          const int net0 = (gi / p.imgs) * p.nets_per_g + hg * p.hpg;
          reload = net0 != last_net0;
          last_net0 = net0;
          if (!last_job) {
            unit_decode(p, p.unit0 + (j + npt) / p.tiles, hg, gi);
            release = (gi / p.imgs) * p.nets_per_g + hg * p.hpg != net0;
          }
          if (reload && ai > 0) wphase ^= 1;
        }
        for (int grp = 0; grp < n_groups; ++grp) {
          // waits of this group (the MMAs queued before keep draining meanwhile)
          if (grp == 0) {
            mbar_wait(&acc_empty[ab], ((ai >> 1) & 1) ^ 1);
            if (new_unit) mbar_wait(&x_full[xb], (xi >> 1) & 1);
          }
          if (p.resident) ws = grp;
          if (reload) mbar_wait(&w_full[ws], wphase);
          tcgen05_after_sync();
          if (ai == 0 && grp == 0) ctl_stamp(p.tl_id, 1);
          tl_stamp(p.debug, 3000 + ai * 32 + grp);
          const int tg0 = grp * p.tap_group, tg1 = min(p.n_taps, tg0 + p.tap_group);
          for (int ti = 0; ti < npt; ++ti) {
            const uint32_t d = tmem + (uint32_t)ab * ACCW + (uint32_t)ti * N2;
            for (int t = tg0; t < tg1; ++t) {
              const uint32_t b_hi = base + L.ring_off + ws * L.slot_bytes + (uint32_t)(t - tg0) * tap_bytes;
              // descriptor low words; offsets in 16-byte units.  B: N groups at LBO = box bytes (hi boxes then lo boxes)
              uint32_t bh = tma::desc_lo32(b_hi, p.b_box_bytes);
              uint32_t ah = tma::desc_lo32(a_hi, 16) + (uint32_t)p.a_shift[t] * 8 + (uint32_t)(tile + ti) * 1024;
              uint32_t al = tma::desc_lo32(a_lo, 16) + (uint32_t)p.a_shift[t] * 8 + (uint32_t)(tile + ti) * 1024;
              for (int j4 = 0; j4 < p.kt; j4 += 4) {
#pragma unroll
                for (int jj = 0; jj < 4; ++jj) {
                  if (t == 0 && j4 == 0 && jj == 0) tma::mma_bf16_split<false>(d, ah, a_hi32, bh, b_hi32, idesc2);
                  else tma::mma_bf16_split<true>(d, ah + 2 * jj, a_hi32, bh + jj * bstep, b_hi32, idesc2);
                  if (A_PLANES == 2) tma::mma_bf16_split<true>(d, al + 2 * jj, a_hi32, bh + jj * bstep, b_hi32, idesc1);
                }
                ah += half16, al += half16, bh += 4 * bstep;
              }
            }
          }
          if (release) mma_commit(&w_empty[ws]);
          const bool last_grp = grp == n_groups - 1;
          if (last_grp) {
            mma_commit(&acc_full[ab]);
            if (unit_ends) mma_commit(&x_empty[xb]);
            if (last_job) ctl_stamp(p.tl_id, 2);
          }
          tl_stamp(p.debug, 3000 + ai * 32 + 16 + grp);
          if (!p.resident && ++ws == p.ring) ws = 0, wphase ^= 1;
        }
        new_unit = unit_ends;
        if (unit_ends) ++xi;
        j += npt;
      }
    }
    __syncwarp();
    pdl_trigger();  // the bulk of this CTA's work is queued
  } else {
    // ===== epilogue warps 3..10: TMEM lane quadrant = warp % 4, 32-column chunks of parity (warp - 3) / 4 =====
    const int q = warp & 3, chalf = (warp - 3) >> 2;
    const int r = q * 32 + lane;  // row inside the tile
    pdl_wait();
    int ai = 0;
    for (int j = j0; j < j1; ++ai) {
      const int npt = PASS_TILES(j);
      const int tile0 = j % p.tiles, u = p.unit0 + j / p.tiles;
      int hg, gi;
      unit_decode(p, u, hg, gi);
      const int g = gi / p.imgs, im = gi - g * p.imgs;
      const int net0 = g * p.nets_per_g + hg * p.hpg;
      const int nb = min(p.hpg, p.nets_per_g - hg * p.hpg);
      const int ab = ai & 1;
      j += npt;
      // dgrad: the relu' masks of this thread's 32-column chunks do not depend on the accumulator: they are requested BEFORE
      // the wait for the MMAs, so their L2 latency hides behind the MMA phase.  Two slots: the two chunks (c0, c0 + 64) of a
      // single-tile pass at N = 128, or the one chunk of each tile of a two-tile pass (N = 64)
      uint4 xa[2][4];
      if (KIND == 1) {
#pragma unroll
        for (int kk = 0; kk < 2; ++kk) {
          const int m = (tile0 + (pair ? kk : 0)) * 128 + r;
          const int my = m / p.P, mx = m - my * p.P;
          const bool rowok = m < p.M_valid && mx < p.W_valid && (!pair || kk < npt);
          const int c0 = chalf * 32 + (pair ? 0 : kk * 64);
          const int blk = c0 / p.OC, ry = blk / p.s, rx = blk - ry * p.s;
          const int iy = my * p.s + ry - p.ph, ix = mx * p.s + rx - p.pw;
          const bool ok = c0 < N && rowok && (unsigned)iy < (unsigned)p.IH && (unsigned)ix < (unsigned)p.IW;
          const int64_t mi = ok ? (int64_t)g * p.mask_net_stride + (((int64_t)im * p.mask_img_rows) + m) * N + c0 : 0;
#pragma unroll
          for (int k4 = 0; k4 < 4; ++k4) xa[kk][k4] = __ldg(reinterpret_cast<const uint4*>(p.mask_hi + mi) + k4);
        }
      }
      // forward: likewise the bias of this thread's first chunk (the same for both tiles of a pass)
      float4 bb0[8];
      if (KIND == 0) {
        const int c0 = chalf * 32, hl = c0 / p.OC, oc = c0 - hl * p.OC;
        const int net = net0 + (hl < nb ? hl : 0);
        const float4* bias = reinterpret_cast<const float4*>(p.w.get<float>(net) + p.b_off + oc);
#pragma unroll
        for (int k4 = 0; k4 < 8; ++k4) bb0[k4] = __ldg(bias + k4);
      }
      mbar_wait(&acc_full[ab], (ai >> 1) & 1);
      tcgen05_after_sync();
      if (warp == 3 && lane == 0) tl_stamp(p.debug, 1200 + 2 * ai);
      for (int ti = 0; ti < npt; ++ti) {
      const int m = (tile0 + ti) * 128 + r;
      const int my = m / p.P, mx = m - my * p.P;
      const bool rowok = m < p.M_valid && mx < p.W_valid;
      const uint32_t taddr = tmem + ((uint32_t)(q * 32) << 16) + (uint32_t)ab * ACCW + (uint32_t)ti * N2;
      // per-row bases, computed once per tile
      int64_t orow = 0, prow = 0;
      if (KIND == 0) {
        orow = (((int64_t)im * p.OH + my) * p.OW + mx) * p.OC;
        prow = plane_index(p.dst, 0, im, my, mx);
      }
      // 32 columns per iteration; every load of the iteration (TMEM, bias / relu mask) is issued before the first
      // use so the four epilogue warps expose one memory latency per iteration, not one per access
      for (int c0 = chalf * 32; c0 < N; c0 += 64) {
        float v[32], v2[32];
        tmem_ld16_nowait(taddr + c0, v);
        tmem_ld16_nowait(taddr + c0 + 16, v + 16);
        tmem_ld16_nowait(taddr + N + c0, v2);
        tmem_ld16_nowait(taddr + N + c0 + 16, v2 + 16);
        if (KIND == 0) {
          const int hl = c0 / p.OC, oc = c0 - hl * p.OC;  // 32 | OC: the 32 columns stay inside one head
          const bool ok = rowok && hl < nb;
          const int net = net0 + (ok ? hl : 0);
          const float4* bias = reinterpret_cast<const float4*>(p.w.get<float>(net) + p.b_off + oc);
          float4 bb[8];
#pragma unroll
          for (int k4 = 0; k4 < 8; ++k4) bb[k4] = c0 < 64 ? bb0[k4] : __ldg(bias + k4);
          tmem_ld_wait();
          if (!ok) continue;
          float o[32];
#pragma unroll
          for (int k4 = 0; k4 < 8; ++k4) {
            o[4 * k4] = fmaxf(fmaf(v[4 * k4] + v2[4 * k4], p.scale, bb[k4].x), 0.f);
            o[4 * k4 + 1] = fmaxf(fmaf(v[4 * k4 + 1] + v2[4 * k4 + 1], p.scale, bb[k4].y), 0.f);
            o[4 * k4 + 2] = fmaxf(fmaf(v[4 * k4 + 2] + v2[4 * k4 + 2], p.scale, bb[k4].z), 0.f);
            o[4 * k4 + 3] = fmaxf(fmaf(v[4 * k4 + 3] + v2[4 * k4 + 3], p.scale, bb[k4].w), 0.f);
          }
          if (p.out) {  // fp32 copy only on request: the planes carry the activation (row-per-thread stores are costly)
            float* dst = p.out + (int64_t)net * p.out_net_stride + orow + oc;
#pragma unroll
            for (int k4 = 0; k4 < 8; ++k4)
              reinterpret_cast<float4*>(dst)[k4] = make_float4(o[4 * k4], o[4 * k4 + 1], o[4 * k4 + 2], o[4 * k4 + 3]);
          }
          const int64_t pi = (int64_t)net * p.dst.net_stride + prow + oc;
#pragma unroll
          for (int h8 = 0; h8 < 4; ++h8) {
            uint4 hh, ll;
            split8(o + 8 * h8, hh, ll);
            reinterpret_cast<uint4*>(p.dst.hi + pi)[h8] = hh;
            reinterpret_cast<uint4*>(p.dst.lo + pi)[h8] = ll;
          }
        } else {
          // row = block (my, mx) of the layer input; columns (ry, rx, c): 32 channels of one input pixel (32 | IC)
          const int blk = c0 / p.OC, c = c0 - blk * p.OC;
          const int ry = blk / p.s, rx = blk - ry * p.s;
          const int iy = my * p.s + ry - p.ph, ix = mx * p.s + rx - p.pw;
          const bool ok = rowok && (unsigned)iy < (unsigned)p.IH && (unsigned)ix < (unsigned)p.IW;
          // relu' mask: the layer input is this very row of the X2 hi plane (hi > 0 <=> x > 0), 32 contiguous bf16
          const int kk = pair ? ti : c0 >> 6;  // mask slot: the tile of a two-tile pass, else this thread's chunk index (N <= 128)
          tmem_ld_wait();
          if (!ok) continue;
          float o[32];
#pragma unroll
          for (int k4 = 0; k4 < 4; ++k4) {
            const uint4 xv = kk ? xa[1][k4] : xa[0][k4];
            const uint32_t w[4] = {xv.x, xv.y, xv.z, xv.w};
#pragma unroll
            for (int e = 0; e < 8; ++e) {
              const uint32_t bits = (w[e >> 1] >> (16 * (e & 1))) & 0xffffu;
              const bool pos = bits != 0 && !(bits & 0x8000u);  // bf16 > 0
              o[8 * k4 + e] = pos ? v[8 * k4 + e] + v2[8 * k4 + e] : 0.f;
            }
          }
          if (p.out) {
            const int64_t oi = (int64_t)g * p.out_net_stride + (((int64_t)im * p.IH + iy) * p.IW + ix) * p.OC + c;
#pragma unroll
            for (int k4 = 0; k4 < 8; ++k4)
              reinterpret_cast<float4*>(p.out + oi)[k4] = make_float4(o[4 * k4], o[4 * k4 + 1], o[4 * k4 + 2], o[4 * k4 + 3]);
          }
          const int64_t pi = plane_index(p.dst, g, im, iy, ix) + c;
#pragma unroll
          for (int h8 = 0; h8 < 4; ++h8) {
            uint4 hh, ll;
            split8(o + 8 * h8, hh, ll);
            reinterpret_cast<uint4*>(p.dst.hi + pi)[h8] = hh;
            reinterpret_cast<uint4*>(p.dst.lo + pi)[h8] = ll;
          }
        }
      }
      }
      tcgen05_before_sync();
      __syncwarp();
      if (warp == 3 && lane == 0) tl_stamp(p.debug, 1201 + 2 * ai);
      if (lane == 0) tma::arrive(&acc_empty[ab]);
    }
  }
#undef PASS_TILES
  tcgen05_before_sync();
  __syncthreads();
  if (tid == 0) ctl_stamp(p.tl_id, 3);
  ktl_end(p.tl_id);
  if (warp == 2) tmem_dealloc(tmem, tmem_cols);
}

// ------------------------------------------------------------------------------------------------------
// conv1 -> conv2 FORWARD CHAIN: one CTA takes a (net, image) unit through BOTH layers; the intermediate activation
// (11 x 11 x 64, as the pitched 13 x 15 space-to-depth image conv2 reads) never leaves the SM: the epilogue of stage A
// writes its bf16 hi / lo planes straight into shared memory in the SWIZZLE_128B layout the stage-B MMAs read.  One
// launch and one pass over the units instead of two kernels with a grid-wide boundary between them (each paid ~3 us
// to its first MMA, ~2 us for its last epilogue and the tail imbalance of the layer before).
//   shared memory: image A (conv1 input, both planes, single buffer: it is free again while stage B runs) | image B
//   (conv2 input, both planes) | weight ring shared by both stages (stage A: one tap per slot, stage B: two)
//   TMEM: stage A accumulators (2 tiles x 2N) in columns [0, 256), stage B in [256, 512): the epilogue of B(u) overlaps
//   the MMAs of A(u+1)
// Both stages are two-tile passes of conv_taps_kernel<0, 2>; the arithmetic (tap order, split products, epilogue) is the
// same instruction sequence, so the results are bit-identical to the two-kernel path.
struct ChainArgs {
  TapsArgs a, b;   // conv1 / conv2 forward as set up for conv_taps_kernel (geometry, taps, TMA coordinates, epilogue)
  int bP, b_off_y, b_off_x;  // where stage A's output pixel (y, x) lands in image B: row (y + off_y) * bP + (x + off_x)
  int b_tap_group;           // taps of stage B per ring slot
  int ring;
};
struct ChainSmem {
  uint32_t a_plane, a_bytes, b_plane, b_bytes, ring_off, slot_bytes, bar_off, total;
};
__host__ __device__ inline ChainSmem chain_smem(const ChainArgs& c) {
  ChainSmem s;
  s.a_plane = (uint32_t)c.a.a_halves * c.a.a_buf_rows * 128;
  s.a_bytes = 2 * s.a_plane;
  s.b_plane = round_up((uint32_t)c.b.a_halves * c.b.a_buf_rows * 128, 1024);
  s.b_bytes = 2 * s.b_plane;
  s.ring_off = s.a_bytes + s.b_bytes;
  const uint32_t sa = 2 * c.a.b_box_bytes, sb = 2 * c.b.b_box_bytes * c.b_tap_group;
  s.slot_bytes = round_up(sa > sb ? sa : sb, 1024);
  s.bar_off = s.ring_off + c.ring * s.slot_bytes;
  s.total = s.bar_off + 256 + 1024;
  return s;
}

__global__ void __launch_bounds__(NTHREADS, 1)
conv_chain_fwd_kernel(const __grid_constant__ CUtensorMap mapA_hi, const __grid_constant__ CUtensorMap mapA_lo,
                      const __grid_constant__ CUtensorMap mapWa_hi, const __grid_constant__ CUtensorMap mapWa_lo,
                      const __grid_constant__ CUtensorMap mapWb_hi, const __grid_constant__ CUtensorMap mapWb_lo,
                      const ChainArgs c) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* smem = smem_raw + (base - smem_u32(smem_raw));
  const ChainSmem L = chain_smem(c);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + L.bar_off);
  uint64_t* x_full = bars;          // image A landed
  uint64_t* x_empty = bars + 1;     // stage-A MMAs reading it complete
  uint64_t* bimg_full = bars + 2;   // image B written by the stage-A epilogue (8 warps)
  uint64_t* bimg_empty = bars + 3;  // stage-B MMAs reading it complete
  uint64_t* accA_full = bars + 4;
  uint64_t* accA_empty = bars + 5;  // 8 warps
  uint64_t* accB_full = bars + 6;
  uint64_t* accB_empty = bars + 7;  // 8 warps
  uint64_t* w_full = bars + 8;      // [ring]
  uint64_t* w_empty = bars + 16;    // [ring]
  __shared__ uint32_t tmem_base_s;

  const TapsArgs& pa = c.a;
  const TapsArgs& pb = c.b;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int N = pa.N, N2 = 2 * N;  // 64 / 128 in both stages
  const int u0 = (int)((int64_t)blockIdx.x * pa.n_units / gridDim.x), u1 = (int)((int64_t)(blockIdx.x + 1) * pa.n_units / gridDim.x);
  const int ngA = pa.n_taps, ngB = (pb.n_taps + c.b_tap_group - 1) / c.b_tap_group;

  // image B: the zero border of the padded conv2 input is written once here and never touched again
  for (uint32_t i = tid; i < L.b_bytes / 16; i += NTHREADS) reinterpret_cast<uint4*>(smem + L.a_bytes)[i] = make_uint4(0, 0, 0, 0);
  if (tid == 0) {
    mbar_init(x_full, 1), mbar_init(x_empty, 1), mbar_init(bimg_full, 8), mbar_init(bimg_empty, 1);
    mbar_init(accA_full, 1), mbar_init(accA_empty, 8), mbar_init(accB_full, 1), mbar_init(accB_empty, 8);
    for (int i = 0; i < c.ring; ++i) mbar_init(&w_full[i], 1), mbar_init(&w_empty[i], 1);
    fence_mbar_init();
  }
  if (warp == 2) tmem_alloc(&tmem_base_s, 512);
  fence_proxy_async_smem();
  tcgen05_before_sync();
  __syncthreads();
  tcgen05_after_sync();
  const uint32_t tmem = tmem_base_s;
  ktl_begin(pa.tl_id);

  if (warp == 0) {
    // ===== image A producer =====
    if (elect_one()) {
      pdl_wait();
      for (int u = u0, i = 0; u < u1; ++u, ++i) {
        mbar_wait(x_empty, (i & 1) ^ 1);
        const uint32_t bytes = 2u * pa.a_halves * pa.a_chunks * pa.a_chunk_rows * 128;
        tma::expect_tx(x_full, bytes);
        const int row0 = u * pa.a_rows_alloc;  // unit = (net, image) linear, as the X2 planes of conv1 are laid out
        for (int pl = 0; pl < 2; ++pl)
          for (int hf = 0; hf < pa.a_halves; ++hf)
            for (int ch = 0; ch < pa.a_chunks; ++ch)
              tma::load_3d(base + pl * L.a_plane + (uint32_t)hf * pa.a_buf_rows * 128 + (uint32_t)ch * pa.a_chunk_rows * 128,
                           pl ? &mapA_lo : &mapA_hi, x_full, 0, hf, row0 + ch * pa.a_chunk_rows);
      }
    }
  } else if (warp == 1) {
    // ===== weight producer: stage A groups (one tap each), then stage B groups, through one ring =====
    if (elect_one()) {
      int ws = 0;
      uint32_t wphase = 0;
      for (int u = u0; u < u1; ++u) {
        const int net = u / pa.imgs;
        for (int t = 0; t < ngA; ++t) {
          mbar_wait(&w_empty[ws], wphase ^ 1);
          tma::expect_tx(&w_full[ws], 2u * pa.b_box_bytes);
          const uint32_t slot = base + L.ring_off + ws * L.slot_bytes;
          tma::load_4d(slot, &mapWa_hi, &w_full[ws], 0, pa.w_c1[t], pa.w_c2[t], net);
          tma::load_4d(slot + pa.b_box_bytes, &mapWa_lo, &w_full[ws], 0, pa.w_c1[t], pa.w_c2[t], net);
          if (++ws == c.ring) ws = 0, wphase ^= 1;
        }
        for (int grp = 0; grp < ngB; ++grp) {
          mbar_wait(&w_empty[ws], wphase ^ 1);
          const int tg0 = grp * c.b_tap_group, tg1 = min(pb.n_taps, tg0 + c.b_tap_group);
          tma::expect_tx(&w_full[ws], 2u * pb.b_box_bytes * (tg1 - tg0));
          for (int t = tg0; t < tg1; ++t) {
            const uint32_t slot = base + L.ring_off + ws * L.slot_bytes + (uint32_t)(t - tg0) * 2u * pb.b_box_bytes;
            tma::load_4d(slot, &mapWb_hi, &w_full[ws], 0, pb.w_c1[t], pb.w_c2[t], net);
            tma::load_4d(slot + pb.b_box_bytes, &mapWb_lo, &w_full[ws], 0, pb.w_c1[t], pb.w_c2[t], net);
          }
          if (++ws == c.ring) ws = 0, wphase ^= 1;
        }
      }
    }
  } else if (warp == 2) {
    // ===== MMA issuer =====
    if (elect_one() && u0 < u1) {
      const uint32_t idesc2 = make_idesc_bf16(128, N2, false, true), idesc1 = make_idesc_bf16(128, N, false, true);
      const uint32_t a_hi32 = tma::desc_hi32(1024, tma::LT_SW128);
      const uint32_t wa_hi32 = tma::desc_hi32(8 * pa.b_row_bytes, pa.b_row_bytes == 128 ? tma::LT_SW128 : tma::LT_SW64);
      const uint32_t wb_hi32 = tma::desc_hi32(8 * pb.b_row_bytes, pb.b_row_bytes == 128 ? tma::LT_SW128 : tma::LT_SW64);
      const uint32_t imgA_hi = base, imgA_lo = base + L.a_plane, imgB_hi = base + L.a_bytes, imgB_lo = imgB_hi + L.b_plane;
      int ws = 0;
      uint32_t wphase = 0;
      for (int u = u0, i = 0; u < u1; ++u, ++i) {
        // ---- stage A: conv1, both tiles per tap ----
        mbar_wait(accA_empty, (i & 1) ^ 1);
        mbar_wait(x_full, i & 1);
        for (int t = 0; t < ngA; ++t) {
          mbar_wait(&w_full[ws], wphase);
          tcgen05_after_sync();
          const uint32_t wslot = base + L.ring_off + ws * L.slot_bytes;
          for (int ti = 0; ti < 2; ++ti) {
            const uint32_t d = tmem + (uint32_t)ti * N2;
            uint32_t bh = tma::desc_lo32(wslot, pa.b_box_bytes);
            uint32_t ah = tma::desc_lo32(imgA_hi, 16) + (uint32_t)pa.a_shift[t] * 8 + (uint32_t)ti * 1024;
            uint32_t al = tma::desc_lo32(imgA_lo, 16) + (uint32_t)pa.a_shift[t] * 8 + (uint32_t)ti * 1024;
            for (int j4 = 0; j4 < pa.kt; j4 += 4) {
#pragma unroll
              for (int jj = 0; jj < 4; ++jj) {
                if (t == 0 && j4 == 0 && jj == 0) tma::mma_bf16_split<false>(d, ah, a_hi32, bh, wa_hi32, idesc2);
                else tma::mma_bf16_split<true>(d, ah + 2 * jj, a_hi32, bh + jj * pa.b_row_bytes, wa_hi32, idesc2);
                tma::mma_bf16_split<true>(d, al + 2 * jj, a_hi32, bh + jj * pa.b_row_bytes, wa_hi32, idesc1);
              }
              ah += (uint32_t)pa.a_buf_rows * 8, al += (uint32_t)pa.a_buf_rows * 8, bh += 4 * pa.b_row_bytes;
            }
          }
          mma_commit(&w_empty[ws]);
          if (++ws == c.ring) ws = 0, wphase ^= 1;
        }
        mma_commit(accA_full);
        mma_commit(x_empty);
        // ---- stage B: conv2 on the image the stage-A epilogue is writing into shared memory ----
        mbar_wait(accB_empty, (i & 1) ^ 1);
        mbar_wait(bimg_full, i & 1);
        for (int grp = 0; grp < ngB; ++grp) {
          mbar_wait(&w_full[ws], wphase);
          tcgen05_after_sync();
          const int tg0 = grp * c.b_tap_group, tg1 = min(pb.n_taps, tg0 + c.b_tap_group);
          for (int ti = 0; ti < 2; ++ti) {
            const uint32_t d = tmem + 256u + (uint32_t)ti * N2;
            for (int t = tg0; t < tg1; ++t) {
              const uint32_t wslot = base + L.ring_off + ws * L.slot_bytes + (uint32_t)(t - tg0) * 2u * pb.b_box_bytes;
              uint32_t bh = tma::desc_lo32(wslot, pb.b_box_bytes);
              uint32_t ah = tma::desc_lo32(imgB_hi, 16) + (uint32_t)pb.a_shift[t] * 8 + (uint32_t)ti * 1024;
              uint32_t al = tma::desc_lo32(imgB_lo, 16) + (uint32_t)pb.a_shift[t] * 8 + (uint32_t)ti * 1024;
              for (int j4 = 0; j4 < pb.kt; j4 += 4) {
#pragma unroll
                for (int jj = 0; jj < 4; ++jj) {
                  if (t == 0 && j4 == 0 && jj == 0) tma::mma_bf16_split<false>(d, ah, a_hi32, bh, wb_hi32, idesc2);
                  else tma::mma_bf16_split<true>(d, ah + 2 * jj, a_hi32, bh + jj * pb.b_row_bytes, wb_hi32, idesc2);
                  tma::mma_bf16_split<true>(d, al + 2 * jj, a_hi32, bh + jj * pb.b_row_bytes, wb_hi32, idesc1);
                }
                ah += (uint32_t)pb.a_buf_rows * 8, al += (uint32_t)pb.a_buf_rows * 8, bh += 4 * pb.b_row_bytes;
              }
            }
          }
          mma_commit(&w_empty[ws]);
          if (++ws == c.ring) ws = 0, wphase ^= 1;
        }
        mma_commit(accB_full);
        mma_commit(bimg_empty);
      }
    }
    __syncwarp();
    pdl_trigger();
  } else {
    // ===== epilogue warps 3..10: TMEM lane quadrant = warp % 4, 32-column chunk (warp - 3) / 4 of the 64 channels =====
    const int q = warp & 3, chalf = (warp - 3) >> 2;
    const int r = q * 32 + lane;
    const int c0 = chalf * 32;
    uint8_t* imgB = smem + L.a_bytes;
    pdl_wait();
    for (int u = u0, i = 0; u < u1; ++u, ++i) {
      const int net = u / pa.imgs, im = u - net * pa.imgs;
      // biases of both layers for this thread's 32 channels: requested before the first accumulator wait
      float4 ba[8], bb[8];
      {
        const float4* pa_bias = reinterpret_cast<const float4*>(pa.w.get<float>(net) + pa.b_off + c0);
        const float4* pb_bias = reinterpret_cast<const float4*>(pb.w.get<float>(net) + pb.b_off + c0);
#pragma unroll
        for (int k4 = 0; k4 < 8; ++k4) ba[k4] = __ldg(pa_bias + k4), bb[k4] = __ldg(pb_bias + k4);
      }
      // ---- stage A epilogue: relu(conv1) -> bf16 hi / lo planes of image B in shared memory ----
      mbar_wait(bimg_empty, (i & 1) ^ 1);  // the previous unit's stage-B MMAs have read image B
      mbar_wait(accA_full, i & 1);
      tcgen05_after_sync();
      for (int ti = 0; ti < 2; ++ti) {
        const int m = ti * 128 + r;
        const int my = m / pa.P, mx = m - my * pa.P;
        const bool rowok = m < pa.M_valid && mx < pa.W_valid;
        const uint32_t taddr = tmem + ((uint32_t)(q * 32) << 16) + (uint32_t)ti * N2;
        float v[32], v2[32];
        tmem_ld16_nowait(taddr + c0, v);
        tmem_ld16_nowait(taddr + c0 + 16, v + 16);
        tmem_ld16_nowait(taddr + N + c0, v2);
        tmem_ld16_nowait(taddr + N + c0 + 16, v2 + 16);
        tmem_ld_wait();
        if (!rowok) continue;
        float o[32];
#pragma unroll
        for (int k4 = 0; k4 < 8; ++k4) {
          o[4 * k4] = fmaxf(fmaf(v[4 * k4] + v2[4 * k4], pa.scale, ba[k4].x), 0.f);
          o[4 * k4 + 1] = fmaxf(fmaf(v[4 * k4 + 1] + v2[4 * k4 + 1], pa.scale, ba[k4].y), 0.f);
          o[4 * k4 + 2] = fmaxf(fmaf(v[4 * k4 + 2] + v2[4 * k4 + 2], pa.scale, ba[k4].z), 0.f);
          o[4 * k4 + 3] = fmaxf(fmaf(v[4 * k4 + 3] + v2[4 * k4 + 3], pa.scale, ba[k4].w), 0.f);
        }
        // image B row of output pixel (my, mx); 128-byte rows, 16-byte chunk j stored at j ^ (row & 7) (SWIZZLE_128B)
        const int row = (my + c.b_off_y) * c.bP + mx + c.b_off_x;
        uint8_t* rowp = imgB + (uint32_t)row * 128;
#pragma unroll
        for (int h8 = 0; h8 < 4; ++h8) {
          uint4 hh, ll;
          split8(o + 8 * h8, hh, ll);
          const uint32_t chunk = (uint32_t)(((c0 >> 3) + h8) ^ (row & 7)) << 4;
          *reinterpret_cast<uint4*>(rowp + chunk) = hh;
          *reinterpret_cast<uint4*>(rowp + L.b_plane + chunk) = ll;
          if (net < pa.w.zsplit) {
            // online heads: the backward pass reads this activation (relu' mask of conv2's data gradient, operand of its
            // weight gradient) from the conv2 input planes in global memory; target nets never need it again
            const int64_t pi = (int64_t)net * pa.dst.net_stride + plane_index(pa.dst, 0, im, my, mx) + c0;
            reinterpret_cast<uint4*>(pa.dst.hi + pi)[h8] = hh;
            reinterpret_cast<uint4*>(pa.dst.lo + pi)[h8] = ll;
          }
        }
      }
      fence_proxy_async_smem();  // generic-proxy writes of image B -> visible to the stage-B MMAs
      tcgen05_before_sync();
      __syncwarp();
      if (lane == 0) {
        tma::arrive(accA_empty);
        tma::arrive(bimg_full);
      }
      // ---- stage B epilogue: relu(conv2) -> planes of the Dense_0 input in global memory ----
      mbar_wait(accB_full, i & 1);
      tcgen05_after_sync();
      for (int ti = 0; ti < 2; ++ti) {
        const int m = ti * 128 + r;
        const int my = m / pb.P, mx = m - my * pb.P;
        const bool rowok = m < pb.M_valid && mx < pb.W_valid;
        const uint32_t taddr = tmem + ((uint32_t)(q * 32) << 16) + 256u + (uint32_t)ti * N2;
        float v[32], v2[32];
        tmem_ld16_nowait(taddr + c0, v);
        tmem_ld16_nowait(taddr + c0 + 16, v + 16);
        tmem_ld16_nowait(taddr + N + c0, v2);
        tmem_ld16_nowait(taddr + N + c0 + 16, v2 + 16);
        tmem_ld_wait();
        if (!rowok) continue;
        float o[32];
#pragma unroll
        for (int k4 = 0; k4 < 8; ++k4) {
          o[4 * k4] = fmaxf(fmaf(v[4 * k4] + v2[4 * k4], pb.scale, bb[k4].x), 0.f);
          o[4 * k4 + 1] = fmaxf(fmaf(v[4 * k4 + 1] + v2[4 * k4 + 1], pb.scale, bb[k4].y), 0.f);
          o[4 * k4 + 2] = fmaxf(fmaf(v[4 * k4 + 2] + v2[4 * k4 + 2], pb.scale, bb[k4].z), 0.f);
          o[4 * k4 + 3] = fmaxf(fmaf(v[4 * k4 + 3] + v2[4 * k4 + 3], pb.scale, bb[k4].w), 0.f);
        }
        const int64_t pi = (int64_t)net * pb.dst.net_stride + plane_index(pb.dst, 0, im, my, mx) + c0;
#pragma unroll
        for (int h8 = 0; h8 < 4; ++h8) {
          uint4 hh, ll;
          split8(o + 8 * h8, hh, ll);
          reinterpret_cast<uint4*>(pb.dst.hi + pi)[h8] = hh;
          reinterpret_cast<uint4*>(pb.dst.lo + pi)[h8] = ll;
        }
      }
      tcgen05_before_sync();
      __syncwarp();
      if (lane == 0) tma::arrive(accB_empty);
    }
  }
  tcgen05_before_sync();
  __syncthreads();
  ktl_end(pa.tl_id);
  if (warp == 2) tmem_dealloc(tmem, 512);
}

// ------------------------------------------------------------------------------------------------------
// weight gradient.  CTA = (head z, image range); accumulators of all M tiles live in TMEM across the images.
struct WgradArgs {
  int heads, groups, imgs;          // grid = heads * groups * tsplit; CTA handles images [gidx*ipg, min(imgs, +ipg))
  int ipg;
  int tsplit, tps;                  // the layer's M tiles are split over tsplit CTAs, tps tiles each
  int x_shared;                     // 1: every head reads the same X2 images (first layer: the staged batch)
  // images
  int x_rows_alloc, x_chunks, x_chunk_rows, x_halves, x_buf_rows;
  int z_rows_alloc, z_chunks, z_chunk_rows, z_buf_rows;
  uint32_t z_row_bytes;             // 128 (OC = 64) or 64 (OC = 32)
  int z_start;                      // (T-1)(P+1): row of dyZ that pairs with X2 row 0
  int k16;                          // K = 16 steps per image (ceil(OH*P / 16))
  // PARTS: an image is streamed as n_parts consecutive ranges [pj[i], pj[i+1]) of its K = 16 steps through TWO buffers
  // (part i+1 loads while part i multiplies; the step order -- hence every rounding -- is that of one whole image).  The
  // x_* / z_* box fields above then describe the box of ONE part: X rows [16 pj, 16 pj + x_buf_rows), dyZ rows from z_start + 16 pj
  int n_parts, pj[4];
  // M tiles: tile i covers two 64-row groups; group 0 at row shift sh0[i] (+ half h0[i]), group 1 at sh1 / h1
  int n_tiles;
  int sh0[MAX_TAPS], sh1[MAX_TAPS], hf0[MAX_TAPS], hf1[MAX_TAPS];
  int row0[MAX_TAPS], row1[MAX_TAPS];  // arena row (of the [Kd][OC] kernel) of group 0 / group 1 row 0; -1 = unused
  int grp_rows;                     // arena rows per 64-row group that are valid (64, or s*IC runs: see row_map)
  int run, run_stride;              // group row j -> arena row  rowX + (j / run) * run_stride + j % run
  int N;                            // OC
  float scale;
  float* part;                      // [heads][groups][span] partial gradients in arena coordinates
  int64_t span, w_off, b_off;       // floats per partial; arena offsets of this layer's kernel / bias
  int debug;
  int tl_id;
};
struct WgradSmem {
  uint32_t x_plane_bytes, x_bytes, z_plane_bytes, z_bytes, buf_bytes, ones_off, bar_off, total;
};
__host__ __device__ inline WgradSmem wgrad_smem(const WgradArgs& p, int a_planes) {
  WgradSmem s;
  s.x_plane_bytes = (uint32_t)p.x_halves * p.x_buf_rows * 128;
  s.x_bytes = a_planes * s.x_plane_bytes;
  s.z_plane_bytes = round_up((uint32_t)p.z_buf_rows * p.z_row_bytes, 1024);
  s.z_bytes = 2 * s.z_plane_bytes;
  s.buf_bytes = s.x_bytes + s.z_bytes;  // one buffer = the X planes and the dyZ planes of one part
  s.ones_off = 2 * s.buf_bytes;
  s.bar_off = s.ones_off + 2048;
  s.total = s.bar_off + 64 + 1024;
  return s;
}

// what the MMA-issuing thread of conv_wgrad_kernel needs per K = 16 step
struct WgradIssue {
  const uint32_t* xlo;   // per tile: descriptor low word of the X hi plane at k = 0
  uint32_t x0, x1, x2;   // the first three of them by value (registers) for the specialised loops
  uint32_t xpl16, x_hi32, zh0, z_hi32, tmem, N2, idesc2, idesc1, dbias, ones_lo, z_row_bytes;
  bool has_bias;
  uint32_t boff;         // 16-byte units added to every X / dyZ descriptor: the buffer of the current part
  int j0;                // first K = 16 step of the current part (descriptor offsets are relative to the part)
};
// generic step (any tile count; ACC = false: the very first step of the CTA, which initialises the accumulators)
template <int A_PLANES, bool ACC>
__device__ __forceinline__ void wgrad_issue_step(const WgradIssue& w, int nt, int j) {
  const uint32_t zh = w.zh0 + w.boff + (uint32_t)(j - w.j0) * w.z_row_bytes;  // 16 rows = row_bytes 16-byte units
  const uint32_t xk = w.boff + (uint32_t)(j - w.j0) * 128;                    // 16 rows of 128 bytes
  for (int t = 0; t < nt; ++t) {
    const uint32_t d = w.tmem + (uint32_t)t * w.N2;
    tma::mma_bf16_split<ACC>(d, w.xlo[t] + xk, w.x_hi32, zh, w.z_hi32, w.idesc2);
    if (A_PLANES == 2) tma::mma_bf16_split<true>(d, w.xlo[t] + xk + w.xpl16, w.x_hi32, zh, w.z_hi32, w.idesc1);
  }
  if (w.has_bias) tma::mma_bf16_split<ACC>(w.dbias, w.ones_lo, w.x_hi32, zh, w.z_hi32, w.idesc2);  // ones^T [dy_hi | dy_lo]
}
// accumulating step with a compile-time tile count: straight-line code
template <int A_PLANES, int NT>
__device__ __forceinline__ void wgrad_issue_tiles(const WgradIssue& w, int j) {
  const uint32_t zh = w.zh0 + w.boff + (uint32_t)(j - w.j0) * w.z_row_bytes;
  const uint32_t xk = w.boff + (uint32_t)(j - w.j0) * 128;
#pragma unroll
  for (int t = 0; t < NT; ++t) {
    const uint32_t d = w.tmem + (uint32_t)t * w.N2;
    const uint32_t x = (t == 0 ? w.x0 : (t == 1 ? w.x1 : w.x2)) + xk;
    tma::mma_bf16_split<true>(d, x, w.x_hi32, zh, w.z_hi32, w.idesc2);
    if (A_PLANES == 2) tma::mma_bf16_split<true>(d, x + w.xpl16, w.x_hi32, zh, w.z_hi32, w.idesc1);
  }
  if (w.has_bias) tma::mma_bf16_split<true>(w.dbias, w.ones_lo, w.x_hi32, zh, w.z_hi32, w.idesc2);
}

// CTA = (head z, image range, tile split ts): tiles [ts*tps, (ts+1)*tps) of the layer, the last split also owns the
// bias tile.  Per K = 16 step and tile: X_hi^T * [dy_hi | dy_lo] (one MMA, width 2N; the two dy planes are N groups
// LBO = plane bytes apart) + X_lo^T * dy_hi (width N); the epilogue sums the two column sets.
template <int A_PLANES>
__global__ void __launch_bounds__(WG_THREADS, 1)
conv_wgrad_kernel(const __grid_constant__ CUtensorMap mapX_hi, const __grid_constant__ CUtensorMap mapX_lo,
                  const __grid_constant__ CUtensorMap mapZ_hi, const __grid_constant__ CUtensorMap mapZ_lo,
                  const WgradArgs p) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* smem = smem_raw + (base - smem_u32(smem_raw));
  const WgradSmem L = wgrad_smem(p, A_PLANES);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + L.bar_off);
  uint64_t* full = bars;       // [2] part landed in buffer b
  uint64_t* empty = bars + 2;  // [2] MMAs reading buffer b complete
  uint64_t* done = bars + 4;   // all MMAs of the CTA complete
  __shared__ uint32_t tmem_base_s;

  pdl_trigger();
  ktl_begin(p.tl_id);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int ts = blockIdx.x % p.tsplit, zg = blockIdx.x / p.tsplit;
  const int z = zg / p.groups, gidx = zg - z * p.groups;
  const int im0 = gidx * p.ipg, im1 = min(p.imgs, im0 + p.ipg);
  const int t_lo = ts * p.tps, t_hi = min(p.n_tiles, t_lo + p.tps);
  const int nt = t_hi - t_lo;                  // tiles of this CTA
  const bool has_bias = ts == p.tsplit - 1;    // + the bias tile
  const int N = p.N, N2 = 2 * p.N;
  const int ncols = (nt + (has_bias ? 1 : 0)) * N2;
  uint32_t tmem_cols = 32;
  while ((int)tmem_cols < ncols) tmem_cols <<= 1;

  for (uint32_t i = tid; i < L.bar_off / 16; i += WG_THREADS) reinterpret_cast<uint4*>(smem)[i] = make_uint4(0, 0, 0, 0);
  __syncthreads();
  // ones tile (MN-major SW128, 16 k-rows x 64 m): element (k, m = 0) = 1 -> accumulator row 0 = sum_k dy[k][:]
  if (tid < 16) {
    // row k at k*128 bytes; 16-byte chunk 0 of row k sits at chunk (0 ^ (k & 7))
    bf16* row = reinterpret_cast<bf16*>(smem + L.ones_off + tid * 128 + ((tid & 7) << 4));
    row[0] = __float2bfloat16(1.0f);
  }
  if (tid == 0) {
    mbar_init(&full[0], 1), mbar_init(&full[1], 1), mbar_init(&empty[0], 1), mbar_init(&empty[1], 1), mbar_init(done, 1);
    fence_mbar_init();
  }
  if (warp == 1) tmem_alloc(&tmem_base_s, tmem_cols);
  fence_proxy_async_smem();
  tcgen05_before_sync();
  __syncthreads();
  tcgen05_after_sync();
  const uint32_t tmem = tmem_base_s;
  const uint32_t xs = base, zs = base + L.x_bytes;
  if (tid == 0) tl_stamp(p.debug, 1);

  if (warp == 0) {
    pdl_wait();
    int i = 0;
    for (int im = im0; im < im1; ++im) {
      for (int part = 0; part < p.n_parts; ++part, ++i) {
        const int b = i & 1;
        mbar_wait(&empty[b], ((i >> 1) & 1) ^ 1);
        if (elect_one()) {
          tl_stamp(p.debug, 1000 + i);
          const uint32_t bytes = (uint32_t)A_PLANES * p.x_halves * p.x_chunks * p.x_chunk_rows * 128 +
                                 2u * p.z_chunks * p.z_chunk_rows * p.z_row_bytes;
          tma::expect_tx(&full[b], bytes);
          const int xrow = ((p.x_shared ? 0 : z) * p.imgs + im) * p.x_rows_alloc + 16 * p.pj[part];
          const int zrow = (z * p.imgs + im) * p.z_rows_alloc + p.z_start + 16 * p.pj[part];
          const uint32_t xb = xs + b * L.buf_bytes, zb = zs + b * L.buf_bytes;
          for (int pl = 0; pl < A_PLANES; ++pl)
            for (int hf = 0; hf < p.x_halves; ++hf)
              for (int ch = 0; ch < p.x_chunks; ++ch)
                tma::load_3d(xb + pl * L.x_plane_bytes + (uint32_t)hf * p.x_buf_rows * 128 + (uint32_t)ch * p.x_chunk_rows * 128,
                             pl ? &mapX_lo : &mapX_hi, &full[b], 0, hf, xrow + ch * p.x_chunk_rows);
          for (int pl = 0; pl < 2; ++pl)
            for (int ch = 0; ch < p.z_chunks; ++ch)
              tma::load_3d(zb + pl * L.z_plane_bytes + (uint32_t)ch * p.z_chunk_rows * p.z_row_bytes, pl ? &mapZ_lo : &mapZ_hi,
                           &full[b], 0, 0, zrow + ch * p.z_chunk_rows);
        }
        __syncwarp();
      }
    }
  } else if (warp == 1) {
    {
      const uint32_t idesc2 = make_idesc_bf16(128, N2, true, true), idesc1 = make_idesc_bf16(128, N, true, true);
      const uint32_t z_lt = p.z_row_bytes == 128 ? tma::LT_SW128 : tma::LT_SW64;
      const uint32_t x_hi32 = tma::desc_hi32(1024, tma::LT_SW128), z_hi32 = tma::desc_hi32(8 * p.z_row_bytes, z_lt);
      // per tile: descriptor low word of the hi plane at k = 0 (start address | LBO = distance to the second M group)
      uint32_t xlo[MAX_TAPS];
#pragma unroll
      for (int t = 0; t < MAX_TAPS; ++t) {
        if (t < nt) {
          const int tt = t_lo + t;
          const uint32_t o0 = (uint32_t)p.hf0[tt] * p.x_buf_rows * 128 + (uint32_t)p.sh0[tt] * 128;
          const uint32_t o1 = (uint32_t)p.hf1[tt] * p.x_buf_rows * 128 + (uint32_t)p.sh1[tt] * 128;
          xlo[t] = tma::desc_lo32(xs + o0, o1 - o0);
        }
      }
      const uint32_t xpl16 = L.x_plane_bytes >> 4, ones_lo = tma::desc_lo32(base + L.ones_off, 16);
      // B = [dy_hi | dy_lo]: the lo plane is the second N group, LBO = plane bytes
      const uint32_t zh0 = tma::desc_lo32(zs, L.z_plane_bytes);  // the part's box starts at dyZ row z_start + 16 pj
      const uint32_t dbias = tmem + (uint32_t)nt * N2;
      int i = 0;
      for (int im = im0; im < im1; ++im)
      for (int part = 0; part < p.n_parts; ++part, ++i) {
        const int b = i & 1;
        mbar_wait(&full[b], (i >> 1) & 1);
        tcgen05_after_sync();
        if (elect_one()) {
        tl_stamp(p.debug, 3000 + 2 * i);
        // The issuing thread is ONE instruction stream: the loop is specialised on the number of accumulator tiles of this
        // CTA (a 16-way predicated unroll cost ~300 cycles per K = 16 step for the one or two MMAs it contained -- 5x the
        // tensor time, tools/mma_rate.cu) and the non-accumulating first step is peeled off.
        const WgradIssue w{xlo, xlo[0], nt > 1 ? xlo[1] : 0u, nt > 2 ? xlo[2] : 0u, xpl16, x_hi32, zh0, z_hi32, tmem, (uint32_t)N2, idesc2, idesc1, dbias, ones_lo, p.z_row_bytes, has_bias,
                           (uint32_t)b * (L.buf_bytes >> 4), p.pj[part]};
        int j = p.pj[part];
        const int jend = p.pj[part + 1];
        if (i == 0) {
          wgrad_issue_step<A_PLANES, false>(w, nt, j);
          ++j;
        }
        switch (nt) {
          case 1: for (; j < jend; ++j) wgrad_issue_tiles<A_PLANES, 1>(w, j); break;
          case 2: for (; j < jend; ++j) wgrad_issue_tiles<A_PLANES, 2>(w, j); break;
          case 3: for (; j < jend; ++j) wgrad_issue_tiles<A_PLANES, 3>(w, j); break;
          default: for (; j < jend; ++j) wgrad_issue_step<A_PLANES, true>(w, nt, j); break;
        }
        mma_commit(&empty[b]);
        tl_stamp(p.debug, 3001 + 2 * i);
        if (im == im1 - 1 && part == p.n_parts - 1) mma_commit(done);
        }
        __syncwarp();
      }
    }
  }
  // ===== epilogue: warps 2..9 (quadrant = warp % 4, 16-column chunks of parity (warp - 2) / 4) write the partial gradient =====
  if (warp >= 2) {
    const int q = warp & 3, r = q * 32 + lane, chalf = (warp - 2) >> 2;
    pdl_wait();
    mbar_wait(done, 0);
    tcgen05_after_sync();
    if (warp == 2 && lane == 0) tl_stamp(p.debug, 1200);
    float* part = p.part + ((int64_t)z * p.groups + gidx) * p.span;
    const int ntot = nt + (has_bias ? 1 : 0);
    for (int t = 0; t < ntot; ++t) {
      int64_t arow = -1;
      float sc = p.scale;
      if (t < nt) {
        const int tt = t_lo + t;
        const int grp = r >> 6, j = r & 63;
        const int r0 = grp ? p.row1[tt] : p.row0[tt];
        if (r0 >= 0 && j < p.grp_rows) arow = p.w_off + ((int64_t)r0 + (j / p.run) * p.run_stride + j % p.run) * N;
      } else if (r == 0) {
        arow = p.b_off, sc = 1.f;
      }
      const uint32_t taddr = tmem + ((uint32_t)(q * 32) << 16) + (uint32_t)t * N2;
      // this thread's 16-column chunks (one at N = 32, two at N = 64): every TMEM load of the tile is in flight before the
      // one wait (warp-uniform trip counts: the loads are .sync.aligned)
      float v[2][16], v2[2][16];
      const int c00 = chalf * 16, nc = c00 + 32 < N ? 2 : (c00 < N ? 1 : 0);
#pragma unroll
      for (int cc = 0; cc < 2; ++cc)
        if (cc < nc) {
          tmem_ld16_nowait(taddr + c00 + 32 * cc, v[cc]);
          tmem_ld16_nowait(taddr + N + c00 + 32 * cc, v2[cc]);
        }
      tmem_ld_wait();
      if (arow < 0) continue;
#pragma unroll
      for (int cc = 0; cc < 2; ++cc)
        if (cc < nc) {
#pragma unroll
          for (int k4 = 0; k4 < 4; ++k4)
            reinterpret_cast<float4*>(part + arow + c00 + 32 * cc)[k4] =
                make_float4((v[cc][4 * k4] + v2[cc][4 * k4]) * sc, (v[cc][4 * k4 + 1] + v2[cc][4 * k4 + 1]) * sc,
                            (v[cc][4 * k4 + 2] + v2[cc][4 * k4 + 2]) * sc, (v[cc][4 * k4 + 3] + v2[cc][4 * k4 + 3]) * sc);
        }
    }
  }
  if (warp == 2 && lane == 0) tl_stamp(p.debug, 1201);
  tcgen05_before_sync();
  __syncthreads();
  ktl_end(p.tl_id);
  if (warp == 1) tmem_dealloc(tmem, tmem_cols);
}

// ------------------------------------------------------------------------------------------------------
// staged batch (uint8 or fp32 NHWC) -> X2 planes of the first conv layer (space-to-depth, padded, pitched)
struct S2dArgs {
  const void* src[2];  // state, next_state
  // slots != nullptr: image im of source g lives at src[g] + slots[im] * src_stride (replay slots read in place) and
  // thread b < imgs of block 0 also gathers the scalars of sample b into the learner's staging
  const int64_t* slots;
  int64_t src_stride;
  const int32_t* g_action;
  const double* g_reward;
  const uint8_t* g_terminal;
  // ring != nullptr (with slots): frame store -- src is unused and value v * stack + p of image g of slot s is value v of
  // frame rows[(s * 2 + g) * stack + p] (id -1: zero), frame id f at ring + (f % n_frames) * frame_bytes
  const uint8_t* ring;
  const int64_t* rows;
  int64_t n_frames, frame_bytes;
  int stack;
  int32_t* o_action;
  float* o_reward;
  uint8_t* o_terminal;
  int u8, imgs, IH, IW, IC, s, ph, pw, BH, BW, P, C2;
  int n_src;           // 2: state and next_state (learning step); 1: state only (best_action)
  int64_t img_rows;    // allocated rows per image
  bf16 *hi, *lo;       // [2][imgs][img_rows][C2]
  int tl_id;
};
// kFrames: the frame-store source (a.ring); a separate instance, so the element paths compile exactly as without it
template <bool kFrames>
__global__ void __launch_bounds__(256) s2d_input_kernel(const S2dArgs a) {
  // one thread per (g, img, by, bx, ry): s*IC contiguous output channels = s input pixels of one input row
  pdl_trigger();
  pdl_wait();
  ktl_begin(a.tl_id);
  const int run = a.s * a.IC;
  const int64_t total = (int64_t)a.n_src * a.imgs * a.BH * a.BW * a.s;
  const int64_t img_elems = (int64_t)a.IH * a.IW * a.IC;
  if (a.slots && blockIdx.x == 0 && (int)threadIdx.x < a.imgs) {
    const int64_t slot = a.slots[threadIdx.x];
    a.o_action[threadIdx.x] = a.g_action[slot];
    a.o_reward[threadIdx.x] = __double2float_rn(a.g_reward[slot]);
    a.o_terminal[threadIdx.x] = a.g_terminal[slot];
  }
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    int64_t t = i;
    const int ry = (int)(t % a.s);
    t /= a.s;
    const int bx = (int)(t % a.BW);
    t /= a.BW;
    const int by = (int)(t % a.BH);
    t /= a.BH;
    const int im = (int)(t % a.imgs), g = (int)(t / a.imgs);
    const int iy = by * a.s + ry - a.ph;
    const int64_t o = (((int64_t)g * a.imgs + im) * a.img_rows + (int64_t)by * a.P + bx) * a.C2 + (int64_t)ry * run;
    if (a.u8 && a.IC == 4 && a.s == 4 && (a.pw & 1) == 0 && (a.IW & 1) == 0 && (!kFrames || a.stack == 4)) {
      // Atari frames: the run is 4 pixels x 4 stacked frames = 16 source bytes, 8-byte aligned pixel pairs
      const int ix0 = bx * 4 - a.pw;
      uint32_t w[4];  // w[q]: the 4 stacked frames of pixel ix0 + q, frame c in byte c
      if constexpr (kFrames) {
        // frame store: the same 16 bytes from the 4 frames, a 2-byte aligned pixel pair of each (ix0 is even, not a
        // multiple of 4), interleaved pixel-major
        const int64_t* row = a.rows + (a.slots[im] * 2 + g) * 4;
        const uint8_t* f[4];
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          const int64_t id = __ldg(row + c);
          f[c] = id < 0 ? nullptr : a.ring + frame_ring_slot(id, a.n_frames) * a.frame_bytes;
        }
#pragma unroll
        for (int hp = 0; hp < 2; ++hp) {
          const int ix = ix0 + 2 * hp;
          const bool ok = (unsigned)iy < (unsigned)a.IH && ix >= 0 && ix + 1 < a.IW;
          uint32_t p[4];
#pragma unroll
          for (int c = 0; c < 4; ++c)
            p[c] = ok && f[c] ? __ldg(reinterpret_cast<const unsigned short*>(f[c] + (int64_t)iy * a.IW + ix)) : 0u;
          const uint32_t p01 = p[0] | (p[1] << 16), p23 = p[2] | (p[3] << 16);
          w[2 * hp] = __byte_perm(p01, p23, 0x6420);      // first pixel of the pair, frames 0..3
          w[2 * hp + 1] = __byte_perm(p01, p23, 0x7531);  // second pixel
        }
      } else {
        const uint8_t* src = (const uint8_t*)(g ? a.src[1] : a.src[0]) + (a.slots ? a.slots[im] * a.src_stride : (int64_t)im * img_elems);
        uint2 raw[2];
#pragma unroll
        for (int hp = 0; hp < 2; ++hp) {
          const int ix = ix0 + 2 * hp;
          const bool ok = (unsigned)iy < (unsigned)a.IH && ix >= 0 && ix + 1 < a.IW;
          raw[hp] = ok ? __ldg(reinterpret_cast<const uint2*>(src + ((int64_t)iy * a.IW + ix) * 4)) : make_uint2(0, 0);
        }
        w[0] = raw[0].x, w[1] = raw[0].y, w[2] = raw[1].x, w[3] = raw[1].y;
      }
#pragma unroll
      for (int hv = 0; hv < 2; ++hv) {
        float x[8];
#pragma unroll
        for (int k = 0; k < 8; ++k) x[k] = (float)((w[2 * hv + (k >> 2)] >> (8 * (k & 3))) & 0xffu);
        *reinterpret_cast<uint4*>(a.hi + o + 8 * hv) = pack8_exact(x);
      }
      continue;
    }
    for (int e = 0; e < run; e += 8) {
      float x[8];
#pragma unroll
      for (int k = 0; k < 8; ++k) {
        const int ee = e + k, rx = ee / a.IC, c = ee - rx * a.IC;
        const int ix = bx * a.s + rx - a.pw;
        float v = 0.f;
        if ((unsigned)iy < (unsigned)a.IH && (unsigned)ix < (unsigned)a.IW) {
          const int64_t si = ((int64_t)iy * a.IW + ix) * a.IC + c;
          const void* src = g ? a.src[1] : a.src[0];
          if constexpr (kFrames) {
            const int64_t id = __ldg(a.rows + (a.slots[im] * 2 + g) * a.stack + si % a.stack);
            if (id >= 0) v = (float)__ldg(a.ring + frame_ring_slot(id, a.n_frames) * a.frame_bytes + si / a.stack);
          } else {
            if (a.slots) v = (float)__ldg((const uint8_t*)src + a.slots[im] * a.src_stride + si);  // replay slots hold uint8 frames here
            else v = a.u8 ? (float)__ldg((const uint8_t*)src + (int64_t)im * img_elems + si) : __ldg((const float*)src + (int64_t)im * img_elems + si);
          }
        }
        x[k] = v;
      }
      uint4 h, l;
      split8(x, h, l);
      *reinterpret_cast<uint4*>(a.hi + o + e) = h;
      if (!a.u8) *reinterpret_cast<uint4*>(a.lo + o + e) = l;
    }
  }
  ktl_end(a.tl_id);
}

// fp32 NHWC activation from the planes of its consumer layout (debug / parity: idqn_download_activation)
__global__ void __launch_bounds__(256) planes_to_f32_kernel(const PlaneDst d, int net, int imgs, int H, int W, int C,
                                                            float* __restrict__ out) {
  const int64_t total = (int64_t)imgs * H * W * C;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    int64_t t = i;
    const int c = (int)(t % C);
    t /= C;
    const int x = (int)(t % W);
    t /= W;
    const int y = (int)(t % H), im = (int)(t / H);
    const int64_t pi = plane_index(d, net, im, y, x) + c;
    out[i] = __bfloat162float(d.hi[pi]) + __bfloat162float(d.lo[pi]);
  }
}

}  // namespace img
