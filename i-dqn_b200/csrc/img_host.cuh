// Host side of the image-resident conv path (conv_img.cuh): geometry, buffers, TMA tensor maps, kernel arguments
// and launches.  Included by net.cu (uses its mark() / CK helpers).
#pragma once
#include "conv_img.cuh"
#include "dense_stream.cuh"
#include "dense_wgrad_tma.cuh"

struct ImgHost {
  img::Geom g[IDQN_IMG_LAYERS];
  img::TapsArgs fwd[IDQN_IMG_LAYERS], dg[IDQN_IMG_LAYERS];
  img::WgradArgs wg[IDQN_IMG_LAYERS];
  img::S2dArgs s2d;
  img::ChainArgs chain;   // conv1 -> conv2 forward in one kernel (conv_chain_fwd_kernel)
  int chain_on;
  // weight-streaming kernels of the big Dense layer (dense_stream.cuh)
  int dense_on;
  alignas(64) CUtensorMap fmapWf[2], fmapWd, dmapX[2], dmapDy[2];  // fp32 Dense_0 kernel: fwd boxes {128 o, 64 i} of the online / target arena, dgrad boxes {64 o, 128 i} (online)
  alignas(64) CUtensorMap wmapX[2], wmapP[3];  // dense_wgrad_tma.cuh: x planes {16 i, 32 b}; fp32 W / mu / nu {256 o, 8 i}
  int wgrad_tma_on;
  dense::Args dfwd, ddg;
  float* dpart;
  int* dtickets;
};

static int img_chunks(int rows, int* chunk_rows, int* rows_alloc) {
  const int n = (rows + 255) / 256;
  int cr = ((rows + n - 1) / n + 7) / 8 * 8;
  *chunk_rows = cr;
  *rows_alloc = cr * n;
  return n;
}

static bool img_geom(const Layer& l, int layer_index, img::Geom& g) {
  const ConvGeom& c = l.g;
  if (!l.is_conv || c.KH != c.KW || c.S < 1 || c.KH % c.S) return false;
  g.s = c.S, g.T = c.KH / c.S, g.ph = c.PH, g.pw = c.PW;
  g.IC = c.IC, g.OC = c.OC, g.C2 = c.S * c.S * c.IC;
  if (g.C2 != 64 && g.C2 != 128) return false;
  if (g.OC != 32 && g.OC != 64) return false;
  if (layer_index > 0 && (g.OC != 64 || g.IC % 32)) return false;  // dgrad: 128-byte dy rows, 32-channel epilogue chunks
  const int run = c.S * c.IC;
  if (run > 64 || 64 % run) return false;
  if (g.T * g.T > img::MAX_TAPS) return false;
  g.halves = g.C2 / 64;
  g.IH = c.IH, g.IW = c.IW, g.OH = c.OH, g.OW = c.OW;
  g.BH = c.OH + g.T - 1, g.BW = c.OW + g.T - 1, g.P = c.OW + 2 * (g.T - 1);
  if ((c.IH - 1 + c.PH) / c.S >= g.BH || (c.IW - 1 + c.PW) / c.S >= g.BW) return false;
  g.XR = g.BH * g.P;
  g.x_chunks = img_chunks(g.XR, &g.x_chunk_rows, &g.XRa);
  g.ZH = c.OH + 2 * (g.T - 1), g.ZR = g.ZH * g.P;
  g.z_chunks = img_chunks(g.ZR, &g.z_chunk_rows, &g.ZRa);
  g.Kd = c.Kd;
  return true;
}

static const size_t IMG_SMEM_MAX = 227 * 1024;
static const size_t IMG_SMEM_OPTIN = 226 * 1024;  // dynamic limit requested per kernel: the device maximum minus room for the kernels' few static __shared__ words
// images per partial-sum group of the conv weight gradients.  3 -> 11 groups at batch 32: with the two tile splits the
// accumulators need, K = 5 heads give 110 CTAs = one wave (2 -> 160 CTAs = two waves measured +14 us per K = 5 step)
static const int IMG_WGRAD_IPG = 3;

// decide whether the handle can run the image path and build everything it needs
static int img_setup(idqn_handle* h) {
  h->img_on = 0;
  const idqn_config& c = h->cfg;
  if (c.arch != IDQN_ARCH_CNN || (c.flags & (IDQN_F_SIMT_ONLY | IDQN_F_NO_IMG))) return IDQN_OK;
  if (h->n_layers < IDQN_IMG_LAYERS + 2 || !tma::encode_fn()) return IDQN_OK;
  ImgHost* H = new ImgHost();
  memset(H, 0, sizeof(*H));
  for (int li = 0; li < IDQN_IMG_LAYERS; ++li)
    if (!img_geom(h->layers[li], li, H->g[li])) {
      delete H;
      return IDQN_OK;
    }
  for (int li = 1; li < IDQN_IMG_LAYERS; ++li)
    if (H->g[li].IC != H->g[li - 1].OC) {
      delete H;
      return IDQN_OK;
    }
  const Layer& dense = h->layers[IDQN_IMG_LAYERS];
  if (dense.is_conv || !tc_dense_ok(h, dense)) {
    delete H;
    return IDQN_OK;
  }
  const int K = h->K, B = h->B;
  h->img_host = H;
  // ---- buffers (zero-initialised once: padding positions are never written afterwards) ----
  for (int li = 0; li < IDQN_IMG_LAYERS; ++li) {
    const img::Geom& g = H->g[li];
    ImgLayerState& S = h->il[li];
    const int xnets = li == 0 ? 2 : 2 * K;
    S.x2_net_stride = (int64_t)B * g.XRa * g.C2;
    S.dz_net_stride = (int64_t)B * g.ZRa * g.OC;
    const size_t xb = sizeof(__nv_bfloat16) * S.x2_net_stride * xnets, zb = sizeof(__nv_bfloat16) * S.dz_net_stride * K;
    CK(cudaMalloc(&S.x2_hi, xb));
    CK(cudaMalloc(&S.x2_lo, xb));
    CK(cudaMalloc(&S.dz_hi, zb));
    CK(cudaMalloc(&S.dz_lo, zb));
    CK(cudaMemsetAsync(S.x2_hi, 0, xb, h->stream));
    CK(cudaMemsetAsync(S.x2_lo, 0, xb, h->stream));
    CK(cudaMemsetAsync(S.dz_hi, 0, zb, h->stream));
    CK(cudaMemsetAsync(S.dz_lo, 0, zb, h->stream));
    // ---- tensor maps ----
    for (int pl = 0; pl < 2; ++pl) {
      {  // X2: {64 channels, halves, rows}
        const uint64_t dims[3] = {64, (uint64_t)g.halves, (uint64_t)xnets * B * g.XRa};
        const uint64_t str[2] = {128, (uint64_t)g.C2 * 2};
        const uint32_t box[3] = {64, 1, (uint32_t)g.x_chunk_rows};
        REQUIRE(tma::encode_bf16(&S.mapX[pl], pl ? S.x2_lo : S.x2_hi, 3, dims, str, box, 128), "tensor map X2 L%d", li);
      }
      {  // W: flax kernel [KH][KW*IC][OC] of every net: {OC, KW*IC, KH, 2K}
        const ConvGeom& cg = h->layers[li].g;
        const uint64_t dims[4] = {(uint64_t)g.OC, (uint64_t)cg.KW * g.IC, (uint64_t)cg.KH, (uint64_t)2 * K};
        const uint64_t str[3] = {(uint64_t)g.OC * 2, (uint64_t)cg.KW * g.IC * g.OC * 2, (uint64_t)h->stride * 2};
        const uint32_t box[4] = {(uint32_t)g.OC, (uint32_t)(g.s * g.IC), (uint32_t)g.s, 1};
        const __nv_bfloat16* wb = (pl ? h->wpl_lo : h->wpl_hi) + h->layers[li].w_off;
        REQUIRE(tma::encode_bf16(&S.mapW[pl], wb, 4, dims, str, box, g.OC * 2), "tensor map W L%d", li);
      }
      {  // dyZ: {OC, 1, rows}
        const uint64_t dims[3] = {(uint64_t)g.OC, 1, (uint64_t)K * B * g.ZRa};
        const uint64_t str[2] = {(uint64_t)g.OC * 2, (uint64_t)g.OC * 2};
        const uint32_t box[3] = {(uint32_t)g.OC, 1, (uint32_t)g.z_chunk_rows};
        REQUIRE(tma::encode_bf16(&S.mapZ[pl], pl ? S.dz_lo : S.dz_hi, 3, dims, str, box, g.OC * 2), "tensor map dyZ L%d", li);
      }
    }
  }
  // ---- partial weight gradients ----
  h->wspan = dense.w_off;  // the conv layers occupy the arena range [0, Dense_0.w_off)
  {
    // Partial sums over FIXED groups of IMG_WGRAD_IPG consecutive images (fp32 accumulation in TMEM inside a group,
    // groups summed in index order by adam_kernel): the grouping -- hence every rounding of the conv weight gradients --
    // depends on the batch size only, not on how many heads this handle owns, so a head computes bit-identical
    // gradients whether it lives in a K-head handle or alone on its own GPU (parallel.py).  What adapts to K is the
    // split of a layer's M tiles over CTAs (tsplit), which does not touch the summation order.
    const int ipg = std::min(IMG_WGRAD_IPG, B);
    h->wgroups = (B + ipg - 1) / ipg;
    const size_t pb = sizeof(float) * h->wspan * h->wgroups * K;
    CK(cudaMalloc(&h->wpart, pb));
    CK(cudaMemsetAsync(h->wpart, 0, pb, h->stream));
  }
  // ---- kernel arguments ----
  for (int li = 0; li < IDQN_IMG_LAYERS; ++li) {
    const img::Geom& g = H->g[li];
    const Layer& l = h->layers[li];
    const ConvGeom& cg = l.g;
    // forward
    {
      img::TapsArgs& a = H->fwd[li];
      a.imgs = B;
      if (li == 0) {
        a.nets_per_g = K;
        a.hpg = std::min(K, std::max(1, 96 / g.OC));
        a.n_hg = (K + a.hpg - 1) / a.hpg;
        a.n_units = 2 * B * a.n_hg;
      } else {
        a.nets_per_g = 1, a.hpg = 1, a.n_hg = 1, a.n_units = 2 * K * B;
      }
      a.a_rows_alloc = g.XRa, a.a_chunks = g.x_chunks, a.a_chunk_rows = g.x_chunk_rows, a.a_halves = g.halves;
      a.a_buf_rows = g.XRa;
      a.P = g.P, a.M_valid = g.OH * g.P, a.W_valid = g.OW;
      a.tiles = (a.M_valid + 127) / 128;
      a.N = a.hpg * g.OC;
      a.tpp = std::max(1, std::min(a.tiles, 128 / a.N));  // 2 buffers x tpp tiles x 2N columns <= 512
      // two-tile passes (conv_taps_kernel): two accumulator buffers x two tiles x 2N columns must fit the 512 TMEM columns
      a.pair = a.tiles == 2 && 8 * a.N <= 512 && !getenv("IDQN_NO_PAIR");
      a.n_taps = g.T * g.T, a.kt = g.C2 / 16;
      for (int ty = 0; ty < g.T; ++ty)
        for (int tx = 0; tx < g.T; ++tx) {
          const int t = ty * g.T + tx;
          a.a_shift[t] = ty * g.P + tx;
          a.w_c1[t] = g.s * tx * g.IC, a.w_c2[t] = g.s * ty;
        }
      a.b_box_bytes = (uint32_t)g.C2 * g.OC * 2, a.b_row_bytes = (uint32_t)g.OC * 2;
      a.OH = g.OH, a.OW = g.OW, a.OC = g.OC;
      a.scale = li == 0 ? 1.0f / 255.0f : 1.0f;  // architectures/dqn.py:44
      a.w = NetPtr{h->online, h->target, h->stride, h->stride, K};
      a.b_off = l.b_off;
      a.out = nullptr, a.out_net_stride = h->act_stride, a.mask_hi = nullptr;  // fp32 copy: idqn_download_activation rebuilds it
      if (li + 1 < IDQN_IMG_LAYERS) {
        const img::Geom& n = H->g[li + 1];
        a.dst = img::PlaneDst{h->il[li + 1].x2_hi, h->il[li + 1].x2_lo, h->il[li + 1].x2_net_stride, n.XRa,
                              n.s, n.ph, n.pw, n.P, g.OC, n.C2};
      } else {
        a.dst = img::PlaneDst{h->act_hi + l.act_off, h->act_lo + l.act_off, h->act_stride, (int64_t)g.OH * g.OW,
                              1, 0, 0, g.OW, g.OC, g.OC};
      }
      // taps per ring slot (one ty row if two such slots fit next to the two image buffers), then the ring depth
      const uint32_t abuf2 = 2u * (li == 0 ? 1 : 2) * a.a_halves * a.a_buf_rows * 128;  // layer 0: uint8 frames, hi plane only
      a.tap_group = g.T;
      if (2 * img::round_up(2 * a.hpg * a.b_box_bytes * a.tap_group, 1024) + abuf2 + 2048 > IMG_SMEM_MAX) a.tap_group = 1;
      const uint32_t slot = img::round_up(2 * a.hpg * a.b_box_bytes * a.tap_group, 1024);
      a.ring = (int)std::min<size_t>(a.tap_group > 1 ? 2 : 4, (IMG_SMEM_MAX - 2048 - abuf2) / slot);
      a.n_units_total = a.n_units;
      {  // resident weights: one slot per tap group if they all fit next to the two image buffers (conv0: 2 x 48 KB + 128 KB).
         // Opt-in (IDQN_RESIDENT=1): measured 0.3014 vs 0.3016 ms per K = 5 step -- conv0 is bound by its epilogue (1.7 us per
         // job against 0.9 us of MMAs), not by the weight loads
        const int ng = (a.n_taps + a.tap_group - 1) / a.tap_group;
        if (ng <= 8 && (size_t)ng * slot + abuf2 + 2048 <= IMG_SMEM_MAX && getenv("IDQN_RESIDENT")) {
          a.resident = 1, a.ring = ng;
          a.hg_major = 1;  // consecutive units of a CTA share their head group, hence their weights
        }
      }
      const int over = a.tiles * 128 + a.a_shift[a.n_taps - 1] - a.a_buf_rows;
      if (a.ring < 2 || over * 128 > (int)(a.ring * slot)) {
        idqn_set_error("internal: image path does not fit shared memory (fwd L%d)", li);
        return IDQN_EINVAL;
      }
    }
    // data gradient (layers >= 1)
    if (li > 0) {
      img::TapsArgs& a = H->dg[li];
      const Layer& prev = h->layers[li - 1];
      const img::Geom& pg = H->g[li - 1];
      a.imgs = B, a.nets_per_g = 1, a.hpg = 1, a.n_hg = 1, a.n_units = K * B;
      a.a_rows_alloc = g.ZRa, a.a_chunks = g.z_chunks, a.a_chunk_rows = g.z_chunk_rows, a.a_halves = 1;
      a.a_buf_rows = g.ZRa;
      a.P = g.P, a.M_valid = g.BH * g.P, a.W_valid = g.BW;
      a.tiles = (a.M_valid + 127) / 128;
      a.N = g.C2;  // <= 128 (img_geom): the epilogue prefetches the relu' masks of at most two 32-column chunks per thread
      a.tpp = std::max(1, std::min(a.tiles, 128 / a.N));
      a.n_taps = g.T * g.T, a.kt = g.OC / 16;
      a.pair = a.tiles == 2 && 8 * a.N <= 512 && !getenv("IDQN_NO_PAIR");  // conv2: N = 64
      int shmax = 0;
      for (int ty = 0; ty < g.T; ++ty)
        for (int tx = 0; tx < g.T; ++tx) {
          const int t = ty * g.T + tx;
          a.a_shift[t] = (g.T - 1 - ty) * g.P + (g.T - 1 - tx);
          shmax = std::max(shmax, a.a_shift[t]);
          a.w_c1[t] = g.s * tx * g.IC, a.w_c2[t] = g.s * ty;
        }
      a.b_box_bytes = (uint32_t)g.C2 * g.OC * 2, a.b_row_bytes = (uint32_t)g.OC * 2;
      a.OC = g.IC, a.s = g.s, a.ph = g.ph, a.pw = g.pw, a.IH = g.IH, a.IW = g.IW;
      a.OH = g.OH, a.OW = g.OW;
      a.scale = 1.f;
      a.out = nullptr, a.out_net_stride = h->act_stride;  // the fp32 gradient is not needed: dyZ planes carry it
      a.mask_hi = h->il[li].x2_hi, a.mask_net_stride = h->il[li].x2_net_stride, a.mask_img_rows = g.XRa;
      (void)prev;
      a.dst = img::PlaneDst{h->il[li - 1].dz_hi, h->il[li - 1].dz_lo, h->il[li - 1].dz_net_stride, pg.ZRa,
                            1, pg.T - 1, pg.T - 1, pg.P, pg.OC, pg.OC};
      const uint32_t abuf2 = 2u * 2 * a.a_buf_rows * 128;
      a.tap_group = g.T;
      if (2 * img::round_up(2 * a.b_box_bytes * a.tap_group, 1024) + abuf2 + 2048 > IMG_SMEM_MAX) a.tap_group = 1;
      const uint32_t slot = img::round_up(2 * a.b_box_bytes * a.tap_group, 1024);
      a.ring = (int)std::min<size_t>(a.tap_group > 1 ? 2 : 4, (IMG_SMEM_MAX - 2048 - abuf2) / slot);
      a.n_units_total = a.n_units;
      {  // resident weights (conv1 data gradient: 2 x 64 KB of weights + 88 KB of dyZ images)
        const int ng = (a.n_taps + a.tap_group - 1) / a.tap_group;
        if (ng <= 8 && (size_t)ng * slot + abuf2 + 2048 <= IMG_SMEM_MAX && getenv("IDQN_RESIDENT")) a.resident = 1, a.ring = ng;
      }
      const int over = a.tiles * 128 + shmax - a.a_buf_rows;
      if (a.ring < 2 || over * 128 > (int)(a.ring * slot)) {
        idqn_set_error("internal: image path does not fit shared memory (dgrad L%d)", li);
        return IDQN_EINVAL;
      }
    }
    // weight gradient
    {
      img::WgradArgs& a = H->wg[li];
      a.heads = K, a.imgs = B;
      a.x_shared = li == 0;
      a.ipg = (B + h->wgroups - 1) / h->wgroups;
      a.groups = h->wgroups;
      a.k16 = (g.OH * g.P + 15) / 16;
      a.z_start = (g.T - 1) * (g.P + 1);
      const int shmax = (g.T - 1) * g.P + (g.T - 1);
      a.x_rows_alloc = g.XRa, a.x_halves = g.halves;
      a.z_rows_alloc = g.ZRa;
      a.z_row_bytes = (uint32_t)g.OC * 2;
      {
        // parts: the K = 16 steps of an image in two halves, each with its own box of X2 rows (+ the tap-shift halo) and
        // of dyZ rows, double-buffered in shared memory
        a.n_parts = a.k16 >= 4 ? 2 : 1;
        const int smax = (a.k16 + a.n_parts - 1) / a.n_parts;
        a.pj[0] = 0, a.pj[1] = a.n_parts == 2 ? smax : a.k16, a.pj[2] = a.k16, a.pj[3] = a.k16;
        const int xrows = 16 * smax + shmax, zrows = 16 * smax;
        a.x_chunks = (xrows + 255) / 256, a.x_chunk_rows = ((xrows + a.x_chunks - 1) / a.x_chunks + 7) / 8 * 8;
        a.x_buf_rows = a.x_chunks * a.x_chunk_rows;
        a.z_chunks = (zrows + 255) / 256, a.z_chunk_rows = ((zrows + a.z_chunks - 1) / a.z_chunks + 7) / 8 * 8;
        a.z_buf_rows = a.z_chunks * a.z_chunk_rows;
        ImgLayerState& S = h->il[li];
        const int xnets = li == 0 ? 2 : 2 * K;
        for (int pl = 0; pl < 2; ++pl) {
          const uint64_t xdims[3] = {64, (uint64_t)g.halves, (uint64_t)xnets * B * g.XRa};
          const uint64_t xstr[2] = {128, (uint64_t)g.C2 * 2};
          const uint32_t xbox[3] = {64, 1, (uint32_t)a.x_chunk_rows};
          REQUIRE(tma::encode_bf16(&S.mapXw[pl], pl ? S.x2_lo : S.x2_hi, 3, xdims, xstr, xbox, 128), "tensor map X2 (wgrad parts) L%d", li);
          const uint64_t zdims[3] = {(uint64_t)g.OC, 1, (uint64_t)K * B * g.ZRa};
          const uint64_t zstr[2] = {(uint64_t)g.OC * 2, (uint64_t)g.OC * 2};
          const uint32_t zbox[3] = {(uint32_t)g.OC, 1, (uint32_t)a.z_chunk_rows};
          REQUIRE(tma::encode_bf16(&S.mapZw[pl], pl ? S.dz_lo : S.dz_hi, 3, zdims, zstr, zbox, g.OC * 2), "tensor map dyZ (wgrad parts) L%d", li);
        }
        REQUIRE(img::wgrad_smem(a, li == 0 ? 1 : 2).total <= IMG_SMEM_OPTIN, "internal: wgrad L%d does not fit shared memory", li);
      }
      // 64-row groups: (tap, c2 / 64), paired into 128-row tiles
      const int run = g.s * g.IC, ry_per_grp = 64 / run;
      int ng = 0, gsh[2 * img::MAX_TAPS], ghf[2 * img::MAX_TAPS], grow[2 * img::MAX_TAPS];
      for (int ty = 0; ty < g.T; ++ty)
        for (int tx = 0; tx < g.T; ++tx)
          for (int gq = 0; gq < g.halves; ++gq) {
            gsh[ng] = ty * g.P + tx, ghf[ng] = gq;
            grow[ng] = ((g.s * ty + gq * ry_per_grp) * cg.KW + g.s * tx) * g.IC;
            ++ng;
          }
      a.n_tiles = (ng + 1) / 2;
      // tile split: the smallest one whose accumulators (+ the bias tile) fit the 512 TMEM columns, raised while the
      // grid still fits the machine in one wave
      const int conv_sms = h->partition ? ((smpart::Partition*)h->partition)->sms[0] : h->sm_count;
      a.tsplit = 0;
      for (int ts = 1; ts <= a.n_tiles; ++ts) {
        const int tps = (a.n_tiles + ts - 1) / ts;
        if ((ts - 1) * tps >= a.n_tiles || (tps + 1) * 2 * g.OC > 512) continue;  // empty last split / TMEM
        if (!a.tsplit || K * h->wgroups * ts <= conv_sms) a.tsplit = ts;
      }
      if (a.n_tiles > img::MAX_TAPS || !a.tsplit) {
        idqn_set_error("internal: wgrad L%d needs too many accumulator tiles", li);
        return IDQN_EINVAL;
      }
      a.tps = (a.n_tiles + a.tsplit - 1) / a.tsplit;
      for (int t = 0; t < a.n_tiles; ++t) {
        const int g0 = 2 * t, g1 = 2 * t + 1 < ng ? 2 * t + 1 : -1;
        a.sh0[t] = gsh[g0], a.hf0[t] = ghf[g0], a.row0[t] = grow[g0];
        a.sh1[t] = g1 >= 0 ? gsh[g1] : gsh[g0], a.hf1[t] = g1 >= 0 ? ghf[g1] : ghf[g0], a.row1[t] = g1 >= 0 ? grow[g1] : -1;
      }
      a.grp_rows = 64, a.run = run, a.run_stride = cg.KW * g.IC;
      a.N = g.OC;
      a.scale = li == 0 ? 1.0f / 255.0f : 1.0f;
      a.part = h->wpart, a.span = h->wspan, a.w_off = l.w_off, a.b_off = l.b_off;
    }
  }
  // ---- conv1 -> conv2 forward chain (conv_chain_fwd_kernel): both layers two-tile, 64 output channels, 128-byte weight rows ----
  {
    const img::TapsArgs &a = H->fwd[1], &b = H->fwd[2];
    img::ChainArgs& c = H->chain;
    c.a = a, c.b = b;
    const img::Geom& n = H->g[2];
    c.bP = n.P, c.b_off_y = n.ph, c.b_off_x = n.pw;
    c.b_tap_group = std::max(1, (int)((2 * a.b_box_bytes) / (2 * b.b_box_bytes)));  // as many conv2 taps as fill a conv1 slot
    c.ring = 2;
    const img::ChainSmem L = img::chain_smem(c);
    H->chain_on = IDQN_IMG_LAYERS == 3 && a.tiles == 2 && b.tiles == 2 && a.N == 64 && b.N == 64 && a.hpg == 1 && b.hpg == 1 &&
                  a.n_units == b.n_units && n.s == 1 && b.a_halves == 1 && a.kt % 4 == 0 && b.kt % 4 == 0 &&
                  (a.n_taps + (b.n_taps + c.b_tap_group - 1) / c.b_tap_group) >= c.ring && L.total <= IMG_SMEM_OPTIN &&
                  // an M tile may read rows past its image: they must stay inside the allocation
                  (uint32_t)(256 + b.a_shift[b.n_taps - 1]) * 128 <= L.b_bytes + c.ring * L.slot_bytes;
  }
  // ---- input space-to-depth ----
  {
    const img::Geom& g = H->g[0];
    img::S2dArgs& a = H->s2d;
    a.src[0] = h->s, a.src[1] = h->s2;
    a.imgs = B, a.IH = g.IH, a.IW = g.IW, a.IC = g.IC, a.s = g.s, a.ph = g.ph, a.pw = g.pw;
    a.BH = g.BH, a.BW = g.BW, a.P = g.P, a.C2 = g.C2, a.img_rows = g.XRa;
    a.hi = h->il[0].x2_hi, a.lo = h->il[0].x2_lo;
    a.n_src = 2;
  }
  // ---- big Dense layer: weight-streaming kernels ----
  {
    const int li = IDQN_IMG_LAYERS;
    const Layer& prev = h->layers[li - 1];
    const int I = dense.g.Kd, O = dense.g.OC;
    H->dense_on = B == dense::NB && O % 128 == 0 && I % 64 == 0 && O % 64 == 0;
    if (H->dense_on) {
      {
        // the fp32 master kernel of every head: {O, I, K}; the streaming kernels split it into bf16 hi/lo in shared memory
        const uint64_t wdims[3] = {(uint64_t)O, (uint64_t)I, (uint64_t)K};
        const uint64_t wstr[2] = {(uint64_t)O * 4, (uint64_t)h->stride * 4};
        const uint32_t boxf[3] = {128, 64, 1}, boxd[3] = {64, 128, 1};
        REQUIRE(tma::encode_f32(&H->fmapWf[0], h->online + dense.w_off, 3, wdims, wstr, boxf), "tensor map dense W (fwd, online)");
        REQUIRE(tma::encode_f32(&H->fmapWf[1], h->target + dense.w_off, 3, wdims, wstr, boxf), "tensor map dense W (fwd, target)");
        REQUIRE(tma::encode_f32(&H->fmapWd, h->online + dense.w_off, 3, wdims, wstr, boxd), "tensor map dense W (dgrad)");
      }
      for (int pl = 0; pl < 2; ++pl) {
        const __nv_bfloat16* xb = (pl ? h->act_lo : h->act_hi) + prev.act_off;
        const uint64_t xdims[3] = {(uint64_t)I, (uint64_t)B, (uint64_t)2 * K};
        const uint64_t xstr[2] = {(uint64_t)I * 2, (uint64_t)h->act_stride * 2};
        const uint32_t boxx[3] = {64, (uint32_t)B, 1};
        REQUIRE(tma::encode_bf16(&H->dmapX[pl], xb, 3, xdims, xstr, boxx, 128), "tensor map dense x");
        const __nv_bfloat16* yb = (pl ? h->dact_lo : h->dact_hi) + dense.act_off;
        const uint64_t ydims[3] = {(uint64_t)O, (uint64_t)B, (uint64_t)K};
        const uint64_t ystr[2] = {(uint64_t)O * 2, (uint64_t)h->act_stride * 2};
        REQUIRE(tma::encode_bf16(&H->dmapDy[pl], yb, 3, ydims, ystr, boxx, 128), "tensor map dense dy");
      }
      // fused wgrad + Adam pipeline (dense_wgrad_tma.cuh)
      H->wgrad_tma_on = O == dwt::CB * dwt::TO && I % dwt::TM == 0 && dense.b_off == dense.w_off + (int64_t)I * O;
      if (H->wgrad_tma_on) {
        for (int pl = 0; pl < 2; ++pl) {
          // x planes as the N-side operand: boxes {16 i, 32 b} (32-byte rows, SWIZZLE_32B); dy^T goes to TMEM from global
          const __nv_bfloat16* xb = (pl ? h->act_lo : h->act_hi) + prev.act_off;
          const uint64_t xdims[3] = {(uint64_t)I, (uint64_t)B, (uint64_t)2 * K};
          const uint64_t xstr[2] = {(uint64_t)I * 2, (uint64_t)h->act_stride * 2};
          const uint32_t xbox[3] = {(uint32_t)dwt::TN, (uint32_t)B, 1};
          REQUIRE(tma::encode_bf16(&H->wmapX[pl], xb, 3, xdims, xstr, xbox, 32), "tensor map dense x (wgrad)");
        }
        float* arenas[3] = {h->online, h->mu, h->nu};
        for (int a = 0; a < 3; ++a) {
          const uint64_t pdims[3] = {(uint64_t)O, (uint64_t)I, (uint64_t)K};
          const uint64_t pstr[2] = {(uint64_t)O * 4, (uint64_t)h->stride * 4};
          const uint32_t pbox[3] = {256, (uint32_t)dwt::TM, 1};
          REQUIRE(tma::encode_f32(&H->wmapP[a], arenas[a] + dense.w_off, 3, pdims, pstr, pbox), "tensor map dense W/mu/nu");
        }
      }
      const int kblocks = (I + 63) / 64;
      {
        dense::Args& a = H->dfwd;
        a.nets = 2 * K, a.tiles = O / 128;
        // split K: the largest divisor of the K-block count (<= 16 splits, >= 4 blocks each; 7744 / 64 = 121 -> 11 x 11).
        // A function of the layer shape only -- not of the number of nets -- so that the summation grouping of the
        // forward pass, like every other reduction of the step, does not depend on how many heads the handle owns.
        int best = 1;
        for (int sp = 1; sp <= 16; ++sp)
          if (kblocks % sp == 0 && kblocks / sp >= 4) best = sp;
        a.splits = best, a.kb_per_unit = (kblocks + best - 1) / best;
        a.n_units = a.nets * a.tiles * a.splits;
        a.stages = 4, a.heads = K;
        a.I = I, a.O = O;
        a.w = NetPtr{h->online, h->target, h->stride, h->stride, K};
        a.b_off = dense.b_off;
        a.y = h->act + dense.act_off, a.yh = h->act_hi + dense.act_off, a.yl = h->act_lo + dense.act_off;
        a.ystride = h->act_stride;
        CK(cudaMalloc(&H->dpart, sizeof(float) * (size_t)a.n_units * dense::NB * 128));
        CK(cudaMalloc(&H->dtickets, sizeof(int) * a.nets * a.tiles));
        CK(cudaMemsetAsync(H->dtickets, 0, sizeof(int) * a.nets * a.tiles, h->stream));
        a.part = H->dpart, a.tickets = H->dtickets;
      }
      {
        dense::Args& a = H->ddg;
        a.nets = K, a.tiles = (I + 127) / 128, a.splits = 1, a.kb_per_unit = O / 64;
        a.n_units = a.nets * a.tiles;
        a.stages = 4, a.heads = K;
        a.I = I, a.O = O;
        a.y = h->dact + prev.act_off, a.xact = nullptr, a.xmask_hi = h->act_hi + prev.act_off, a.ystride = h->act_stride;
        a.yh = h->dact_hi + prev.act_off, a.yl = h->dact_lo + prev.act_off;
        a.zP = 0;
      }
    }
  }
  h->img_on = 1;
  // Dense_0 lives in HBM as fp32 only (no bf16 planes are maintained for it) when both its streaming kernels and the
  // TMA wgrad+Adam pipeline serve it; the generic kernels rebuild the planes they need on demand (ensure_dense0_planes)
  h->fast_dense = H->dense_on && H->wgrad_tma_on && !(c.flags & (IDQN_F_OLD_WGRAD | IDQN_F_SIMT_ONLY));
  h->d0_lo = dense.w_off, h->d0_hi = dense.b_off;
  return IDQN_OK;
}

static void img_free(idqn_handle* h) {
  for (int li = 0; li < IDQN_IMG_LAYERS; ++li) {
    void* ptrs[] = {h->il[li].x2_hi, h->il[li].x2_lo, h->il[li].dz_hi, h->il[li].dz_lo};
    for (void* p : ptrs)
      if (p) cudaFree(p);
  }
  if (h->wpart) cudaFree(h->wpart);
  if (h->img_host) {
    ImgHost* H = (ImgHost*)h->img_host;
    if (H->dpart) cudaFree(H->dpart);
    if (H->dtickets) cudaFree(H->dtickets);
    delete H;
  }
}

// IDQN_TL=fwd2 / dgrad1 / wgrad0 ...: the matching launch records its pipeline timeline (conv_img.cuh)
static int img_debug_on(const char* kind, int li) {
  const char* e = getenv("IDQN_TL");
  if (!e) return 0;
  char tag[32];
  snprintf(tag, sizeof(tag), "%s%d", kind, li);
  if (strcmp(e, tag)) return 0;
  static unsigned long long zeros[img::TL_MAX];
  cudaMemcpyToSymbol(img::g_tl, zeros, sizeof(zeros));
  return 1;
}
extern "C" int idqn_debug_timeline(unsigned long long* out, int max_entries) {
  cudaDeviceSynchronize();
  const int n = std::min((int)img::TL_MAX, max_entries);
  cudaMemcpyFromSymbol(out, img::g_tl, sizeof(unsigned long long) * n);
  return n;
}

// L2 eviction priorities of the Dense_0 streams: the weight planes of the first `keep` online heads are loaded / stored
// evict_last, every other plane (target heads) and the fp32 W / mu / nu streams evict_first.  Measured (K = 5): the data
// gradient, which re-reads the online planes ~20 us after the forward, drops from 28.7 to 22.6 us with keep = 2; the
// planes do NOT survive from the wgrad+Adam of one step to the forward of the next (250 us, ~250 MB of other traffic),
// and a persisting-L2 set-aside (cudaLimitPersistingL2CacheSize) makes the streaming kernels 35-100% slower.
static int l2_keep_heads(const idqn_handle* h) {
  static const int env = getenv("IDQN_L2_KEEP_HEADS") ? atoi(getenv("IDQN_L2_KEEP_HEADS")) : 2;
  return std::min(env, h->K);
}

// The dynamic shared-memory limit of a kernel is raised ONCE to the device maximum and never lowered: the same
// instantiation is launched with different sizes (conv layers 1 and 2), and a profiler that re-launches the kernel nodes
// of the captured graph one by one (ncu) launches them under the function's CURRENT attribute -- lowering it for the
// second layer made the first layer's node fail with LaunchFailed under ncu (round-1 GPUTEST: ncu_rc=9).
template <class Kern>
static cudaError_t img_set_smem(Kern kern, size_t bytes) {
  if (bytes > IMG_SMEM_OPTIN) return cudaErrorInvalidValue;
  return cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)IMG_SMEM_OPTIN);
}

// act_imgs > 0: only the first act_imgs images of `state` (acting); otherwise the whole batch of state and next_state
static int img_launch_s2d(idqn_handle* h, int x_u8, int act_imgs = 0) {
  ImgHost* H = (ImgHost*)h->img_host;
  img::S2dArgs a = H->s2d;
  a.u8 = x_u8;
  const bool single_state = act_imgs > 0;
  a.tl_id = single_state ? -1 : tl_next(h);
  if (single_state) a.imgs = act_imgs, a.n_src = 1;
  a.src[0] = h->s, a.src[1] = h->s2;  // the staging set of this step (idqn_submit_batch_host points it at its slot)
  a.slots = nullptr, a.ring = nullptr;
  if (h->rsrc_on) {  // idqn_learn_from_replay: frames read from the replay slots in place, scalars gathered here
    a.src[0] = h->rsrc.state, a.src[1] = h->rsrc.next_state;
    a.slots = h->rsrc.slots, a.src_stride = h->rsrc.state_bytes;
    a.ring = h->rsrc.ring, a.rows = h->rsrc.rows, a.n_frames = h->rsrc.n_frames, a.frame_bytes = h->rsrc.frame_bytes;
    a.stack = h->rsrc.stack;
    a.g_action = h->rsrc.action, a.g_reward = h->rsrc.reward, a.g_terminal = h->rsrc.terminal;
    a.o_action = h->action, a.o_reward = h->reward, a.o_terminal = h->terminal;
  }
  const int64_t total = (int64_t)a.n_src * a.imgs * a.BH * a.BW * a.s;
  // first kernel of the step: launched WITHOUT the programmatic attribute, so everything enqueued before the step (the
  // previous step's Adam kernels when the step is not graph-replayed) has completed before any kernel of this step --
  // several of which prefetch weight tiles ahead of their griddepcontrol.wait -- can start
  const dim3 grid((unsigned)((total + 255) / 256));
  if (a.ring) CK(launch_pdl(false, img::s2d_input_kernel<true>, grid, dim3(256), 0, h->stream, a));
  else CK(launch_pdl(false, img::s2d_input_kernel<false>, grid, dim3(256), 0, h->stream, a));
  mark(h, "s2d_input_L%d", 0);
  return IDQN_OK;
}

// unit0 / n_units >= 0: run only that window of the layer's units (best_action: one (net, image) of the training layout)
static int img_launch_taps(idqn_handle* h, int li, bool dgrad, int a_planes, int unit0 = -1, int n_units = -1) {
  ImgHost* H = (ImgHost*)h->img_host;
  img::TapsArgs a = dgrad ? H->dg[li] : H->fwd[li];
  if (unit0 >= 0) {
    // a window of the layer's units in the (input, image)-major order (best_action: one image): per-pass weight loads
    a.unit0 = unit0, a.n_units = n_units;
    a.hg_major = 0;
    if (a.resident) a.resident = 0, a.ring = std::min(a.ring, 2);
  }
  a.tl_id = unit0 >= 0 ? -1 : tl_next(h);
  a.debug = img_debug_on(dgrad ? "dgrad" : "fwd", li);
  const ImgLayerState& S = h->il[li];
  const img::TapsSmem L = img::taps_smem(a, a_planes);
  const int grid = std::min(a.n_units * a.tiles, h->sm_avail);
  const CUtensorMap* mA = dgrad ? S.mapZ : S.mapX;
#define IMG_TAPS_LAUNCH(KIND, PL)                                                                            \
  do {                                                                                                       \
    CK(img_set_smem(img::conv_taps_kernel<KIND, PL>, L.total));                                              \
    CK(launch_pdl(h->pdl, img::conv_taps_kernel<KIND, PL>, dim3(grid), dim3(img::NTHREADS), L.total, h->stream, mA[0],  \
                  mA[1], S.mapW[0], S.mapW[1], a));                                                           \
  } while (0)
  if (dgrad) IMG_TAPS_LAUNCH(1, 2);
  else if (a_planes == 1) IMG_TAPS_LAUNCH(0, 1);
  else IMG_TAPS_LAUNCH(0, 2);
#undef IMG_TAPS_LAUNCH
  CK(cudaGetLastError());
  mark(h, dgrad ? "img_dgrad_L%d" : "img_fwd_L%d", li);
  return IDQN_OK;
}

// conv1 + conv2 forward of every net as one launch
static int img_launch_chain_fwd(idqn_handle* h) {
  ImgHost* H = (ImgHost*)h->img_host;
  img::ChainArgs c = H->chain;
  c.a.tl_id = tl_next(h);
  const img::ChainSmem L = img::chain_smem(c);
  const int per = (c.a.n_units + h->sm_avail - 1) / h->sm_avail;  // units of the busiest CTA
  const int grid = (c.a.n_units + per - 1) / per;                  // the fewest CTAs with that maximum
  CK(img_set_smem(img::conv_chain_fwd_kernel, L.total));
  CK(launch_pdl(h->pdl, img::conv_chain_fwd_kernel, dim3(grid), dim3(img::NTHREADS), L.total, h->stream, h->il[1].mapX[0],
                h->il[1].mapX[1], h->il[1].mapW[0], h->il[1].mapW[1], h->il[2].mapW[0], h->il[2].mapW[1], c));
  CK(cudaGetLastError());
  mark(h, "img_fwd_chain_L%d", 1);
  return IDQN_OK;
}

static int img_launch_wgrad(idqn_handle* h, int li, int a_planes) {
  ImgHost* H = (ImgHost*)h->img_host;
  img::WgradArgs a = H->wg[li];
  a.debug = img_debug_on("wgrad", li);
  a.tl_id = tl_next(h);
  const ImgLayerState& S = h->il[li];
  const img::WgradSmem L = img::wgrad_smem(a, a_planes);
  const int grid = a.heads * a.groups * a.tsplit;
  if (a_planes == 1) {
    CK(img_set_smem(img::conv_wgrad_kernel<1>, L.total));
    CK(launch_pdl(h->pdl, img::conv_wgrad_kernel<1>, dim3(grid), dim3(img::WG_THREADS), L.total, h->stream, S.mapXw[0], S.mapXw[1],
                  S.mapZw[0], S.mapZw[1], a));
  } else {
    CK(img_set_smem(img::conv_wgrad_kernel<2>, L.total));
    CK(launch_pdl(h->pdl, img::conv_wgrad_kernel<2>, dim3(grid), dim3(img::WG_THREADS), L.total, h->stream, S.mapXw[0], S.mapXw[1],
                  S.mapZw[0], S.mapZw[1], a));
  }
  CK(cudaGetLastError());
  mark(h, "img_wgrad_L%d", li);
  return IDQN_OK;
}

// forward (dgrad == false) or data gradient of the big Dense layer; z_dst: dgrad planes go to the dyZ layout of the
// preceding conv layer
static int dense_launch(idqn_handle* h, bool dgrad, bool z_dst, int unit0 = -1, int n_units = -1) {
  ImgHost* H = (ImgHost*)h->img_host;
  dense::Args a = dgrad ? H->ddg : H->dfwd;
  if (unit0 >= 0) a.unit0 = unit0, a.n_units = n_units;
  a.tl_id = unit0 >= 0 ? -1 : tl_next(h);
  const int li = IDQN_IMG_LAYERS;
  a.debug = img_debug_on(dgrad ? "ddgrad" : "dfwd", li);
  if (dgrad && z_dst) {
    const img::Geom& pg = H->g[li - 1];
    a.yh = h->il[li - 1].dz_hi, a.yl = h->il[li - 1].dz_lo;
    a.zP = pg.P, a.zW = pg.OW, a.zC = pg.OC, a.zOff = pg.T - 1, a.zRows = pg.ZRa, a.zstride = h->il[li - 1].dz_net_stride;
  }
  a.keep_heads = l2_keep_heads(h);
  const dense::Smem L = dense::smem_layout(a);
  int grid = std::min(a.n_units, h->sm_count);
  {
    // whole rounds: with u units on g CTAs the kernel takes ceil(u / g) units of time whatever g is; the fewest CTAs with
    // that maximum leave the partial last round (305 data-gradient units on 148 CTAs: nine CTAs with a third unit) no
    // idle bandwidth to wait for -- every CTA streams all the time and shares HBM with fewer others
    static const bool rounds_env = !getenv("IDQN_NO_ROUNDS");
    if (rounds_env && unit0 < 0) {
      const int per = (a.n_units + grid - 1) / grid;
      grid = (a.n_units + per - 1) / per;
    }
  }
  if (dgrad) {
    CK(img_set_smem(dense::dense_stream_kernel<1>, L.total));
    CK(launch_pdl(h->pdl, dense::dense_stream_kernel<1>, dim3(grid), dim3(dense::NTHREADS), L.total, h->stream,
                  H->fmapWd, H->fmapWd, H->dmapDy[0], H->dmapDy[1], a));
  } else {
    CK(img_set_smem(dense::dense_stream_kernel<0>, L.total));
    CK(launch_pdl(h->pdl, dense::dense_stream_kernel<0>, dim3(grid), dim3(dense::NTHREADS), L.total, h->stream,
                  H->fmapWf[0], H->fmapWf[1], H->dmapX[0], H->dmapX[1], a));
  }
  CK(cudaGetLastError());
  mark(h, dgrad ? "dense_dgrad_L%d" : "dense_fwd_L%d", li);
  return IDQN_OK;
}

// Dense_0 wgrad + Adam over the 8-row tiles [tile0, tile0 + ntiles) of every head (dense_wgrad_tma.cuh)
static int dense_wgrad_launch(idqn_handle* h, int tile0, int ntiles, bool keep_grads) {
  ImgHost* H = (ImgHost*)h->img_host;
  const Layer& l = h->layers[IDQN_IMG_LAYERS];
  dwt::Args a;
  a.heads = h->K, a.tile0 = tile0, a.ntiles = ntiles;
  a.I = l.g.Kd, a.O = l.g.OC;
  a.count = h->count;
  a.lr = h->cfg.learning_rate, a.b1 = 0.9f, a.b2 = 0.999f, a.eps = h->cfg.adam_eps;
  a.grad = keep_grads ? h->grad : nullptr;
  a.dyh = h->dact_hi + l.act_off, a.dyl = h->dact_lo + l.act_off, a.dystride = h->act_stride;
  // measured: 98.6 us with the default policy for the fp32 streams, 100.8 us with evict_first
  static const int sp = getenv("IDQN_L2_STREAM") ? atoi(getenv("IDQN_L2_STREAM")) : 0;
  a.stream_policy = sp == 0 ? tma::L2_EVICT_NORMAL : (sp == 2 ? tma::L2_EVICT_LAST : tma::L2_EVICT_FIRST);
  a.stride = h->stride, a.w_off = l.w_off;
  a.tl_id = tl_next(h);
  const int grid = std::min(a.heads * a.ntiles, h->sm_avail);
  CK(img_set_smem(dwt::dense_wgrad_adam_kernel, dwt::SMEM_TOTAL));
  CK(launch_pdl(0, dwt::dense_wgrad_adam_kernel, dim3(grid), dim3(dwt::NTHREADS), dwt::SMEM_TOTAL, h->stream, H->wmapX[0],
                H->wmapX[1], H->wmapP[0], H->wmapP[1], H->wmapP[2], a));
  CK(cudaGetLastError());
  mark(h, "dense_wgrad_adam_L%d", IDQN_IMG_LAYERS);
  return IDQN_OK;
}

// rebuild the fp32 activation of conv layer `layer` of net `net` from the planes the image path wrote
static int img_rebuild_activation(idqn_handle* h, int net, int layer) {
  ImgHost* H = (ImgHost*)h->img_host;
  const img::Geom& g = H->g[layer];
  img::PlaneDst d = H->fwd[layer].dst;
  float* out = h->act + (int64_t)net * h->act_stride + h->layers[layer].act_off;
  const int64_t total = (int64_t)h->B * g.OH * g.OW * g.OC;
  img::planes_to_f32_kernel<<<(int)std::min<int64_t>((total + 255) / 256, 4096), 256, 0, h->stream>>>(d, net, h->B, g.OH, g.OW,
                                                                                                 g.OC, out);
  CK(cudaGetLastError());
  return IDQN_OK;
}
