// libidqn_b200 — the i-DQN learning step (idqn.py:96-124 of the reference) on one B200.
//
// One step = forward of 2K nets (K online heads on s, K target heads on s'), the fused
// final-layer + Bellman-target + TD-loss kernel, backward of the K online heads, Adam.
// The sequence is captured once into a CUDA graph and replayed.
#include "common.cuh"
#include "gemm_simt.cuh"
#include "gemm_tc.cuh"
#include "sm_partition.cuh"

#include <algorithm>
#include <cmath>

// ------------------------------------------------------------------------------------------
static thread_local char g_err[512] = "";
void idqn_set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}
extern "C" const char* idqn_last_error(void) { return g_err; }
extern "C" int idqn_version(void) { return 100; }

// ------------------------------------------------------------------------------------------
// geometry
static void same_pad(int in, int k, int s, int* out, int* lo) {
  *out = (in + s - 1) / s;
  int total = std::max((*out - 1) * s + k - in, 0);
  *lo = total / 2;  // XLA: pad_lo = total // 2
}

static void finish_geom(ConvGeom& g) {
  g.Kd = g.KH * g.KW * g.IC;
  g.d_ohow = FastDiv(g.OH * g.OW);
  g.d_ow = FastDiv(g.OW);
  g.d_kwic = FastDiv(g.KW * g.IC);
  g.d_ic = FastDiv(g.IC);
  g.d_oc = FastDiv(g.OC);
}

static int build_layers(idqn_handle* h) {
  const idqn_config& c = h->cfg;
  int L = 0;
  int ih, iw, ic, start = 0;
  if (c.arch == IDQN_ARCH_CNN) {
    REQUIRE(c.n_features >= 3, "cnn needs >= 3 features (architectures/dqn.py:43-51)");
    static const int ks[3][2] = {{8, 4}, {4, 2}, {3, 1}};
    ih = c.obs[0], iw = c.obs[1], ic = c.obs[2];
    for (int i = 0; i < 3; ++i) {
      Layer& l = h->layers[L++];
      memset(&l, 0, sizeof(l));
      l.is_conv = 1, l.relu_out = 1, l.skip_from = -1;
      ConvGeom& g = l.g;
      g.B = c.batch_size;
      g.IH = ih, g.IW = iw, g.IC = ic;
      g.KH = g.KW = ks[i][0];
      g.S = ks[i][1];
      g.OC = c.features[i];
      same_pad(ih, g.KH, g.S, &g.OH, &g.PH);
      same_pad(iw, g.KW, g.S, &g.OW, &g.PW);
      finish_geom(g);
      snprintf(l.name, sizeof(l.name), "Conv_%d", i);
      ih = g.OH, iw = g.OW, ic = g.OC;
    }
    start = 3;
    h->in_elems = (int64_t)c.obs[0] * c.obs[1] * c.obs[2];
  } else if (c.arch == IDQN_ARCH_IMPALA) {
    // architectures/dqn.py:54-60: Stack(features[0]), Stack(features[1]), relu(Stack(features[2])); a Stack (:7-29) is
    // Conv_0 3x3 (no activation), max-pool 3x3 / 2 SAME, then twice x -> x + Conv(relu(Conv(relu(x))))
    REQUIRE(c.n_features >= 3, "impala needs >= 3 features (architectures/dqn.py:56-58)");
    ih = c.obs[0], iw = c.obs[1], ic = c.obs[2];
    for (int st = 0; st < 3; ++st) {
      for (int j = 0; j < 6; ++j) {  // j: 0 = Conv_0, 1 = pool, 2..5 = Conv_1..Conv_4
        REQUIRE(L < IDQN_MAX_LAYERS, "too many layers");
        Layer& l = h->layers[L++];
        memset(&l, 0, sizeof(l));
        l.is_conv = 1, l.skip_from = -1;
        ConvGeom& g = l.g;
        g.B = c.batch_size;
        g.IH = ih, g.IW = iw, g.IC = ic;
        g.KH = g.KW = 3;
        if (j == 1) {
          l.kind = IDQN_LAYER_POOL;
          g.S = 2, g.OC = ic;
          snprintf(l.name, sizeof(l.name), "Stack_%d/pool", st);
        } else {
          g.S = 1, g.OC = c.features[st];
          const int cj = j == 0 ? 0 : j - 1;
          snprintf(l.name, sizeof(l.name), "Stack_%d/Conv_%d", st, cj);
          if (cj == 1 || cj == 3) l.relu_in = 1, l.relu_out = 1;   // first conv of a block: relu(Conv(relu(x)))
          if (cj == 2 || cj == 4) l.skip_from = L - 3;             // second conv of a block: + block input
        }
        same_pad(ih, g.KH, g.S, &g.OH, &g.PH);
        same_pad(iw, g.KW, g.S, &g.OW, &g.PW);
        finish_geom(g);
        ih = g.OH, iw = g.OW, ic = g.OC;
      }
    }
    start = 3;
    h->in_elems = (int64_t)c.obs[0] * c.obs[1] * c.obs[2];
  } else if (c.arch == IDQN_ARCH_FC) {
    ih = iw = 1;
    ic = c.obs[0] * std::max(c.obs[1], 1) * std::max(c.obs[2], 1);
    h->in_elems = ic;
  } else {
    REQUIRE(false, "unknown architecture %d", c.arch);
  }
  int fan_in = ih * iw * ic;
  for (int i = start; i <= c.n_features; ++i) {
    REQUIRE(L < IDQN_MAX_LAYERS, "too many layers");
    Layer& l = h->layers[L++];
    memset(&l, 0, sizeof(l));
    l.skip_from = -1;
    l.relu_out = i < c.n_features;                          // every Dense but the last (architectures/dqn.py:67-70)
    l.relu_in = c.arch == IDQN_ARCH_IMPALA && i == start;   // relu(Stack_2(x)) feeds the trunk (:59)
    ConvGeom& g = l.g;
    g.B = c.batch_size;
    g.IH = g.IW = g.OH = g.OW = 1;
    g.KH = g.KW = g.S = 1;
    g.IC = fan_in;
    g.OC = (i == c.n_features) ? c.n_actions : c.features[i];
    finish_geom(g);
    snprintf(l.name, sizeof(l.name), "Dense_%d", i - start);
    fan_in = g.OC;
  }
  h->n_layers = L;
  h->n_param_layers = 0;
  int64_t off = 0, aoff = 0;
  for (int i = 0; i < L; ++i) {
    Layer& l = h->layers[i];
    REQUIRE(l.g.OC > 0 && l.g.Kd > 0, "layer %d has an empty dimension", i);
    if (l.kind == IDQN_LAYER_GEMM) {
      h->param_layer[h->n_param_layers++] = i;
      off = (off + 31) / 32 * 32;  // 128-byte aligned layer start
      l.w_off = off;
      l.b_off = off + (int64_t)l.g.Kd * l.g.OC;  // bias directly after the kernel: [Kd+1, OC] block
      off = l.b_off + l.g.OC;
    }
    l.act_off = aoff;
    l.act_size = (int64_t)c.batch_size * l.g.OH * l.g.OW * l.g.OC;
    aoff += (l.act_size + 31) / 32 * 32;
  }
  h->stride = (off + 127) / 128 * 128;
  h->act_stride = aoff;
  return IDQN_OK;
}

// ------------------------------------------------------------------------------------------
// launch planning (tile shape, split-K) — shared by workspace sizing and launching
struct GemmPlan {
  int bn, gx, gy, S, kchunk;
  int64_t part_floats;
  int tickets;
};
static GemmPlan plan_gemm(int M, int N, int K, int nz, int sms, bool allow_split) {
  GemmPlan p;
  p.bn = N <= 32 ? 32 : 64;
  p.gx = (M + 63) / 64;
  p.gy = (N + p.bn - 1) / p.bn;
  int tiles = p.gx * p.gy * nz;
  int kiters = (K + 15) / 16;
  int S = 1;
  if (allow_split && tiles < 2 * sms) {
    S = (2 * sms + tiles - 1) / tiles;
    S = std::min(S, std::max(1, kiters / 4));
    S = std::min(S, 64);
  }
  int it_per = (kiters + S - 1) / S;
  p.kchunk = it_per * 16;
  S = (K + p.kchunk - 1) / p.kchunk;
  p.S = S;
  p.part_floats = S > 1 ? (int64_t)nz * p.gx * p.gy * S * 64 * p.bn : 0;
  p.tickets = S > 1 ? nz * p.gx * p.gy : 0;
  return p;
}

// ------------------------------------------------------------------------------------------
// fused final Dense layer (fwd + bwd) + Bellman target + TD loss     (idqn.py:111-124; dqn.py:77-87)
struct HeadArgs {
  NetPtr hid;  // last hidden activations, nets [0,K) online / [K,2K) target, [B][H] each
  int H, A, B, K;
  const float* online;
  const float* target;
  int64_t stride, w_off, b_off;
  const int32_t* action;
  const float* reward;
  const uint8_t* terminal;
  float gamma_n;
  float* grad;   // arena
  float* dhid;   // [K][dstride] gradient w.r.t. the hidden activations (masked by relu'), may be null
  __nv_bfloat16 *dhid_hi, *dhid_lo;  // its bf16 planes (same offsets)
  int64_t dstride;
  int relu_mask;
  float* loss;
  double* loss_sum;
  float* td_abs;               // [K][B] |Q(s_b, a_b) - y_b| of this step: the priorities of prioritised replay (rb.update)
  const int32_t* loss_acc_on;  // device flag: 0 = this step's losses are NOT added to loss_sum (direct learn_on_batch calls)
  int32_t* count;
  float* q;      // [2K][B][A]
  // deferred split-K reduce of the preceding Dense layer (dense_stream.cuh): partial tiles [net*ptiles + tile][split][32][128]
  const float* part;
  int ptiles, psplits;
  int64_t pb_off;  // arena offset of that layer's bias
  int64_t hbias_off;  // >= 0: also write the bias gradient of the hidden layer (sum_b dhid) at this arena offset
  int cta0;           // head_q: first (net, sample) pair of this launch (best_action runs a single one)
  int tl_id;          // kernel timeline slot (IDQN_F_TIMELINE) or -1
};
#define HEAD_MAXA 32

// Q-values of the final Dense layer: one 128-thread CTA per (net, sample); threads stride the hidden units, keep all
// A partial sums (W rows are [A] contiguous) and finish with warp shuffles + a fixed-order cross-warp sum.  When the preceding Dense layer ran split-K
// (dense_stream.cuh) its partial tiles are summed here, in split order, together with its bias and relu, and the
// hidden activations are materialised for the backward kernels.
__global__ void __launch_bounds__(128) head_q_kernel(const HeadArgs a) {
  __shared__ float red[4][HEAD_MAXA];
  pdl_trigger();
  pdl_wait();
  ktl_begin(a.tl_id);
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int pair = blockIdx.x + a.cta0;
  const int net = pair / a.B, b = pair - net * a.B;
  const int k = net < a.K ? net : net - a.K;
  const float* base = (net < a.K ? a.online : a.target) + (int64_t)k * a.stride;
  const float* W = base + a.w_off;
  float* hv = const_cast<float*>(a.hid.get<float>(net)) + (int64_t)b * a.H;
  float acc[HEAD_MAXA];
#pragma unroll
  for (int i = 0; i < HEAD_MAXA; ++i) acc[i] = 0.f;
  if (a.part && a.H <= 4 * 128 && (a.H & 127) == 0 && a.psplits <= 16) {
    // latency path (Dense_0 of the NatureCNN: H = 512, 11 splits): every load of the thread -- bias, split partials,
    // final-layer weights -- is issued before the first use, so the CTA pays ONE memory round trip
    const int JT = a.H >> 7;
    float hb[4], pv[4][16];
#pragma unroll
    for (int t = 0; t < 4; ++t) {
      const int j = t * 128 + tid;
      hb[t] = t < JT ? __ldg(base + a.pb_off + j) : 0.f;
      const float* src = a.part + ((int64_t)(net * a.ptiles + t) * a.psplits) * (32 * 128) + b * 128 + tid;
#pragma unroll
      for (int sp = 0; sp < 16; ++sp) pv[t][sp] = (t < JT && sp < a.psplits) ? __ldcg(src + (int64_t)sp * (32 * 128)) : 0.f;
    }
#pragma unroll
    for (int t = 0; t < 4; ++t) {
      if (t < JT) {
        const int j = t * 128 + tid;
        float h = hb[t];
#pragma unroll
        for (int sp = 0; sp < 16; ++sp)
          if (sp < a.psplits) h += pv[t][sp];  // fixed order
        h = fmaxf(h, 0.f);
        hv[j] = h;
        const float* wr = W + (int64_t)j * a.A;
#pragma unroll
        for (int i = 0; i < HEAD_MAXA; ++i)
          if (i < a.A) acc[i] = fmaf(h, __ldg(wr + i), acc[i]);
      }
    }
  } else {
    for (int j = tid; j < a.H; j += 128) {
      float h;
      if (a.part) {
        const float* src = a.part + ((int64_t)(net * a.ptiles + (j >> 7)) * a.psplits) * (32 * 128) + b * 128 + (j & 127);
        h = __ldg(base + a.pb_off + j);
#pragma unroll 4
        for (int sp = 0; sp < a.psplits; ++sp) h += __ldcg(src + (int64_t)sp * (32 * 128));  // fixed order
        h = fmaxf(h, 0.f);
        hv[j] = h;
      } else {
        h = hv[j];
      }
      const float* wr = W + (int64_t)j * a.A;
#pragma unroll
      for (int i = 0; i < HEAD_MAXA; ++i)
        if (i < a.A) acc[i] = fmaf(h, __ldg(wr + i), acc[i]);
    }
  }
#pragma unroll
  for (int i = 0; i < HEAD_MAXA; ++i) {
    if (i < a.A) {
      float s = acc[i];
#pragma unroll
      for (int o = 16; o; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
      if (lane == 0) red[warp][i] = s;
    }
  }
  __syncthreads();
  if (tid < a.A) a.q[((int64_t)net * a.B + b) * a.A + tid] = ((red[0][tid] + red[1][tid]) + (red[2][tid] + red[3][tid])) + __ldg(base + a.b_off + tid);
  ktl_end(a.tl_id);
}

// y = r + (1-done) gamma^n max_a' Q_target; delta = Q(s,a) - y; loss_k = mean delta^2 and the backward of the
// final layer.  grid (ceil(H/32), K), 256 threads: every CTA recomputes the B coefficients (cheap) and owns 32
// hidden units: thread (b-slot, 4 units) writes dL/dhidden, threads (unit, action) the kernel gradient.
__global__ void __launch_bounds__(256) head_bwd_kernel(const HeadArgs a) {
  extern __shared__ float sm[];
  pdl_trigger();
  pdl_wait();
  ktl_begin(a.tl_id);
  const int k = blockIdx.y, B = a.B, A = a.A, H = a.H, tid = threadIdx.x;
  float* coef = sm;        // [B]
  float* lterm = sm + B;   // [B]
  int* act_s = reinterpret_cast<int*>(sm + 2 * B);  // [B]
  float* htile = sm + 3 * B;                        // [B][32] hidden activations of this CTA's units
  float* wtile = htile + 32 * B;                    // [32][A] final-layer weights of this CTA's units
  float* dtile = wtile + 32 * A;                    // [B][32] dL/dhidden of this CTA's units (hbias_off >= 0)
  const int j0 = blockIdx.x * 32;
  const float* hid = a.hid.get<float>(k);
  const float* Wk = a.online + (int64_t)k * a.stride + a.w_off;
  // every global load of the CTA is issued here, before the first use: one memory round trip
  for (int e = tid; e < 32 * B; e += blockDim.x) {
    const int b = e >> 5, j = j0 + (e & 31);
    htile[e] = j < H ? __ldg(hid + (int64_t)b * H + j) : 0.f;
  }
  for (int e = tid; e < 32 * A; e += blockDim.x) wtile[e] = j0 + e / A < H ? __ldg(Wk + (int64_t)j0 * A + e) : 0.f;
  const float* qo = a.q + (int64_t)k * B * A;
  const float* qt = a.q + (int64_t)(a.K + k) * B * A;
  for (int b = tid; b < B; b += blockDim.x) {
    float mx = qt[b * A];
    for (int i = 1; i < A; ++i) mx = fmaxf(mx, qt[b * A + i]);
    const float notdone = a.terminal[b] ? 0.f : 1.f;
    const float y = a.reward[b] + (notdone * a.gamma_n) * mx;
    const int ab = a.action[b];
    const float d = qo[b * A + ab] - y;
    if (blockIdx.x == 0) a.td_abs[k * B + b] = fabsf(d);
    lterm[b] = d * d;
    coef[b] = 2.f * d / (float)B;  // d mean_b(delta^2) / d Q(s_b, a_b)
    act_s[b] = ab;
  }
  __syncthreads();
  if (blockIdx.x == 0) {
    if (tid == 0) {
      float s = 0.f;
      for (int b = 0; b < B; ++b) s += lterm[b];
      s /= (float)B;
      a.loss[k] = s;
      if (*a.loss_acc_on) a.loss_sum[k] += (double)s;  // idqn.py:72 accumulates inside update_online_params only
      a.count[k] += 1;  // ScaleByAdamState.count, read by the Adam kernels that follow
    }
    float* gb = a.grad + (int64_t)k * a.stride + a.b_off;
    for (int i = tid; i < A; i += blockDim.x) {
      float s = 0.f;
      for (int b = 0; b < B; ++b)
        if (act_s[b] == i) s += coef[b];
      gb[i] = s;
    }
  }
  // kernel gradient: 32 units x A actions
  for (int e = tid; e < 32 * A; e += blockDim.x) {
    const int u = e / A, i = e - u * A;
    if (j0 + u < H) {
      float s = 0.f;
      for (int b = 0; b < B; ++b)
        if (act_s[b] == i) s = fmaf(coef[b], htile[b * 32 + u], s);
      a.grad[(int64_t)k * a.stride + a.w_off + (int64_t)(j0 + u) * A + i] = s;
    }
  }
  if (a.dhid) {
    // dL/dhidden[b][j] = coef_b W[j][a_b], masked by relu'; thread = (b-slot of 8 lanes x 4 units)
    float* dh = a.dhid + (int64_t)k * a.dstride;
    __nv_bfloat16* dhh = a.dhid_hi + (int64_t)k * a.dstride;
    __nv_bfloat16* dhl = a.dhid_lo + (int64_t)k * a.dstride;
    const int jj = (tid & 7) * 4;
    const bool vec = (H & 3) == 0 && (a.dstride & 3) == 0;  // 4 units of a thread: one float4 + two 8-byte plane stores
    for (int b = tid >> 3; b < B; b += blockDim.x >> 3) {
      const float cb = coef[b];
      const int ab = act_s[b];
      float v[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        v[u] = cb * wtile[(jj + u) * A + ab];
        if ((a.relu_mask && !(htile[b * 32 + jj + u] > 0.f)) || j0 + jj + u >= H) v[u] = 0.f;
        if (a.hbias_off >= 0) dtile[b * 32 + jj + u] = v[u];
      }
      const int64_t o = (int64_t)b * H + j0 + jj;
      if (vec && j0 + jj + 3 < H) {
        const float4 v4 = make_float4(v[0], v[1], v[2], v[3]);
        *reinterpret_cast<float4*>(dh + o) = v4;
        uint2 h2, l2;
        tc::split4(v4, h2, l2);
        *reinterpret_cast<uint2*>(dhh + o) = h2;
        *reinterpret_cast<uint2*>(dhl + o) = l2;
      } else {
#pragma unroll
        for (int u = 0; u < 4; ++u)
          if (j0 + jj + u < H) {
            dh[o + u] = v[u];
            tc::st1_planes(dhh + o + u, dhl + o + u, v[u]);
          }
      }
    }
    if (a.hbias_off >= 0) {
      // bias gradient of the hidden layer = sum_b dL/dhidden[b][j], fixed order (dense_wgrad_tma.cuh leaves it to us)
      __syncthreads();
      if (tid < 32 && j0 + tid < H) {
        float s = 0.f;
        for (int b = 0; b < B; ++b) s += dtile[b * 32 + tid];
        a.grad[(int64_t)k * a.stride + a.hbias_off + j0 + tid] = s;
      }
    }
  }
  ktl_end(a.tl_id);
}

// ------------------------------------------------------------------------------------------
// optax.adam (scale_by_adam b1=.9 b2=.999 eps, eps_root=0; scale(-lr); apply_updates)  idqn.py:52,106-107
// over the float4 range [off4, off4 + n4) of every head's arena
// Two arena ranges per launch: blocks [0, nblk_a) walk range A, the rest range B.  part != nullptr: the gradient of
// range A is the sum, in a fixed order, of `groups` partial gradients laid out [head][group][span] in arena
// coordinates (conv_wgrad_kernel); gout (optional) receives the reduced gradient.  Range B reads g.
__global__ void __launch_bounds__(256) adam_kernel(float4* __restrict__ p, const float4* __restrict__ g,
                                                   float4* __restrict__ m, float4* __restrict__ v,
                                                   uint2* __restrict__ ph, uint2* __restrict__ pl,
                                                   const int32_t* __restrict__ count, int64_t stride4, int64_t off4_a,
                                                   int64_t n4_a, int nblk_a, int64_t off4_b, int64_t n4_b, float lr,
                                                   float b1, float b2, float eps, const float4* __restrict__ part_a,
                                                   int groups, int64_t span4, float4* __restrict__ gout, int tl_id) {
  pdl_trigger();
  pdl_wait();
  ktl_begin(tl_id);
  const int k = blockIdx.y;
  const tc::AdamCoef ac = tc::adam_coef(b1, b2, lr, eps, count[k]);  // count already incremented for this step
  const bool in_a = (int)blockIdx.x < nblk_a;
  const int64_t off4 = in_a ? off4_a : off4_b, n4 = in_a ? n4_a : n4_b;
  const int bx = in_a ? blockIdx.x : blockIdx.x - nblk_a, nbx = in_a ? nblk_a : gridDim.x - nblk_a;
  const float4* part = in_a ? part_a : nullptr;
  const int64_t base = (int64_t)k * stride4 + off4;
  for (int64_t i = (int64_t)bx * blockDim.x + threadIdx.x; i < n4; i += (int64_t)nbx * blockDim.x) {
    float4 G;
    const float4 P0 = p[base + i], M0 = m[base + i], V0 = v[base + i];  // requested before the partial sums are needed
    if (part) {
      G = make_float4(0.f, 0.f, 0.f, 0.f);
      const float4* src = part + (int64_t)k * groups * span4 + off4 + i;
      if (groups <= 16) {
        // every partial of this quad is requested before the first add: one memory round trip; fixed summation order
        float4 t[16];
#pragma unroll
        for (int u = 0; u < 16; ++u) t[u] = u < groups ? __ldcs(src + (int64_t)u * span4) : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
        for (int u = 0; u < 16; ++u)
          if (u < groups) G.x += t[u].x, G.y += t[u].y, G.z += t[u].z, G.w += t[u].w;
      } else {
#pragma unroll 4
        for (int u = 0; u < groups; ++u) {
          const float4 t = __ldcs(src + (int64_t)u * span4);
          G.x += t.x, G.y += t.y, G.z += t.z, G.w += t.w;
        }
      }
      if (gout) gout[base + i] = G;
    } else {
      G = __ldcs(g + base + i);
    }
    float4 P = P0, M = M0, V = V0;
    tc::adam_elem(ac, G.x, P.x, M.x, V.x);
    tc::adam_elem(ac, G.y, P.y, M.y, V.y);
    tc::adam_elem(ac, G.z, P.z, M.z, V.z);
    tc::adam_elem(ac, G.w, P.w, M.w, V.w);
    p[base + i] = P;
    m[base + i] = M;
    v[base + i] = V;
    uint2 h2, l2;
    tc::split4(P, h2, l2);  // keep the bf16 hi/lo planes of the weights current
    ph[base + i] = h2;
    pl[base + i] = l2;
  }
  ktl_end(tl_id);
}

__global__ void argmax_kernel(const float* __restrict__ q, int A, int32_t* out) {
  if (threadIdx.x == 0 && blockIdx.x == 0) {
    int best = 0;
    float bv = q[0];
    for (int i = 1; i < A; ++i)
      if (q[i] > bv) bv = q[i], best = i;  // first maximum, like jnp.argmax
    *out = best;
  }
}

// idqn_select_actions: one warp per environment.  code[i] >= 0: greedy, out[i] = the first argmax of the Q row code[i]
// (argmax_kernel's result, NaN included: a NaN at index 0 wins, any later NaN is never taken); code[i] < 0: exploring,
// out[i] = -1 - code[i], the random action drawn on the host.  code == nullptr: every environment is greedy on row i.
__global__ void act_select_kernel(const float* __restrict__ q, int A, const int32_t* __restrict__ code, int n,
                                  int32_t* __restrict__ out) {
  const int i = (int)((blockIdx.x * blockDim.x + threadIdx.x) >> 5), lane = threadIdx.x & 31;
  if (i >= n) return;
  const int c = code ? code[i] : i;
  if (c < 0) {
    if (lane == 0) out[i] = -1 - c;
    return;
  }
  const float* row = q + (int64_t)c * A;
  float v = lane < A ? row[lane] : 0.f;
  int idx = lane < A && !(lane > 0 && v != v) ? lane : HEAD_MAXA;  // HEAD_MAXA: no candidate
  for (int o = 16; o; o >>= 1) {
    const float v2 = __shfl_xor_sync(0xffffffffu, v, o);
    const int i2 = __shfl_xor_sync(0xffffffffu, idx, o);
    if (i2 < HEAD_MAXA && (idx == HEAD_MAXA || v2 > v || (v2 == v && i2 < idx) || (i2 == 0 && v2 != v2))) v = v2, idx = i2;
  }
  if (lane == 0) out[i] = idx;
}

// ------------------------------------------------------------------------------------------
// every kernel launch of the step goes through mark(): counts launches and, when profiling, drops an event
// timeline slot of the launch about to be enqueued (its index inside the step), -1 when the timeline is off
static int tl_next(const idqn_handle* h) {
  return ((h->cfg.flags & IDQN_F_TIMELINE) && h->n_launch < IDQN_KTL_MAX) ? h->n_launch : -1;
}
static void mark(idqn_handle* h, const char* fmt, int li) {
  if ((h->cfg.flags & IDQN_F_TIMELINE) && h->n_launch < IDQN_KTL_MAX) snprintf(h->tl_name[h->n_launch], 32, fmt, li);
  h->n_launch++;
  if (h->prof_on && h->prof_n < IDQN_PROF_MAX) {
    snprintf(h->prof_name[h->prof_n], 32, fmt, li);
    cudaEventRecord(h->prof_ev[h->prof_n + 1], h->stream);
    h->prof_n++;
  }
}

static inline int round16(int n) { return (n + 15) / 16 * 16; }
static bool use_tc(const idqn_handle* h) { return !(h->cfg.flags & IDQN_F_SIMT_ONLY); }

// which layers the tensor-core kernels cover (vector-load friendly shapes); everything else runs the fp32 SIMT path
static bool tc_conv_ok(const Layer& l) {
  const ConvGeom& g = l.g;
  const bool ic_ok = (g.IC % 8 == 0) || g.IC == 4;  // 16-byte operand units, or two 8-byte taps of four channels
  return l.is_conv && ic_ok && g.OC % 8 == 0 && g.OC <= 256 && g.IC <= 256;
}
static bool tc_dense_ok(const idqn_handle* h, const Layer& l) {
  const ConvGeom& g = l.g;
  return !l.is_conv && g.IC % 8 == 0 && g.OC % 16 == 0 && h->B <= 256 && g.IC >= 64;
}
static int splitk_for(int tiles, int kiters, int sms) {
  int S = 1;
  if (tiles < 2 * sms) {
    S = (2 * sms + tiles - 1) / tiles;
    S = std::min(S, std::max(1, kiters / 2));
    S = std::min(S, 64);
  }
  return std::max(S, 1);
}

static int check_ws(idqn_handle* h, int64_t part, int tickets, const char* what, int li) {
  if (part > h->part_floats || tickets > h->n_tickets) {
    idqn_set_error("internal: split-K workspace too small (%s layer %d: %lld floats, %d tickets)", what, li,
                   (long long)part, tickets);
    return IDQN_EINVAL;
  }
  return IDQN_OK;
}

#include "img_host.cuh"

// the TMA-pipelined wgrad+Adam kernel (dense_wgrad_tma.cuh) covers the big Dense layer of the image path
static bool dense_wgrad_tma_ok(const idqn_handle* h, int li) {
  if (!h->img_on || !h->img_host || (h->cfg.flags & (IDQN_F_OLD_WGRAD | IDQN_F_SIMT_ONLY))) return false;
  const ImgHost* H = (const ImgHost*)h->img_host;
  return li == IDQN_IMG_LAYERS && H->dense_on && H->wgrad_tma_on;
}

// ---- planes -----------------------------------------------------------------------------------------------
// bf16 planes of the input batch (first layer operand of the tensor-core path); part of the captured step
static int launch_input_planes(idqn_handle* h, int x_u8, int nsamples, int two) {
  const int64_t n = (int64_t)nsamples * h->in_elems;
  if (n % 8 != 0) {
    idqn_set_error("internal: input of %lld elements is not a multiple of 8", (long long)n);
    return IDQN_EINVAL;
  }
  const int64_t full = (int64_t)h->B * h->in_elems;
  const int blocks = (int)std::min<int64_t>((n / 8 + 255) / 256, 4096);
  for (int i = 0; i < (two ? 2 : 1); ++i) {
    const void* src = i ? h->s2 : h->s;
    if (x_u8)
      tcg::u8_to_plane_kernel<<<blocks, 256, 0, h->stream>>>((const uint8_t*)src, h->in_hi + i * full, n / 8);
    else
      tcg::to_planes_kernel<<<blocks, 256, 0, h->stream>>>((const float*)src, h->in_hi + i * full, h->in_lo + i * full,
                                                         n / 8);
    CK(cudaGetLastError());
    mark(h, "input_planes_%d", i);
  }
  return IDQN_OK;
}

static int to_planes_range(idqn_handle* h, int w, int head, int64_t lo_f, int64_t hi_f) {
  if (hi_f <= lo_f) return IDQN_OK;
  const float* src = (w ? h->target : h->online) + (int64_t)head * h->stride;
  __nv_bfloat16* ph = (w ? h->wtg_hi : h->won_hi) + (int64_t)head * h->stride;
  __nv_bfloat16* pl = (w ? h->wtg_lo : h->won_lo) + (int64_t)head * h->stride;
  const int64_t n8 = (hi_f - lo_f) / 8;
  const int blocks = (int)std::min<int64_t>((n8 + 255) / 256, 8192);
  tcg::to_planes_kernel<<<blocks, 256, 0, h->stream>>>(src + lo_f, ph + lo_f, pl + lo_f, n8);
  CK(cudaGetLastError());
  return IDQN_OK;
}

// weights uploaded from the host / received from a neighbour: rebuild their planes (outside the captured step).  With
// fast_dense the big Dense layer keeps no planes: only the small ranges around it are converted.
static int refresh_planes(idqn_handle* h) {
  for (int w = 0; w < 2; ++w) {
    unsigned long long dirty = h->planes_dirty[w];
    if (!dirty) continue;
    if (h->fast_dense) {
      for (int k = 0; k < h->K; ++k) {
        if (!((dirty >> 63) || (k < 63 && ((dirty >> k) & 1ull)))) continue;
        int rc = to_planes_range(h, w, k, 0, h->d0_lo);
        if (!rc) rc = to_planes_range(h, w, k, h->d0_hi, h->stride);
        if (rc) return rc;
        if (k < 64) h->dense0_valid[w] &= ~(1ull << k);
      }
      h->planes_dirty[w] = 0;
      continue;
    }
    const float* src = w ? h->target : h->online;
    __nv_bfloat16 *hi = w ? h->wtg_hi : h->won_hi, *lo = w ? h->wtg_lo : h->won_lo;
    int first = 0, count = h->K;  // one launch over a contiguous run of heads
    if (!(dirty >> 63)) {
      while (!((dirty >> first) & 1ull)) ++first;
      int last = first;
      for (int k = first; k < h->K && k < 63; ++k)
        if ((dirty >> k) & 1ull) last = k;
      count = last - first + 1;
    }
    const int64_t n8 = (int64_t)count * h->stride / 8, o = (int64_t)first * h->stride;
    const int blocks = (int)std::min<int64_t>((n8 + 255) / 256, 8192);
    tcg::to_planes_kernel<<<blocks, 256, 0, h->stream>>>(src + o, hi + o, lo + o, n8);
    CK(cudaGetLastError());
    h->planes_dirty[w] = 0;
  }
  return IDQN_OK;
}

// the generic tensor-core kernels (network.apply on arbitrary arenas / batch sizes) read planes of EVERY layer: rebuild the
// big Dense layer's planes of one head from its fp32 master when they are not current
static int ensure_dense0_planes(idqn_handle* h, int w, int head) {
  if (!h->fast_dense) return IDQN_OK;
  if (head < 64 && ((h->dense0_valid[w] >> head) & 1ull)) return IDQN_OK;
  int rc = to_planes_range(h, w, head, h->d0_lo, h->d0_hi);
  if (rc) return rc;
  if (head < 64) h->dense0_valid[w] |= 1ull << head;
  return IDQN_OK;
}

// copy the maintained planes of `nheads` heads (fp32 masters are copied by the caller): all of them, or with fast_dense
// only the ranges around the big Dense layer
static int copy_planes(idqn_handle* h, __nv_bfloat16* dhi, __nv_bfloat16* dlo, const __nv_bfloat16* shi,
                       const __nv_bfloat16* slo, int nheads) {
  if (nheads <= 0) return IDQN_OK;
  if (!h->fast_dense) {
    CK(cudaMemcpyAsync(dhi, shi, 2 * h->stride * nheads, cudaMemcpyDeviceToDevice, h->stream));
    CK(cudaMemcpyAsync(dlo, slo, 2 * h->stride * nheads, cudaMemcpyDeviceToDevice, h->stream));
    return IDQN_OK;
  }
  const size_t pitch = 2 * (size_t)h->stride;
  const int64_t r0[2] = {0, h->d0_hi}, r1[2] = {h->d0_lo, h->stride};
  for (int r = 0; r < 2; ++r) {
    const size_t width = 2 * (size_t)(r1[r] - r0[r]);
    if (!width) continue;
    CK(cudaMemcpy2DAsync(dhi + r0[r], pitch, shi + r0[r], pitch, width, nheads, cudaMemcpyDeviceToDevice, h->stream));
    CK(cudaMemcpy2DAsync(dlo + r0[r], pitch, slo + r0[r], pitch, width, nheads, cudaMemcpyDeviceToDevice, h->stream));
  }
  return IDQN_OK;
}

// ---- forward ---------------------------------------------------------------------------------------------
// nets: total nets; groups of `nh` consecutive nets share one input (conv0: online heads share s, target heads s')
// xkind: 0 = layer input is the staged batch (h->s / h->s2, planes in_hi/in_lo), 1 = previous layer's activations
struct FwdIO {
  NetPtr x;        // fp32 / u8 input (SIMT path)
  NetPtr xh, xl;   // its planes (tensor-core path)
  NetPtr w;        // fp32 arenas
  NetPtr wh, wl;   // weight planes
  float* y;
  __nv_bfloat16 *yh, *yl;
  int64_t ystride;
};

// the consumer of layer li reads relu(output): its planes hold relu(y) while the fp32 activation stays linear (residual input)
static bool planes_relu_of(const idqn_handle* h, int li) { return li + 1 < h->n_layers && h->layers[li + 1].relu_in; }

static int launch_fwd_layer(idqn_handle* h, int li, int nz, int nh, int nsamples, const FwdIO& io, int x_u8, int relu,
                            bool dry, int64_t* ws_part, int* ws_tick) {
  const Layer& l = h->layers[li];
  const float* skip = (l.skip_from >= 0 && io.y) ? io.y - l.act_off + h->layers[l.skip_from].act_off : nullptr;
  const float scale = (li == 0 && h->cfg.arch != IDQN_ARCH_FC) ? (1.0f / 255.0f) : 1.0f;  // architectures/dqn.py:44,57
  if (use_tc(h) && tc_conv_ok(l) && nsamples * l.g.OH * l.g.OW >= 64) {
    tcg::TcFwdConv p;
    p.g = l.g, p.g.B = nsamples;
    p.xh = io.xh, p.xl = io.xl, p.wh = io.wh, p.wl = io.wl, p.w = io.w;
    p.w_off = l.w_off, p.b_off = l.b_off;
    p.y = io.y, p.yh = io.yh, p.yl = io.yl, p.ystride = io.ystride, p.scale = scale, p.relu = relu;
    p.skip = skip, p.planes_relu = planes_relu_of(h, li);
    p.nh = nh;
    p.hpt = std::max(1, std::min(nh, 256 / l.g.OC));
    p.M = nsamples * l.g.OH * l.g.OW, p.K = l.g.Kd;
    p.NT = round16(p.hpt * l.g.OC);
    const int planes = (li == 0 && x_u8) ? 1 : 2;
    p.nstage = tcg::pick_stages(planes, p.NT, (p.K + 31) / 32);
    if (dry) return IDQN_OK;
    dim3 grid((p.M + 127) / 128, (nh + p.hpt - 1) / p.hpt, nz / nh);
    const bool halfu = l.g.IC == 4;
    if (planes == 1 && halfu) CK((tcg::launch_tc<false, true, 1, true, false, false>(p, grid, h->part, h->tickets, h->stream)));
    else if (planes == 1) CK((tcg::launch_tc<false, true, 1, false, false, false>(p, grid, h->part, h->tickets, h->stream)));
    else if (halfu) CK((tcg::launch_tc<false, true, 2, true, false, false>(p, grid, h->part, h->tickets, h->stream)));
    else CK((tcg::launch_tc<false, true, 2, false, false, false>(p, grid, h->part, h->tickets, h->stream)));
    mark(h, "tc_fwd_L%d", li);
    return IDQN_OK;
  }
  if (use_tc(h) && tc_dense_ok(h, l) && nsamples <= 256) {
    tcg::TcFwdDenseT p;
    p.xh = io.xh, p.xl = io.xl, p.wh = io.wh, p.wl = io.wl, p.w = io.w;
    p.w_off = l.w_off, p.b_off = l.b_off;
    p.y = io.y, p.yh = io.yh, p.yl = io.yl, p.ystride = io.ystride, p.relu = relu;
    p.I = l.g.Kd, p.O = l.g.OC, p.B = nsamples;
    p.NT = round16(nsamples);
    const int mt = (p.O + 127) / 128;
    p.S = splitk_for(mt * nz, (p.I + 31) / 32, 2 * h->sm_count);  // weight streaming: more CTAs in flight
    const int it_per = ((p.I + 31) / 32 + p.S - 1) / p.S;
    p.kchunk = it_per * 32;
    p.S = (p.I + p.kchunk - 1) / p.kchunk;
    p.nstage = tcg::pick_stages(2, p.NT, it_per);
    const int64_t part = p.S > 1 ? (int64_t)nz * mt * p.S * p.NT * 128 : 0;
    const int tick = p.S > 1 ? nz * mt : 0;
    if (dry) {
      *ws_part = std::max(*ws_part, part), *ws_tick = std::max(*ws_tick, tick);
      return IDQN_OK;
    }
    int rc = check_ws(h, part, tick, "tc fwd dense", li);
    if (rc) return rc;
    dim3 grid(mt, 1, nz * p.S);
    CK((tcg::launch_tc<true, false, 2, false, false, true>(p, grid, h->part, h->tickets, h->stream)));
    mark(h, "tc_fwd_L%d", li);
    return IDQN_OK;
  }
  FwdProb p;
  p.g = l.g;
  p.g.B = nsamples;
  p.x = io.x;
  p.x_u8 = x_u8;
  p.w = io.w;
  p.w_off = l.w_off;
  p.b_off = l.b_off;
  p.y = io.y, p.yh = io.yh, p.yl = io.yl;
  p.ystride = io.ystride;
  p.scale = scale;
  p.relu = relu;
  p.relu_in = l.relu_in;
  p.planes_relu = planes_relu_of(h, li);
  p.skip = skip;  // the residual input lives in the same activation block as y (same base, same net stride)
  p.nz = nz;
  p.M = nsamples * l.g.OH * l.g.OW;
  p.N = l.g.OC;
  p.K = l.g.Kd;
  GemmPlan gp = plan_gemm(p.M, p.N, p.K, nz, h->sm_count, true);
  p.S = gp.S;
  p.kchunk = gp.kchunk;
  if (dry) {
    *ws_part = std::max(*ws_part, gp.part_floats), *ws_tick = std::max(*ws_tick, gp.tickets);
    return IDQN_OK;
  }
  int rc = check_ws(h, gp.part_floats, gp.tickets, "fwd", li);
  if (rc) return rc;
  CK((launch_gemm_simt<true, false>(p, nz * p.S, h->part, h->tickets, h->stream)));
  mark(h, "fwd_L%d", li);
  return IDQN_OK;
}

// ---- max-pool (impala) ---------------------------------------------------------------------------------------------
static PoolArgs pool_args(const Layer& l, int nz, int nsamples) {
  PoolArgs a;
  memset(&a, 0, sizeof(a));
  a.nz = nz, a.B = nsamples, a.IH = l.g.IH, a.IW = l.g.IW, a.C = l.g.IC, a.OH = l.g.OH, a.OW = l.g.OW;
  a.PH = l.g.PH, a.PW = l.g.PW, a.K = l.g.KH, a.S = l.g.S;
  return a;
}
// step = the learning step's forward over [online K | target K]: the choices of the online nets are recorded for the backward
static int launch_pool_fwd(idqn_handle* h, int li, int nz, int nsamples, const float* x, float* y, int64_t stride, bool step = false) {
  PoolArgs a = pool_args(h->layers[li], nz, nsamples);
  a.x = x, a.y = y, a.xstride = a.ystride = stride;
  a.ph = h->act_hi + (y - h->act), a.pl = h->act_lo + (y - h->act), a.planes_relu = planes_relu_of(h, li);
  const int64_t total = (int64_t)nz * nsamples * a.OH * a.OW * a.C;
  const bool fast = pool3_v4_ok(a, a.x, a.y, a.y);
  if (step) {
    h->pool_arg_ok[li] = fast && h->pool_arg != nullptr;
    if (h->pool_arg_ok[li]) a.arg = h->pool_arg + (y - h->act), a.arg_nets = h->K;
  }
  if (fast)
    maxpool3_fwd_v4_kernel<<<dim3((unsigned)((a.OH * a.OW * (a.C / 4) + 255) / 256), (unsigned)(nz * nsamples)), 256, 0, h->stream>>>(a);
  else
    maxpool_fwd_kernel<<<(unsigned)std::min<int64_t>((total + 255) / 256, h->sm_count * 16), 256, 0, h->stream>>>(a);
  CK(cudaGetLastError());
  mark(h, "pool_fwd_L%d", li);
  return IDQN_OK;
}
// dact of layer li-1 from dact of the pool layer li (online nets)
static int launch_pool_bwd(idqn_handle* h, int li) {
  const Layer &l = h->layers[li], &prev = h->layers[li - 1];
  PoolArgs a = pool_args(l, h->K, h->B);
  a.x = h->act + prev.act_off, a.dy = h->dact + l.act_off, a.dx = h->dact + prev.act_off;
  a.ph = h->dact_hi + prev.act_off, a.pl = h->dact_lo + prev.act_off;
  a.xstride = a.ystride = h->act_stride;
  if (h->pool_arg_ok[li]) a.arg = h->pool_arg + l.act_off, a.arg_nets = h->K;  // else the kernel re-scans the windows
  const int64_t total = (int64_t)h->K * h->B * a.IH * a.IW * a.C;
  if (pool3_v4_ok(a, a.x, a.dy, a.dx))
    maxpool3_bwd_v4_kernel<<<dim3((unsigned)((a.IH * a.IW * (a.C / 4) + 255) / 256), (unsigned)(h->K * h->B)), 256, 0, h->stream>>>(a);
  else
    maxpool_bwd_kernel<<<(unsigned)std::min<int64_t>((total + 255) / 256, h->sm_count * 16), 256, 0, h->stream>>>(a);
  CK(cudaGetLastError());
  mark(h, "pool_bwd_L%d", li);
  return IDQN_OK;
}

// ---- weight gradient (+ bias gradient through the ones row) -------------------------------------------------
static int launch_wgrad_layer(idqn_handle* h, int li, int x_u8, bool dry, int64_t* ws_part, int* ws_tick) {
  const Layer& l = h->layers[li];
  const int K = h->K;
  NetPtr x, xh, xl;
  if (li == 0) {
    x = NetPtr{h->s, h->s, 0, 0, K};
    xh = NetPtr{h->in_hi, h->in_hi, 0, 0, K};
    xl = NetPtr{h->in_lo, h->in_lo, 0, 0, K};
  } else {
    const int64_t o = h->layers[li - 1].act_off;
    x = NetPtr{h->act + o, h->act + o, h->act_stride, h->act_stride, K};
    xh = NetPtr{h->act_hi + o, h->act_hi + o, h->act_stride, h->act_stride, K};
    xl = NetPtr{h->act_lo + o, h->act_lo + o, h->act_stride, h->act_stride, K};
  }
  const int xu = (li == 0) ? x_u8 : 0;
  const float scale = (li == 0 && h->cfg.arch != IDQN_ARCH_FC) ? (1.0f / 255.0f) : 1.0f;
  const bool keep = (h->cfg.flags & IDQN_F_KEEP_GRADS) != 0;
  if (dense_wgrad_tma_ok(h, li)) {
    if (dry) return IDQN_OK;
    const int mt = l.g.Kd / dwt::TM;
    const int t0 = h->wg_tiles > 0 ? h->wg_tile0 : 0;
    const int nt = h->wg_tiles > 0 ? std::min(h->wg_tiles, mt - t0) : mt;
    return nt > 0 ? dense_wgrad_launch(h, t0, nt, keep) : IDQN_OK;
  }
  if (use_tc(h) && tc_dense_ok(h, l)) {
    // dW = x^T dy with K = batch: the tile is final after one k-block, so Adam runs in the epilogue and the
    // gradient of the (98%-of-all-parameters) Dense_0 kernel never goes to HBM.  h->wg_tile0 / wg_tiles select a
    // range of 128-row tiles (the step splits this HBM-bound kernel over an SM partition and the whole machine)
    tcg::TcWgradDenseAdam p;
    p.xh = xh, p.xl = xl;
    p.dyh = h->dact_hi + l.act_off, p.dyl = h->dact_lo + l.act_off, p.dystride = h->act_stride;
    p.ones = h->ones;
    p.W = h->online, p.mu = h->mu, p.nu = h->nu, p.grad = keep ? h->grad : nullptr;
    p.Wh = h->won_hi, p.Wl = h->won_lo;
    p.stride = h->stride, p.w_off = l.w_off;
    p.count = h->count;
    p.lr = h->cfg.learning_rate, p.b1 = 0.9f, p.b2 = 0.999f, p.eps = h->cfg.adam_eps;
    p.I = l.g.Kd, p.O = l.g.OC, p.B = h->B;
    p.NT = std::min(128, round16(p.O));  // 128 TMEM columns -> more CTAs per SM for the Adam streams
    p.nstage = 2;
    p.adam = 1;
    if (dry) return IDQN_OK;
    const int mt = (p.I + 1 + 127) / 128;
    p.bx0 = h->wg_tiles > 0 ? h->wg_tile0 : 0;
    const int nt = h->wg_tiles > 0 ? std::min(h->wg_tiles, mt - p.bx0) : mt;
    if (nt <= 0) return IDQN_OK;
    dim3 grid(nt, (p.O + p.NT - 1) / p.NT, K);
    CK((tcg::launch_tc<true, true, 2, false, false, false>(p, grid, h->part, h->tickets, h->stream, h->pdl != 0)));
    mark(h, "tc_wgrad_adam_L%d", li);
    return IDQN_OK;
  }
  if (use_tc(h) && tc_conv_ok(l)) {
    tcg::TcWgradConv p;
    p.g = l.g;
    p.xh = xh, p.xl = xl;
    p.dyh = h->dact_hi + l.act_off, p.dyl = h->dact_lo + l.act_off, p.dystride = h->act_stride;
    p.ones = h->ones;
    p.gout = h->grad, p.gstride = h->stride, p.w_off = l.w_off;
    p.scale = scale;
    p.M = l.g.Kd + 1, p.K = h->B * l.g.OH * l.g.OW;
    p.NT = round16(l.g.OC);
    const int mt = (p.M + 127) / 128;
    p.S = splitk_for(mt * K, (p.K + 31) / 32, h->sm_count);
    const int it_per = ((p.K + 31) / 32 + p.S - 1) / p.S;
    p.kchunk = it_per * 32;
    p.S = (p.K + p.kchunk - 1) / p.kchunk;
    const int planes = xu ? 1 : 2;
    p.nstage = tcg::pick_stages(planes, p.NT, it_per);
    const int64_t part = p.S > 1 ? (int64_t)K * mt * p.S * p.NT * 128 : 0;
    const int tick = p.S > 1 ? K * mt : 0;
    if (dry) {
      *ws_part = std::max(*ws_part, part), *ws_tick = std::max(*ws_tick, tick);
      return IDQN_OK;
    }
    int rc = check_ws(h, part, tick, "tc wgrad", li);
    if (rc) return rc;
    dim3 grid(mt, 1, K * p.S);
    const bool halfu = l.g.IC == 4;
    if (planes == 1 && halfu) CK((tcg::launch_tc<true, true, 1, true, false, true>(p, grid, h->part, h->tickets, h->stream)));
    else if (planes == 1) CK((tcg::launch_tc<true, true, 1, false, false, true>(p, grid, h->part, h->tickets, h->stream)));
    else if (halfu) CK((tcg::launch_tc<true, true, 2, true, false, true>(p, grid, h->part, h->tickets, h->stream)));
    else CK((tcg::launch_tc<true, true, 2, false, false, true>(p, grid, h->part, h->tickets, h->stream)));
    mark(h, "tc_wgrad_L%d", li);
    return IDQN_OK;
  }
  WgradProb p;
  p.g = l.g;
  p.x = x;
  p.x_u8 = xu;
  p.dy = h->dact + l.act_off;
  p.dystride = h->act_stride;
  p.gout = h->grad;
  p.gstride = h->stride;
  p.w_off = l.w_off;
  p.scale = scale;
  p.relu_in = l.relu_in;
  p.nz = K;
  p.M = l.g.Kd + 1;
  p.N = l.g.OC;
  p.K = h->B * l.g.OH * l.g.OW;
  GemmPlan gp = plan_gemm(p.M, p.N, p.K, K, h->sm_count, true);
  p.S = gp.S;
  p.kchunk = gp.kchunk;
  if (dry) {
    *ws_part = std::max(*ws_part, gp.part_floats), *ws_tick = std::max(*ws_tick, gp.tickets);
    return IDQN_OK;
  }
  int rc = check_ws(h, gp.part_floats, gp.tickets, "wgrad", li);
  if (rc) return rc;
  CK((launch_gemm_simt<false, false>(p, K * p.S, h->part, h->tickets, h->stream)));
  mark(h, "wgrad_L%d", li);
  return IDQN_OK;
}

// ---- data gradient: writes dact of layer li-1 ------------------------------------------------------------------
static int launch_dgrad_layer(idqn_handle* h, int li, bool img_dst = false) {
  const Layer& l = h->layers[li];
  const Layer& prev = h->layers[li - 1];
  const int K = h->K;
  const int S = l.g.S;
  if (S * S > IDQN_MAX_CLASSES) {
    idqn_set_error("stride %d not supported in dgrad", S);
    return IDQN_EINVAL;
  }
  const NetPtr wh{h->won_hi, h->won_hi, h->stride, h->stride, K}, wl{h->won_lo, h->won_lo, h->stride, h->stride, K};
  // relu' of the input: it was the previous layer's relu output, or this layer applied the relu itself (impala blocks)
  const int mask = (l.relu_in || prev.relu_out) ? 1 : 0;
  const float* add = nullptr;
  for (int j = li + 1; j < h->n_layers; ++j)  // a later layer that adds this activation to its output (residual)
    if (h->layers[j].skip_from == li - 1) add = h->dact + h->layers[j].act_off;
  if (use_tc(h) && tc_dense_ok(h, l)) {
    REQUIRE(mask && !add, "internal: the dense data-gradient kernel always applies the relu mask");
    tcg::TcDgradDenseT p;
    p.dyh = h->dact_hi + l.act_off, p.dyl = h->dact_lo + l.act_off, p.dystride = h->act_stride;
    p.wh = wh, p.wl = wl;
    p.w_off = l.w_off;
    p.xact = h->act + prev.act_off, p.dx = h->dact + prev.act_off;
    p.dxh = h->dact_hi + prev.act_off, p.dxl = h->dact_lo + prev.act_off, p.xstride = h->act_stride;
    p.I = l.g.Kd, p.O = l.g.OC, p.B = h->B;
    p.zP = 0;
    if (img_dst) {  // the preceding layer is a conv of the image path: its dy planes live in the dyZ layout
      const img::Geom& pg = ((ImgHost*)h->img_host)->g[li - 1];
      p.dxh = h->il[li - 1].dz_hi, p.dxl = h->il[li - 1].dz_lo;
      p.zP = pg.P, p.zW = pg.OW, p.zC = pg.OC, p.zOff = pg.T - 1, p.zRows = pg.ZRa, p.zstride = h->il[li - 1].dz_net_stride;
    }
    p.NT = round16(h->B);
    p.nstage = tcg::pick_stages(2, p.NT, (p.O + 31) / 32);
    dim3 grid((p.I + 127) / 128, 1, K);
    CK((tcg::launch_tc<false, false, 2, false, true, false>(p, grid, h->part, h->tickets, h->stream)));
    mark(h, "tc_dgrad_L%d", li);
    return IDQN_OK;
  }
  int cls_niy[IDQN_MAX_CLASSES], cls_nix[IDQN_MAX_CLASSES], maxM = 0;
  for (int cl = 0; cl < S * S; ++cl) {
    const int py = cl / S, px = cl % S;
    cls_niy[cl] = std::max((l.g.IH - py + S - 1) / S, 0);
    cls_nix[cl] = std::max((l.g.IW - px + S - 1) / S, 0);
    maxM = std::max(maxM, h->B * cls_niy[cl] * cls_nix[cl]);
  }
  const int JH = (l.g.KH + S - 1) / S, JW = (l.g.KW + S - 1) / S;
  if (use_tc(h) && tc_conv_ok(l)) {
    tcg::TcDgradConv p;
    p.g = l.g;
    p.dyh = h->dact_hi + l.act_off, p.dyl = h->dact_lo + l.act_off, p.dystride = h->act_stride;
    p.wh = wh, p.wl = wl;
    p.w_off = l.w_off;
    p.xact = h->act + prev.act_off, p.dx = h->dact + prev.act_off;
    p.mask = mask, p.add = add;
    p.dxh = h->dact_hi + prev.act_off, p.dxl = h->dact_lo + prev.act_off, p.xstride = h->act_stride;
    p.ncls = S * S, p.JH = JH, p.JW = JW;
    p.d_jwoc = FastDiv(JW * l.g.OC);
    p.K = JH * JW * l.g.OC;
    p.NT = round16(l.g.IC);
    p.nstage = tcg::pick_stages(2, p.NT, (p.K + 31) / 32);
    for (int cl = 0; cl < p.ncls; ++cl) {
      p.cls_niy[cl] = cls_niy[cl], p.cls_nix[cl] = cls_nix[cl];
      p.cls_d_n[cl] = FastDiv(std::max(cls_niy[cl] * cls_nix[cl], 1));
      p.cls_d_nix[cl] = FastDiv(std::max(cls_nix[cl], 1));
    }
    dim3 grid((maxM + 127) / 128, 1, K * p.ncls);
    CK((tcg::launch_tc<false, false, 2, false, true, false>(p, grid, h->part, h->tickets, h->stream)));
    mark(h, "tc_dgrad_L%d", li);
    return IDQN_OK;
  }
  DgradProb p;
  p.g = l.g;
  p.dy = h->dact + l.act_off;
  p.dystride = h->act_stride;
  p.w = NetPtr{h->online, h->online, h->stride, h->stride, K};
  p.w_off = l.w_off;
  p.xact = h->act + prev.act_off;
  p.mask = mask, p.add = add;
  p.dx = h->dact + prev.act_off;
  p.dxh = h->dact_hi + prev.act_off, p.dxl = h->dact_lo + prev.act_off;
  p.xstride = h->act_stride;
  p.nz = K;
  p.S = 1;
  p.ncls = S * S;
  p.JH = JH, p.JW = JW;
  p.d_jwoc = FastDiv(JW * l.g.OC);
  p.N = l.g.IC;
  p.K = JH * JW * l.g.OC;
  p.kchunk = p.K;
  for (int cl = 0; cl < p.ncls; ++cl) {
    p.cls_niy[cl] = cls_niy[cl], p.cls_nix[cl] = cls_nix[cl];
    p.cls_d_n[cl] = FastDiv(std::max(cls_niy[cl] * cls_nix[cl], 1));
    p.cls_d_nix[cl] = FastDiv(std::max(cls_nix[cl], 1));
  }
  p.M = maxM;
  CK((launch_gemm_simt<true, true>(p, K * p.ncls, h->part, h->tickets, h->stream)));
  mark(h, "dgrad_L%d", li);
  return IDQN_OK;
}

// Adam over the arena ranges [off_a, off_a + len_a) and [off_b, off_b + len_b) of every head, one launch
// coresident: 128-thread CTAs (one 64-register warp per SM sub-partition) with the shared-memory carve-out of the big
// kernels, so that the launch runs NEXT to the persistent Dense_0 wgrad+Adam CTAs instead of after them
static int launch_adam_ranges(idqn_handle* h, int64_t off_a, int64_t len_a, bool a_from_partials, int64_t off_b,
                              int64_t len_b, bool coresident = false) {
  len_a = std::max<int64_t>(len_a, 0), len_b = std::max<int64_t>(len_b, 0);
  if (len_a + len_b <= 0) return IDQN_OK;
  const int64_t n4a = len_a / 4, n4b = len_b / 4;
  const int cap = h->sm_count * 8;
  const int bt = coresident ? 128 : 256;
  const int ba = n4a ? (int)std::min<int64_t>((n4a + bt - 1) / bt, cap) : 0;
  const int bb = n4b ? (int)std::min<int64_t>((n4b + bt - 1) / bt, cap) : 0;
  if (coresident) {
    static bool carve_set = false;
    if (!carve_set) {
      CK(cudaFuncSetAttribute(adam_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
      carve_set = true;
    }
  }
  dim3 grid(std::max(ba + bb, 1), h->K);
  const bool keep = (h->cfg.flags & IDQN_F_KEEP_GRADS) != 0;
  CK(launch_pdl(h->pdl && !coresident, adam_kernel, grid, dim3(bt), 0, h->stream, (float4*)h->online, (const float4*)h->grad, (float4*)h->mu, (float4*)h->nu,
                                           (uint2*)h->won_hi, (uint2*)h->won_lo, h->count, h->stride / 4, off_a / 4, n4a, ba,
                                           off_b / 4, n4b, h->cfg.learning_rate, 0.9f, 0.999f, h->cfg.adam_eps,
                                           a_from_partials ? (const float4*)h->wpart : nullptr, h->wgroups, h->wspan / 4,
                                           (a_from_partials && keep) ? (float4*)h->grad : nullptr, tl_next(h)));
  mark(h, "adam_%d", 0);
  return IDQN_OK;
}

// enqueue one whole learning step on h->stream (batch already staged in h->s/s2/action/reward/terminal);
static int dense_update_ctas(const idqn_handle* h) {
  static const int env = getenv("IDQN_WG_OVERLAP") ? atoi(getenv("IDQN_WG_OVERLAP")) : -1;
  if (h->update_ctas_set > 0) return std::min(h->sm_count, h->update_ctas_set - 1);
  return env >= 0 ? env : (h->K <= 10 ? std::min(h->sm_count, (116 + 13 * h->K) / 2 * h->sm_count / 148) : 0);
}

// dry = only size the split-K workspace
static int enqueue_learn_step(idqn_handle* h, int x_u8, bool dry = false, int64_t* ws_part = nullptr,
                              int* ws_tick = nullptr) {
  const int K = h->K, L = h->n_layers, B = h->B;
  h->n_launch = 0;
  // image-resident TMA conv kernels for the conv stack (uint8 frames); the generic kernels otherwise
  const bool use_img = h->img_on && x_u8 && !dry;
  const int n_img = use_img ? IDQN_IMG_LAYERS : 0;
  if (!dry) h->img_last = use_img;
  // bf16 planes of the staged batch (operand of the first layer's tensor-core kernels)
  const bool in_planes = use_tc(h) && (tc_conv_ok(h->layers[0]) || tc_dense_ok(h, h->layers[0]));
  if (use_img) {
    int rc = img_launch_s2d(h, x_u8);
    if (rc) return rc;
    // opt-in (IDQN_F_CHAIN): measured 49.5 us for the chain against 26 + 25 us for the two launches at K = 5 (0.3025 vs
    // 0.3005 ms per step) and 18.8 vs 19.5 us at K = 1: a (net, image) unit is then ONE serial MMA stream of both layers on
    // one SM (320 units on 107 CTAs at K = 5), whereas the two launches split every unit's M tiles over two CTAs
    const bool chain = ((ImgHost*)h->img_host)->chain_on && (h->cfg.flags & IDQN_F_CHAIN);
    for (int li = 0; li < n_img; ++li) {
      if (chain && li == 1) {
        rc = img_launch_chain_fwd(h);  // conv1 and conv2 of a (net, image) in one CTA, the intermediate image in shared memory
        li = 2;
      } else {
        rc = img_launch_taps(h, li, false, li == 0 ? 1 : 2);
      }
      if (rc) return rc;
    }
  } else if (in_planes && !dry) {
    int rc = launch_input_planes(h, x_u8, B, 1);
    if (rc) return rc;
  }
  // forward of 2K nets through all hidden layers
  const int64_t in_full = (int64_t)B * h->in_elems;
  const bool use_dense = h->img_on && !dry && ((ImgHost*)h->img_host)->dense_on;  // dense_stream.cuh for Dense_0
  for (int li = n_img; li < L - 1; ++li) {
    if (use_dense && li == IDQN_IMG_LAYERS) {
      int rc = dense_launch(h, false, false);
      if (rc) return rc;
      continue;
    }
    FwdIO io;
    int nh = 1;
    if (li == 0) {
      io.x = NetPtr{h->s, h->s2, 0, 0, K};
      io.xh = NetPtr{h->in_hi, h->in_hi + in_full, 0, 0, K};
      io.xl = NetPtr{h->in_lo, h->in_lo + in_full, 0, 0, K};
      nh = K;  // all online heads read s, all target heads read s': concatenate them along N
    } else {
      const int64_t o = h->layers[li - 1].act_off;
      io.x = NetPtr{h->act + o, h->act + o, h->act_stride, h->act_stride, 2 * K};
      io.xh = NetPtr{h->act_hi + o, h->act_hi + o, h->act_stride, h->act_stride, 2 * K};
      io.xl = NetPtr{h->act_lo + o, h->act_lo + o, h->act_stride, h->act_stride, 2 * K};
    }
    io.w = NetPtr{h->online, h->target, h->stride, h->stride, K};
    io.wh = NetPtr{h->won_hi, h->wtg_hi, h->stride, h->stride, K};
    io.wl = NetPtr{h->won_lo, h->wtg_lo, h->stride, h->stride, K};
    const int64_t o = h->layers[li].act_off;
    io.y = h->act + o, io.yh = h->act_hi + o, io.yl = h->act_lo + o, io.ystride = h->act_stride;
    if (h->layers[li].kind == IDQN_LAYER_POOL) {
      if (dry) continue;
      int rc = launch_pool_fwd(h, li, 2 * K, B, h->act + h->layers[li - 1].act_off, h->act + o, h->act_stride, true);
      if (rc) return rc;
      continue;
    }
    int rc = launch_fwd_layer(h, li, 2 * K, nh, B, io, li == 0 ? x_u8 : 0, h->layers[li].relu_out, dry, ws_part, ws_tick);
    if (rc) return rc;
  }
  // final layer + loss + its backward
  if (!dry) {
    const Layer& l = h->layers[L - 1];
    HeadArgs a;
    if (L >= 2) {
      const float* hid = h->act + h->layers[L - 2].act_off;
      a.hid = NetPtr{hid, hid, h->act_stride, h->act_stride, 2 * K};
      a.dhid = h->dact + h->layers[L - 2].act_off;
      a.dhid_hi = h->dact_hi + h->layers[L - 2].act_off, a.dhid_lo = h->dact_lo + h->layers[L - 2].act_off;
      a.relu_mask = 1;
    } else {
      REQUIRE(!x_u8, "a network without hidden layers needs float32 inputs");
      a.hid = NetPtr{h->s, h->s2, 0, 0, K};
      a.dhid = nullptr;
      a.dhid_hi = a.dhid_lo = nullptr;
      a.relu_mask = 0;
    }
    a.H = l.g.Kd, a.A = h->A, a.B = B, a.K = K;
    a.online = h->online, a.target = h->target;
    a.stride = h->stride, a.w_off = l.w_off, a.b_off = l.b_off;
    a.action = h->action, a.reward = h->reward, a.terminal = h->terminal;
    a.gamma_n = h->cfg.gamma_n;
    a.grad = h->grad;
    a.dstride = h->act_stride;
    a.loss = h->loss, a.loss_sum = h->loss_sum, a.count = h->count;
    a.loss_acc_on = h->loss_acc_on;
    a.td_abs = h->td_abs;
    a.q = h->q;
    a.part = nullptr, a.ptiles = a.psplits = 0, a.pb_off = 0;
    a.cta0 = 0;
    a.tl_id = tl_next(h);
    if (use_dense && L - 2 == IDQN_IMG_LAYERS) {
      const dense::Args& df = ((ImgHost*)h->img_host)->dfwd;
      if (df.splits > 1) a.part = df.part, a.ptiles = df.tiles, a.psplits = df.splits, a.pb_off = h->layers[L - 2].b_off;
    }
    CK(launch_pdl(h->pdl, head_q_kernel, dim3(2 * K * B), dim3(128), 0, h->stream, a));
    mark(h, "head_q_L%d", L - 1);
    a.hbias_off = -1;
    a.tl_id = tl_next(h);
    if (L >= 2 && dense_wgrad_tma_ok(h, L - 2)) a.hbias_off = h->layers[L - 2].b_off;
    const size_t smem = (size_t)(3 * B + 32 * B + 32 * a.A + 32 * B) * sizeof(float);
    REQUIRE(smem <= IMG_SMEM_OPTIN, "head_bwd_kernel needs %zu bytes of shared memory (batch %d, %d actions)", smem, B, a.A);
    if (smem > 48 * 1024) CK(cudaFuncSetAttribute(head_bwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)IMG_SMEM_OPTIN));
    CK(launch_pdl(h->pdl, head_bwd_kernel, dim3((a.H + 31) / 32, K), dim3(256), smem, h->stream, a));
    mark(h, "head_bwd_L%d", L - 1);
  }
  // backward through the hidden layers
  int64_t fused_lo = -1, fused_hi = -1;  // arena range whose Adam update was fused into a wgrad epilogue
  smpart::Partition* part = (smpart::Partition*)h->partition;
  const bool split = part && use_img && n_img == L - 2 && !h->prof_on && !dry && use_dense;
  const bool fork_conv = n_img > 0 && !split && !h->prof_on && !dry && !(h->cfg.flags & IDQN_F_NO_FORK);
  // With the two-branch graph the HBM-bound Dense_0 wgrad+Adam (TMA pipeline, one persistent CTA per SM) is deferred to
  // the END of the backward pass: the conv chain (main: dgrads, side: wgrads) runs first, then the final Adam launch
  // -- small CTAs that fit next to the persistent ones -- hides under the 97 us of the HBM kernel.
  int deferred_li = -1;
  bool overlapped = false;
  int deferred_t0 = 0;
  static const float overlap_frac = getenv("IDQN_WG_FRAC") ? (float)atof(getenv("IDQN_WG_FRAC")) : 1.0f;
  // CTAs of the Dense_0 update when it runs next to the conv backward chain instead of after it (0: after): 58 + 6.5 K.
  // Measured on B200 (tools/r2l.sh / r2n.sh, ms per step, update after the chain -> next to it): K=1 0.122 -> 0.112 at
  // 64-80 CTAs, K=3 0.208 -> 0.197 at 72-80, K=5 0.295 -> 0.274 at 88, K=8 0.417 -> 0.394 at 88-112; fewer CTAs starve the
  // update (~52 GB/s per SM), more starve the chain.  IDQN_WG_OVERLAP=<n> overrides, 0 restores the back-to-back order.
  const int overlap_ctas = dense_update_ctas(h);
  // idqn_profile_step times the kernels one by one on one stream: same grids as in the graph, so that its per-kernel times
  // (bench.py: kernel_ms, roofline) describe the launches the timed step makes
  const bool same_grids = h->prof_on && overlap_ctas > 0 && use_img && use_dense && n_img == L - 2 && !(h->cfg.flags & (IDQN_F_NO_FORK | IDQN_F_NO_DEFER));
  for (int li = L - 2; li >= 0; --li) {
    // the dgrad of this layer reads the weights the fused wgrad+Adam kernel overwrites: dgrad first
    if (li < n_img) {
      // dyZ of this layer is complete at this point of the main stream: its weight gradient goes to the side branch
      // and runs next to the data-gradient chain (both are one-CTA-per-SM kernels with 25-30% of the SMs idle in
      // their last wave; as independent graph branches they fill each other's tails)
      if (fork_conv) {
        CK(cudaEventRecord(h->ev_conv[li], h->stream));
        CK(cudaStreamWaitEvent(h->side, h->ev_conv[li], 0));
      }
      // next to the Dense_0 update the data-gradient kernels are persistent over the SMs it leaves (they would otherwise sit on
      // all of them, waiting, when it becomes ready)
      static const int bwd_sms_env = getenv("IDQN_CONV_BWD_SMS") ? atoi(getenv("IDQN_CONV_BWD_SMS")) : -1;
      const int sm_all = h->sm_avail;
      if (overlapped || same_grids) h->sm_avail = std::max(8, std::min(sm_all, bwd_sms_env > 0 ? bwd_sms_env : (bwd_sms_env == 0 ? sm_all : sm_all - overlap_ctas)));
      int rc = li > 0 ? img_launch_taps(h, li, true, 2) : IDQN_OK;
      h->sm_avail = sm_all;
      if (rc) return rc;
      cudaStream_t main_stream = h->stream;
      // conv0's weight gradient stays on the main stream (unless IDQN_WGRAD0_SIDE): it depends on conv1's data gradient only, and
      // as the side branch's third kernel it would also wait for conv1's weight gradient
      static const bool wgrad0_side = getenv("IDQN_WGRAD0_SIDE") != nullptr;
      if (fork_conv && (li > 0 || wgrad0_side)) h->stream = h->side;
      rc = img_launch_wgrad(h, li, li == 0 ? 1 : 2);
      h->stream = main_stream;
      if (rc) return rc;
      if (fork_conv && li == 0) {
        CK(cudaEventRecord(h->ev_side_done, h->side));
        CK(cudaStreamWaitEvent(h->stream, h->ev_side_done, 0));
        if (deferred_li >= 0) {
          // main: the HBM kernel (after the last conv weight gradient, so it does not take the SMs from it);
          // side: the final Adam next to it; join
          if (!wgrad0_side) {  // the final Adam (side) also reads conv0's partial gradients, computed on the main stream
            CK(cudaEventRecord(h->ev_fork, h->stream));
            CK(cudaStreamWaitEvent(h->side, h->ev_fork, 0));
          }
          if (deferred_t0 > 0) h->wg_tile0 = deferred_t0, h->wg_tiles = h->layers[deferred_li].g.Kd / dwt::TM - deferred_t0;
          rc = launch_wgrad_layer(h, deferred_li, x_u8, dry, ws_part, ws_tick);
          h->wg_tile0 = h->wg_tiles = 0;
          if (rc) return rc;
          h->stream = h->side;
          const int64_t hi = (fused_hi + 3) / 4 * 4;
          rc = launch_adam_ranges(h, 0, fused_lo, fused_lo == h->wspan, hi, h->stride - hi, true);
          h->stream = main_stream;
          if (rc) return rc;
          CK(cudaEventRecord(h->ev_join[0], h->side));
          CK(cudaStreamWaitEvent(h->stream, h->ev_join[0], 0));
          if (overlapped) CK(cudaStreamWaitEvent(h->stream, h->ev_join[1], 0));
          return IDQN_OK;
        }
      }
      continue;
    }
    if (h->layers[li].kind == IDQN_LAYER_POOL) {  // no parameters: only the data gradient
      if (!dry) {
        int rc = launch_pool_bwd(h, li);
        if (rc) return rc;
      }
      continue;
    }
    if (li > 0 && !dry) {
      int rc = (use_dense && li == IDQN_IMG_LAYERS) ? dense_launch(h, true, n_img > 0)
                                                   : launch_dgrad_layer(h, li, li == n_img && n_img > 0);
      if (rc) return rc;
    }
    const bool fused = use_tc(h) && tc_dense_ok(h, h->layers[li]);
    if (fused) {
      REQUIRE(fused_lo < 0, "internal: at most one fused wgrad+Adam layer is supported");
      fused_lo = h->layers[li].w_off;
      fused_hi = h->layers[li].b_off + (dense_wgrad_tma_ok(h, li) ? 0 : h->layers[li].g.OC);  // the TMA kernel leaves the bias to Adam
    }
    if (fused && split) {
      // Two SM partitions (sm_partition.cuh): the conv backward chain below this layer on part->stream[0], the first
      // part_frac of this layer's HBM-bound wgrad+Adam tiles on part->stream[1]; the rest of the tiles run on the
      // whole machine after the join.
      cudaStream_t main_stream = h->stream;
      const int mt = dense_wgrad_tma_ok(h, li) ? h->layers[li].g.Kd / dwt::TM : (h->layers[li].g.Kd + 1 + 127) / 128;
      const int t1 = std::min(mt, std::max(0, (int)(mt * h->part_frac + 0.5f)));
      CK(cudaEventRecord(h->ev_fork, main_stream));
      CK(cudaStreamWaitEvent(part->stream[0], h->ev_fork, 0));
      CK(cudaStreamWaitEvent(part->stream[1], h->ev_fork, 0));
      int rc = IDQN_OK;
      h->stream = part->stream[1], h->sm_avail = part->sms[1];
      h->wg_tile0 = 0, h->wg_tiles = t1;
      if (t1 > 0) rc = launch_wgrad_layer(h, li, x_u8, dry, ws_part, ws_tick);
      h->stream = part->stream[0], h->sm_avail = part->sms[0];
      for (int lj = li - 1; lj >= 0 && !rc; --lj) {
        if (lj > 0) rc = img_launch_taps(h, lj, true, 2);
        if (!rc) rc = img_launch_wgrad(h, lj, lj == 0 ? 1 : 2);
      }
      h->stream = main_stream, h->sm_avail = h->sm_count;
      if (rc) return rc;
      CK(cudaEventRecord(h->ev_join[0], part->stream[0]));
      CK(cudaEventRecord(h->ev_join[1], part->stream[1]));
      CK(cudaStreamWaitEvent(main_stream, h->ev_join[0], 0));
      CK(cudaStreamWaitEvent(main_stream, h->ev_join[1], 0));
      h->wg_tile0 = t1, h->wg_tiles = mt - t1;
      if (mt - t1 > 0) rc = launch_wgrad_layer(h, li, x_u8, dry, ws_part, ws_tick);
      h->wg_tile0 = h->wg_tiles = 0;
      if (rc) return rc;
      break;
    }
    if (fused && fork_conv && li == n_img && dense_wgrad_tma_ok(h, li) && !(h->cfg.flags & IDQN_F_NO_DEFER)) {
      if (overlap_ctas > 0) {
        // few heads: the conv backward kernels leave SMs idle, so the HBM-bound update runs NEXT TO them on a third
        // branch, on overlap_ctas persistent CTAs (it must follow the data gradient, which reads the weights it rewrites)
        CK(cudaEventRecord(h->ev_fork2, h->stream));
        CK(cudaStreamWaitEvent(h->side2, h->ev_fork2, 0));
        cudaStream_t main_stream = h->stream;
        const int sm = h->sm_avail;
        h->stream = h->side2, h->sm_avail = std::min(sm, overlap_ctas);
        const int mt = h->layers[li].g.Kd / dwt::TM;
        const int t1 = std::max(1, std::min(mt, (int)(mt * overlap_frac + 0.5f)));
        h->wg_tile0 = 0, h->wg_tiles = t1;
        int rc = launch_wgrad_layer(h, li, x_u8, dry, ws_part, ws_tick);
        h->stream = main_stream, h->sm_avail = sm;
        h->wg_tile0 = h->wg_tiles = 0;
        if (rc) return rc;
        CK(cudaEventRecord(h->ev_join[1], h->side2));
        overlapped = true;
        if (t1 < mt) deferred_li = li, deferred_t0 = t1;  // the rest of the tiles after the chain, on the whole machine
        continue;
      }
      deferred_li = li;
      continue;
    }
    const int sm_all = h->sm_avail;
    if (same_grids && fused && li == n_img && dense_wgrad_tma_ok(h, li)) h->sm_avail = std::min(sm_all, overlap_ctas);
    int rc = launch_wgrad_layer(h, li, x_u8, dry, ws_part, ws_tick);
    h->sm_avail = sm_all;
    if (rc) return rc;
  }
  if (dry) return IDQN_OK;
  // Adam over the rest of the arena of every head
  if (fused_lo < 0) return launch_adam_ranges(h, 0, h->stride, false, 0, 0);
  const int64_t hi = (fused_hi + 3) / 4 * 4;  // layer starts are 128-byte aligned, so this stays inside the gap
  int rc = launch_adam_ranges(h, 0, fused_lo, use_img && fused_lo == h->wspan, hi, h->stride - hi);
  if (!rc && overlapped) CK(cudaStreamWaitEvent(h->stream, h->ev_join[1], 0));
  return rc;
}

int idqn_learn_step_resident(idqn_handle* h, int x_u8, float* losses_host) {
  x_u8 = x_u8 ? 1 : 0;
  {
    int rc = refresh_planes(h);
    if (rc) return rc;
  }
  h->dense0_valid[0] = 0;  // the step rewrites the big Dense layer's fp32 master only
  if (h->cfg.flags & IDQN_F_NO_GRAPH) {
    int rc = enqueue_learn_step(h, x_u8);
    if (rc) return rc;
  } else {
    cudaGraphExec_t& gexec = h->graph[2 * h->graph_set + x_u8];
    if (!gexec) {
      cudaGraph_t g;
      CK(cudaStreamBeginCapture(h->stream, cudaStreamCaptureModeThreadLocal));
      int rc = enqueue_learn_step(h, x_u8);
      cudaError_t e = cudaStreamEndCapture(h->stream, &g);
      if (rc) {
        if (e == cudaSuccess && g) cudaGraphDestroy(g);  // a failed enqueue must not leak the partial capture
        return rc;
      }
      CK(e);
      CK(cudaGraphInstantiate(&gexec, g, 0));
      CK(cudaGraphDestroy(g));
    }
    CK(cudaGraphLaunch(gexec, h->stream));
  }
  if (losses_host) {
    CK(cudaMemcpyAsync(h->h_loss, h->loss, sizeof(float) * h->K, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    memcpy(losses_host, h->h_loss, sizeof(float) * h->K);
  }
  return IDQN_OK;
}

extern "C" int idqn_kernels_per_step(idqn_handle* h) {
  return h ? h->n_launch : 0;  // launches enqueued by the most recent step capture / profile
}

extern "C" int idqn_profile_step(idqn_handle* h, int x_u8, int max_entries, float* ms, char* names, int* n_out) {
  REQUIRE(h && ms && names && n_out, "null argument");
  CK(cudaSetDevice(h->cfg.device));
  for (int i = 0; i <= IDQN_PROF_MAX; ++i)
    if (!h->prof_ev[i]) CK(cudaEventCreate(&h->prof_ev[i]));
  {
    int rc = refresh_planes(h);
    if (rc) return rc;
  }
  h->prof_on = 1, h->prof_n = 0;
  h->dense0_valid[0] = 0;
  CK(cudaEventRecord(h->prof_ev[0], h->stream));
  int rc = enqueue_learn_step(h, x_u8 ? 1 : 0);
  h->prof_on = 0;
  if (rc) return rc;
  CK(cudaStreamSynchronize(h->stream));
  int n = std::min(h->prof_n, max_entries);
  for (int i = 0; i < n; ++i) {
    CK(cudaEventElapsedTime(&ms[i], h->prof_ev[i], h->prof_ev[i + 1]));
    memcpy(names + 32 * i, h->prof_name[i], 32);
  }
  *n_out = n;
  return IDQN_OK;
}

// ------------------------------------------------------------------------------------------
// C ABI
extern "C" int idqn_create(const idqn_config* cfg, idqn_handle** out) {
  REQUIRE(cfg && out, "null argument");
  REQUIRE(cfg->n_heads >= 1 && cfg->batch_size >= 1 && cfg->n_actions >= 1, "bad sizes");
  REQUIRE(cfg->n_features >= 0 && cfg->n_features <= IDQN_MAX_FEATURES, "bad n_features");
  REQUIRE(cfg->n_actions <= HEAD_MAXA, "n_actions = %d: the fused final-layer kernels hold at most %d actions", cfg->n_actions, HEAD_MAXA);
  idqn_handle* h = new idqn_handle();
  memset(h, 0, sizeof(*h));
  h->cfg = *cfg;
  // impala runs on the generic kernels, layer by layer: tcgen05 implicit GEMM (gemm_tc.cuh) where the channel counts allow
  // vector loads, the fp32 CUDA-core problems (gemm_simt.cuh) elsewhere (first conv: 4 channels x 3 taps; 1..7-channel test
  // nets), plus the pool kernels.  IDQN_IMPALA_SIMT=1 keeps everything on the CUDA cores.
  if (cfg->arch == IDQN_ARCH_IMPALA && getenv("IDQN_IMPALA_SIMT")) h->cfg.flags |= IDQN_F_SIMT_ONLY;
  h->K = cfg->n_heads, h->B = cfg->batch_size, h->A = cfg->n_actions;
  int rc = build_layers(h);
  if (rc) {
    delete h;
    return rc;
  }
  CK(cudaSetDevice(cfg->device));
  cudaDeviceProp prop;
  CK(cudaGetDeviceProperties(&prop, cfg->device));
  REQUIRE(prop.major == 10, "libidqn_b200 is built for sm_100a only (device is sm_%d%d)", prop.major, prop.minor);
  h->sm_count = prop.multiProcessorCount;
  {
    // the learner's stream carries the critical chain of the step (forward, data gradients, the HBM-bound update); the side
    // branch of the step graph (conv weight gradients) gets the LOWEST priority so that its CTAs only fill SMs the chain
    // leaves idle (kernel nodes captured from a stream inherit its priority)
    int lo = 0, hi = 0;
    CK(cudaDeviceGetStreamPriorityRange(&lo, &hi));
    const bool prio = !getenv("IDQN_NO_PRIORITY");
    CK(cudaStreamCreateWithPriority(&h->stream, cudaStreamNonBlocking, prio ? hi : 0));
    CK(cudaStreamCreateWithPriority(&h->side, cudaStreamNonBlocking, prio ? lo : 0));
    CK(cudaStreamCreateWithPriority(&h->side2, cudaStreamNonBlocking, prio ? lo : 0));
  }
  h->sm_avail = h->sm_count;
  CK(cudaEventCreateWithFlags(&h->ev_fork, cudaEventDisableTiming));
  CK(cudaEventCreateWithFlags(&h->ev_fork2, cudaEventDisableTiming));
  CK(cudaEventCreateWithFlags(&h->ev_join[0], cudaEventDisableTiming));
  CK(cudaEventCreateWithFlags(&h->ev_join[1], cudaEventDisableTiming));
  CK(cudaEventCreateWithFlags(&h->ev_side_done, cudaEventDisableTiming));
  for (int i = 0; i < IDQN_IMG_LAYERS; ++i) CK(cudaEventCreateWithFlags(&h->ev_conv[i], cudaEventDisableTiming));
  if ((cfg->flags & IDQN_F_PARTITION) && !(cfg->flags & (IDQN_F_SIMT_ONLY | IDQN_F_NO_IMG)) && cfg->arch == IDQN_ARCH_CNN) {
    // conv chain on 112 of the 148 SMs (its grids are <= 110 CTAs at K = 5), the HBM stream on the other 36
    const char* e_sms = getenv("IDQN_PART_SMS");
    const char* e_frac = getenv("IDQN_PART_FRAC");
    const int conv_sms = e_sms ? atoi(e_sms) : (h->sm_count * 3 / 4 + 7) / 8 * 8;
    h->part_frac = e_frac ? (float)atof(e_frac) : 0.6f;
    smpart::Partition* P = new smpart::Partition();
    if (smpart::create(cfg->device, conv_sms, P)) h->partition = P;
    else {
      smpart::destroy(P);
      delete P;
    }
  }
  const int K = h->K, B = h->B;
  const size_t arena = sizeof(float) * h->stride * K;
  float** arenas[5] = {&h->online, &h->target, &h->mu, &h->nu, &h->grad};
  for (auto a : arenas) {
    CK(cudaMalloc(a, arena));
    CK(cudaMemsetAsync(*a, 0, arena, h->stream));
  }
  CK(cudaMalloc(&h->count, sizeof(int32_t) * K));
  CK(cudaMemsetAsync(h->count, 0, sizeof(int32_t) * K, h->stream));
  CK(cudaMalloc(&h->loss, sizeof(float) * K));
  CK(cudaMemsetAsync(h->loss, 0, sizeof(float) * K, h->stream));
  CK(cudaMalloc(&h->loss_sum, sizeof(double) * K));
  CK(cudaMemsetAsync(h->loss_sum, 0, sizeof(double) * K, h->stream));
  CK(cudaMalloc(&h->td_abs, sizeof(float) * K * B));
  CK(cudaMemsetAsync(h->td_abs, 0, sizeof(float) * K * B, h->stream));
  CK(cudaEventCreateWithFlags(&h->ev_step, cudaEventDisableTiming));
  CK(cudaMalloc(&h->loss_acc_on, sizeof(int32_t)));
  CK(cudaMemsetAsync(h->loss_acc_on, 0, sizeof(int32_t), h->stream));
  CK(cudaMemsetAsync(h->loss_acc_on, 1, 1, h->stream));  // little-endian int32 1
  h->loss_acc_host = 1;
  CK(cudaMalloc(&h->s, sizeof(float) * h->in_elems * B));
  CK(cudaMalloc(&h->s2, sizeof(float) * h->in_elems * B));
  CK(cudaMalloc(&h->action, sizeof(int32_t) * B));
  CK(cudaMalloc(&h->reward, sizeof(float) * B));
  CK(cudaMalloc(&h->terminal, B));
  CK(cudaMalloc(&h->act, sizeof(float) * h->act_stride * 2 * K));
  CK(cudaMalloc(&h->dact, sizeof(float) * h->act_stride * K));
  CK(cudaMemsetAsync(h->dact, 0, sizeof(float) * h->act_stride * K, h->stream));
  CK(cudaMalloc(&h->q, sizeof(float) * 2 * K * B * h->A));
  {  // bf16 hi/lo planes
    const size_t wp = sizeof(__nv_bfloat16) * h->stride * K;
    __nv_bfloat16** wps[2] = {&h->wpl_hi, &h->wpl_lo};  // [2K][stride]: online heads, then target heads
    for (auto pp : wps) {
      CK(cudaMalloc(pp, 2 * wp));
      CK(cudaMemsetAsync(*pp, 0, 2 * wp, h->stream));
    }
    h->won_hi = h->wpl_hi, h->wtg_hi = h->wpl_hi + h->stride * K;
    h->won_lo = h->wpl_lo, h->wtg_lo = h->wpl_lo + h->stride * K;
    const size_t ap = sizeof(__nv_bfloat16) * h->act_stride;
    CK(cudaMalloc(&h->act_hi, ap * 2 * K));
    CK(cudaMalloc(&h->act_lo, ap * 2 * K));
    CK(cudaMalloc(&h->dact_hi, ap * K));
    CK(cudaMalloc(&h->dact_lo, ap * K));
    CK(cudaMemsetAsync(h->act_hi, 0, ap * 2 * K, h->stream));
    CK(cudaMemsetAsync(h->act_lo, 0, ap * 2 * K, h->stream));
    CK(cudaMemsetAsync(h->dact_hi, 0, ap * K, h->stream));
    CK(cudaMemsetAsync(h->dact_lo, 0, ap * K, h->stream));
    const size_t ip = sizeof(__nv_bfloat16) * h->in_elems * B * 2;
    CK(cudaMalloc(&h->in_hi, ip));
    CK(cudaMalloc(&h->in_lo, ip));
    CK(cudaMemsetAsync(h->in_hi, 0, ip, h->stream));
    CK(cudaMemsetAsync(h->in_lo, 0, ip, h->stream));
    if (cfg->arch == IDQN_ARCH_IMPALA && !getenv("IDQN_POOL_RESCAN")) {
      CK(cudaMalloc(&h->pool_arg, (size_t)h->act_stride * K));
      CK(cudaMemsetAsync(h->pool_arg, 0, (size_t)h->act_stride * K, h->stream));
    }
    CK(cudaMalloc(&h->ones, sizeof(__nv_bfloat16) * 16));
    CK(cudaMemsetAsync(h->ones, 0, sizeof(__nv_bfloat16) * 16, h->stream));
    const uint16_t one_bits = 0x3F80;  // bf16(1.0)
    CK(cudaMemcpyAsync(h->ones, &one_bits, 2, cudaMemcpyHostToDevice, h->stream));
    h->planes_dirty[0] = h->planes_dirty[1] = 0;  // all-zero weights have all-zero planes
  }
  h->pdl = (cfg->flags & IDQN_F_NO_PDL) ? 0 : 1;  // measured: 0.353 ms/step with PDL vs 0.358 without (B200, K=5)
  rc = img_setup(h);
  if (rc) return rc;
  // split-K workspace: maximum over every launch the step (and a stand-alone apply) will make
  int64_t part = 0;
  int tickets = 0;
  rc = enqueue_learn_step(h, 0, true, &part, &tickets);
  if (rc) return rc;
  {
    FwdIO nul;
    memset(&nul, 0, sizeof(nul));
    for (int li = 0; li < h->n_layers; ++li) {
      if (h->layers[li].kind == IDQN_LAYER_POOL) continue;
      rc = launch_fwd_layer(h, li, 1, 1, B, nul, 0, 0, true, &part, &tickets);
      if (rc) return rc;
    }
  }
  h->part_floats = std::max<int64_t>(part, 1);
  h->n_tickets = std::max(tickets, 1);
  CK(cudaMalloc(&h->part, sizeof(float) * h->part_floats));
  CK(cudaMalloc(&h->tickets, sizeof(int) * h->n_tickets));
  CK(cudaMemsetAsync(h->tickets, 0, sizeof(int) * h->n_tickets, h->stream));
  CK(cudaMallocHost(&h->h_loss, sizeof(float) * std::max(K, B * h->A)));
  CK(cudaMallocHost(&h->h_i32, sizeof(int32_t) * std::max(K, 4)));
  CK(cudaMalloc(&h->best_idx, sizeof(int32_t) * 4));
  h->act_graph = new cudaGraphExec_t[K]();
  CK(cudaMallocHost(&h->h_state, (size_t)h->in_elems * 4));
  if (cfg->flags & IDQN_F_TIMELINE) {
    unsigned long long buf[2 * IDQN_KTL_MAX];
    for (int i = 0; i < IDQN_KTL_MAX; ++i) buf[2 * i] = ~0ull, buf[2 * i + 1] = 0;
    CK(cudaMemcpyToSymbol(g_ktl, buf, sizeof(buf)));
  }
  CK(cudaStreamSynchronize(h->stream));
  *out = h;
  return IDQN_OK;
}

extern "C" int idqn_destroy(idqn_handle* h) {
  if (!h) return IDQN_OK;
  cudaSetDevice(h->cfg.device);
  cudaStreamSynchronize(h->stream);
  for (int i = 0; i < 8; ++i)
    if (h->graph[i]) cudaGraphExecDestroy(h->graph[i]);
  for (int i = 0; i <= IDQN_PROF_MAX; ++i)
    if (h->prof_ev[i]) cudaEventDestroy(h->prof_ev[i]);
  if (h->loss_acc_on) cudaFree(h->loss_acc_on);
  if (h->td_abs) cudaFree(h->td_abs);
  if (h->ev_step) cudaEventDestroy(h->ev_step);
  void* ptrs[] = {h->online, h->target, h->mu,     h->nu,  h->grad, h->count, h->loss, h->loss_sum, h->s,
                  h->s2,     h->action, h->reward, h->terminal, h->act,  h->dact,  h->q,    h->part,     h->tickets};
  for (void* p : ptrs)
    if (p) cudaFree(p);
  void* planes[] = {h->wpl_hi, h->wpl_lo, h->act_hi, h->act_lo, h->dact_hi, h->dact_lo, h->in_hi, h->in_lo, h->ones, h->pool_arg};
  img_free(h);
  for (void* p : planes)
    if (p) cudaFree(p);
  if (h->h_loss) cudaFreeHost(h->h_loss);
  if (h->h_i32) cudaFreeHost(h->h_i32);
  if (h->best_idx) cudaFree(h->best_idx);
  if (h->act_graph) {
    for (int k = 0; k < h->K; ++k)
      if (h->act_graph[k]) cudaGraphExecDestroy(h->act_graph[k]);
    delete[] h->act_graph;
  }
  if (h->h_state) cudaFreeHost(h->h_state);
  for (int i = 0; i < 8; ++i) {
    if (h->vact_exec[i]) cudaGraphExecDestroy(h->vact_exec[i]);
    if (h->vact_graph[i]) cudaGraphDestroy(h->vact_graph[i]);
  }
  if (h->h_vact) cudaFreeHost(h->h_vact);
  if (h->h_vout) cudaFreeHost(h->h_vout);
  if (h->d_vact) cudaFree(h->d_vact);
  if (h->d_vout) cudaFree(h->d_vout);
  if (h->ev_fork) cudaEventDestroy(h->ev_fork);
  for (int i = 0; i < 2; ++i)
    if (h->ev_join[i]) cudaEventDestroy(h->ev_join[i]);
  if (h->copy_stream) {
    for (int i = 0; i < 2; ++i) {
      void* ptrs[] = {h->alt_s[i], h->alt_s2[i], h->alt_action[i], h->alt_reward[i], h->alt_terminal[i]};
      for (void* q : ptrs)
        if (q) cudaFree(q);
      cudaEventDestroy(h->ev_h2d[i]), cudaEventDestroy(h->ev_consumed[i]), cudaEventDestroy(h->ev_done[i]);
    }
    if (h->h_loss_ring) cudaFreeHost(h->h_loss_ring);
    cudaStreamDestroy(h->copy_stream);
  }
  if (h->ev_side_done) cudaEventDestroy(h->ev_side_done);
  for (int i = 0; i < IDQN_IMG_LAYERS; ++i)
    if (h->ev_conv[i]) cudaEventDestroy(h->ev_conv[i]);
  if (h->side) cudaStreamDestroy(h->side);
  if (h->side2) cudaStreamDestroy(h->side2);
  if (h->ev_fork2) cudaEventDestroy(h->ev_fork2);
  if (h->partition) {
    smpart::destroy((smpart::Partition*)h->partition);
    delete (smpart::Partition*)h->partition;
  }
  cudaStreamDestroy(h->stream);
  delete h;
  return IDQN_OK;
}

extern "C" int64_t idqn_arena_stride(const idqn_handle* h) { return h ? h->stride : 0; }
extern "C" int idqn_leaf_count(const idqn_handle* h) { return h ? 2 * h->n_param_layers : 0; }
extern "C" int idqn_leaf_info(const idqn_handle* h, int leaf, int64_t* offset, int64_t* size, int32_t shape[4],
                              int32_t* ndim, char name[16]) {
  REQUIRE(h && leaf >= 0 && leaf < 2 * h->n_param_layers, "bad leaf index");
  const Layer& l = h->layers[h->param_layer[leaf / 2]];
  if (leaf % 2 == 0) {
    *offset = l.w_off;
    *size = (int64_t)l.g.Kd * l.g.OC;
    if (l.is_conv) {
      shape[0] = l.g.KH, shape[1] = l.g.KW, shape[2] = l.g.IC, shape[3] = l.g.OC;
      *ndim = 4;
    } else {
      shape[0] = l.g.Kd, shape[1] = l.g.OC, shape[2] = shape[3] = 0;
      *ndim = 2;
    }
  } else {
    *offset = l.b_off;
    *size = l.g.OC;
    shape[0] = l.g.OC, shape[1] = shape[2] = shape[3] = 0;
    *ndim = 1;
  }
  memcpy(name, l.name, 16);
  return IDQN_OK;
}

static float* arena_of(idqn_handle* h, int which) {
  switch (which) {
    case IDQN_ONLINE: return h->online;
    case IDQN_TARGET: return h->target;
    case IDQN_MU: return h->mu;
    case IDQN_NU: return h->nu;
    case IDQN_GRAD: return h->grad;
  }
  return nullptr;
}

extern "C" void* idqn_arena_ptr(idqn_handle* h, int which) { return h ? arena_of(h, which) : nullptr; }
extern "C" void* idqn_stream(idqn_handle* h) { return h ? (void*)h->stream : nullptr; }

extern "C" int idqn_upload(idqn_handle* h, int which, int head, int64_t offset, const float* src, int64_t n) {
  float* a = h ? arena_of(h, which) : nullptr;
  REQUIRE(a && which != IDQN_GRAD, "bad arena");
  REQUIRE(head >= 0 && head < h->K && offset >= 0 && n >= 0 && offset + n <= h->stride, "range outside the arena");
  CK(cudaSetDevice(h->cfg.device));
  CK(cudaMemcpyAsync(a + (int64_t)head * h->stride + offset, src, sizeof(float) * n, cudaMemcpyHostToDevice,
                     h->stream));
  CK(cudaStreamSynchronize(h->stream));
  if (which == IDQN_ONLINE) h->planes_dirty[0] |= head < 63 ? 1ull << head : 1ull << 63;
  if (which == IDQN_TARGET) h->planes_dirty[1] |= head < 63 ? 1ull << head : 1ull << 63;
  return IDQN_OK;
}
extern "C" int idqn_download(idqn_handle* h, int which, int head, int64_t offset, float* dst, int64_t n) {
  float* a = h ? arena_of(h, which) : nullptr;
  REQUIRE(a, "bad arena");
  REQUIRE(head >= 0 && head < h->K && offset >= 0 && n >= 0 && offset + n <= h->stride, "range outside the arena");
  CK(cudaSetDevice(h->cfg.device));
  CK(cudaMemcpyAsync(dst, a + (int64_t)head * h->stride + offset, sizeof(float) * n, cudaMemcpyDeviceToHost,
                     h->stream));
  CK(cudaStreamSynchronize(h->stream));
  return IDQN_OK;
}
extern "C" int idqn_download_activation(idqn_handle* h, int net, int layer, float* dst, int64_t n) {
  REQUIRE(h && dst, "null argument");
  REQUIRE(net >= 0 && net < 2 * h->K && layer >= 0 && layer < h->n_layers - 1, "bad net/layer");
  REQUIRE(n >= 0 && n <= h->layers[layer].act_size, "too many elements");
  CK(cudaSetDevice(h->cfg.device));
  if (h->img_on && h->img_last && layer < IDQN_IMG_LAYERS) {  // the image path keeps conv activations as planes
    REQUIRE(!(layer == 1 && net >= h->K && ((ImgHost*)h->img_host)->chain_on && (h->cfg.flags & IDQN_F_CHAIN)),
            "the conv1 activation of a target net is not materialised by the forward chain (IDQN_F_CHAIN)");
    int rc = img_rebuild_activation(h, net, layer);
    if (rc) return rc;
  }
  CK(cudaMemcpyAsync(dst, h->act + (int64_t)net * h->act_stride + h->layers[layer].act_off, sizeof(float) * n,
                     cudaMemcpyDeviceToHost, h->stream));
  CK(cudaStreamSynchronize(h->stream));
  return IDQN_OK;
}
extern "C" int idqn_set_count(idqn_handle* h, const int32_t* c) {
  REQUIRE(h && c, "null argument");
  CK(cudaMemcpyAsync(h->count, c, sizeof(int32_t) * h->K, cudaMemcpyHostToDevice, h->stream));
  CK(cudaStreamSynchronize(h->stream));
  return IDQN_OK;
}
extern "C" int idqn_get_count(idqn_handle* h, int32_t* c) {
  REQUIRE(h && c, "null argument");
  CK(cudaMemcpyAsync(c, h->count, sizeof(int32_t) * h->K, cudaMemcpyDeviceToHost, h->stream));
  CK(cudaStreamSynchronize(h->stream));
  return IDQN_OK;
}

static int stage_batch(idqn_handle* h, const void* s, const void* s2, int u8, const int32_t* a, const float* r,
                       const uint8_t* d, cudaMemcpyKind kind) {
  REQUIRE(h && s && s2 && a && r && d, "null argument");
  CK(cudaSetDevice(h->cfg.device));
  const size_t sb = (size_t)h->in_elems * h->B * (u8 ? 1 : 4);
  CK(cudaMemcpyAsync(h->s, s, sb, kind, h->stream));
  CK(cudaMemcpyAsync(h->s2, s2, sb, kind, h->stream));
  CK(cudaMemcpyAsync(h->action, a, sizeof(int32_t) * h->B, kind, h->stream));
  CK(cudaMemcpyAsync(h->reward, r, sizeof(float) * h->B, kind, h->stream));
  CK(cudaMemcpyAsync(h->terminal, d, h->B, kind, h->stream));
  return IDQN_OK;
}

extern "C" int idqn_learn_on_batch_host(idqn_handle* h, const void* s, const void* s2, int u8, const int32_t* a,
                                        const float* r, const uint8_t* d, float* losses) {
  int rc = stage_batch(h, s, s2, u8, a, r, d, cudaMemcpyHostToDevice);
  if (rc) return rc;
  return idqn_learn_step_resident(h, u8, losses);
}
extern "C" int idqn_learn_on_batch_dev(idqn_handle* h, const void* s, const void* s2, int u8, const int32_t* a,
                                       const float* r, const uint8_t* d, float* losses) {
  int rc = stage_batch(h, s, s2, u8, a, r, d, cudaMemcpyDeviceToDevice);
  if (rc) return rc;
  return idqn_learn_step_resident(h, u8, losses);
}

// ---- pipelined host path --------------------------------------------------------------------------------------
// submit: the H2D copies of this batch go to the copy stream and land in one of two staging slots while the previous
// step still computes; the main stream picks the slot up with device-to-device copies, runs the step and sends the
// losses to a pinned ring.  wait: blocks on that step's completion event only.
static int pipeline_setup(idqn_handle* h) {
  if (h->copy_stream) return IDQN_OK;
  CK(cudaStreamCreateWithFlags(&h->copy_stream, cudaStreamNonBlocking));
  const size_t sb = (size_t)h->in_elems * h->B * 4;
  for (int i = 0; i < 2; ++i) {
    CK(cudaMalloc(&h->alt_s[i], sb));
    CK(cudaMalloc(&h->alt_s2[i], sb));
    CK(cudaMalloc(&h->alt_action[i], sizeof(int32_t) * h->B));
    CK(cudaMalloc(&h->alt_reward[i], sizeof(float) * h->B));
    CK(cudaMalloc(&h->alt_terminal[i], h->B));
    CK(cudaEventCreateWithFlags(&h->ev_h2d[i], cudaEventDisableTiming));
    CK(cudaEventCreateWithFlags(&h->ev_consumed[i], cudaEventDisableTiming));
    CK(cudaEventCreateWithFlags(&h->ev_done[i], cudaEventDisableTiming));
  }
  CK(cudaMallocHost(&h->h_loss_ring, sizeof(float) * 2 * h->K));
  h->next_ticket = 0;
  return IDQN_OK;
}

extern "C" int idqn_submit_batch_host(idqn_handle* h, const void* s, const void* s2, int u8, const int32_t* a,
                                      const float* r, const uint8_t* d, int64_t* ticket) {
  REQUIRE(h && s && s2 && a && r && d && ticket, "null argument");
  CK(cudaSetDevice(h->cfg.device));
  u8 = u8 ? 1 : 0;
  int rc = pipeline_setup(h);
  if (rc) return rc;
  rc = refresh_planes(h);
  if (rc) return rc;
  const int64_t t = h->next_ticket;
  const int slot = (int)(t & 1);
  if (t >= 2) CK(cudaEventSynchronize(h->ev_done[slot]));  // at most two steps in flight: the slot's loss entry is free
  const size_t sb = (size_t)h->in_elems * h->B * (u8 ? 1 : 4);
  if (t >= 2) CK(cudaStreamWaitEvent(h->copy_stream, h->ev_consumed[slot], 0));
  CK(cudaMemcpyAsync(h->alt_s[slot], s, sb, cudaMemcpyHostToDevice, h->copy_stream));
  CK(cudaMemcpyAsync(h->alt_s2[slot], s2, sb, cudaMemcpyHostToDevice, h->copy_stream));
  CK(cudaMemcpyAsync(h->alt_action[slot], a, sizeof(int32_t) * h->B, cudaMemcpyHostToDevice, h->copy_stream));
  CK(cudaMemcpyAsync(h->alt_reward[slot], r, sizeof(float) * h->B, cudaMemcpyHostToDevice, h->copy_stream));
  CK(cudaMemcpyAsync(h->alt_terminal[slot], d, h->B, cudaMemcpyHostToDevice, h->copy_stream));
  CK(cudaEventRecord(h->ev_h2d[slot], h->copy_stream));
  CK(cudaStreamWaitEvent(h->stream, h->ev_h2d[slot], 0));
  {
    // the step reads the slot in place: one captured graph per slot, no device-to-device staging copies
    void *s0 = h->s, *s20 = h->s2;
    int32_t* a0 = h->action;
    float* r0 = h->reward;
    uint8_t* d0 = h->terminal;
    float* l0 = h->loss;
    h->s = h->alt_s[slot], h->s2 = h->alt_s2[slot], h->action = h->alt_action[slot], h->reward = h->alt_reward[slot];
    h->terminal = h->alt_terminal[slot];
    // the K losses of this step are written by the loss kernel STRAIGHT into the slot's entry of the pinned host ring
    // (mapped memory, posted PCIe writes): no device-to-host copy operation sits between two steps on the compute stream
    h->loss = h->h_loss_ring + (size_t)slot * h->K;
    h->graph_set = 1 + slot;
    rc = idqn_learn_step_resident(h, u8, nullptr);
    h->graph_set = 0;
    h->s = s0, h->s2 = s20, h->action = a0, h->reward = r0, h->terminal = d0, h->loss = l0;
  }
  if (rc) return rc;
  CK(cudaEventRecord(h->ev_consumed[slot], h->stream));
  CK(cudaEventRecord(h->ev_done[slot], h->stream));
  *ticket = t;
  h->next_ticket = t + 1;
  return IDQN_OK;
}

extern "C" int idqn_wait_losses(idqn_handle* h, int64_t ticket, float* losses) {
  REQUIRE(h && h->copy_stream, "no batch was submitted");
  REQUIRE(ticket >= 0 && ticket < h->next_ticket && ticket + 2 >= h->next_ticket, "ticket %lld is not one of the two most recent submissions",
          (long long)ticket);
  CK(cudaSetDevice(h->cfg.device));
  const int slot = (int)(ticket & 1);
  CK(cudaEventSynchronize(h->ev_done[slot]));
  if (losses) memcpy(losses, h->h_loss_ring + (size_t)slot * h->K, sizeof(float) * h->K);
  return IDQN_OK;
}

// idqn.py:72: `self.cumulated_losses += losses` lives in update_online_params; a direct learn_on_batch call
// (idqn.py:96-109) leaves the running sums alone.  The switch is a device word the loss kernel reads, so the captured
// graph serves both callers.
extern "C" int idqn_set_loss_accumulation(idqn_handle* h, int on) {
  REQUIRE(h, "null handle");
  on = on ? 1 : 0;
  if (on == h->loss_acc_host) return IDQN_OK;
  CK(cudaSetDevice(h->cfg.device));
  // stream-ordered fill: steps already enqueued keep the value they were enqueued under
  CK(cudaMemsetAsync(h->loss_acc_on, on ? 1 : 0, 1, h->stream));
  h->loss_acc_host = on;
  return IDQN_OK;
}

// per-sample absolute TD errors of the most recent step, [K][B] (what rb.update(keys, priorities) is fed with)
extern "C" int idqn_read_td_abs(idqn_handle* h, float* out) {
  REQUIRE(h && out, "null argument");
  CK(cudaSetDevice(h->cfg.device));
  CK(cudaMemcpyAsync(out, h->td_abs, sizeof(float) * h->K * h->B, cudaMemcpyDeviceToHost, h->stream));
  CK(cudaStreamSynchronize(h->stream));
  return IDQN_OK;
}

extern "C" int idqn_read_cumulated_losses(idqn_handle* h, double* sums, int reset) {
  REQUIRE(h && sums, "null argument");
  CK(cudaSetDevice(h->cfg.device));
  CK(cudaMemcpyAsync(sums, h->loss_sum, sizeof(double) * h->K, cudaMemcpyDeviceToHost, h->stream));
  if (reset) CK(cudaMemsetAsync(h->loss_sum, 0, sizeof(double) * h->K, h->stream));
  CK(cudaStreamSynchronize(h->stream));
  return IDQN_OK;
}
extern "C" int idqn_write_cumulated_losses(idqn_handle* h, const double* sums) {
  REQUIRE(h && sums, "null argument");
  CK(cudaSetDevice(h->cfg.device));
  CK(cudaMemcpyAsync(h->loss_sum, sums, sizeof(double) * h->K, cudaMemcpyHostToDevice, h->stream));
  CK(cudaStreamSynchronize(h->stream));
  return IDQN_OK;
}

// the target events move the bf16 planes together with their fp32 masters
// The three target events move the bf16 planes together with the fp32 arenas: planes that are still stale (arena
// uploaded or rewritten since the last step) are rebuilt FIRST, otherwise the copy would propagate stale planes into
// an arena whose dirty bit is clear (a freshly constructed agent does upload(ONLINE) + copy_online_to_target()).
extern "C" int idqn_shift_params(idqn_handle* h) {  // idqn.py:13-17
  REQUIRE(h, "null handle");
  CK(cudaSetDevice(h->cfg.device));
  {
    int rc = refresh_planes(h);
    if (rc) return rc;
  }
  for (int k = 0; k + 1 < h->K; ++k) {
    const int64_t d = (int64_t)k * h->stride, s = (int64_t)(k + 1) * h->stride;
    CK(cudaMemcpyAsync(h->online + d, h->online + s, sizeof(float) * h->stride, cudaMemcpyDeviceToDevice, h->stream));
    int rc = copy_planes(h, h->won_hi + d, h->won_lo + d, h->won_hi + s, h->won_lo + s, 1);
    if (rc) return rc;
  }
  h->dense0_valid[0] = 0;
  return IDQN_OK;
}
extern "C" int idqn_sync_target(idqn_handle* h) {  // idqn.py:20-24
  REQUIRE(h, "null handle");
  CK(cudaSetDevice(h->cfg.device));
  {
    int rc = refresh_planes(h);
    if (rc) return rc;
  }
  if (h->K > 1) {
    const int64_t n = h->stride * (h->K - 1);
    CK(cudaMemcpyAsync(h->target + h->stride, h->online, sizeof(float) * n, cudaMemcpyDeviceToDevice, h->stream));
    int rc = copy_planes(h, h->wtg_hi + h->stride, h->wtg_lo + h->stride, h->won_hi, h->won_lo, h->K - 1);
    if (rc) return rc;
    h->dense0_valid[1] &= 1ull;  // only head 0 of the target arena keeps what it had
  }
  return IDQN_OK;
}
extern "C" int idqn_copy_online_to_target(idqn_handle* h) {  // idqn.py:78, dqn.py:52
  REQUIRE(h, "null handle");
  CK(cudaSetDevice(h->cfg.device));
  {
    int rc = refresh_planes(h);
    if (rc) return rc;
  }
  const int64_t n = h->stride * h->K;
  CK(cudaMemcpyAsync(h->target, h->online, sizeof(float) * n, cudaMemcpyDeviceToDevice, h->stream));
  int rc = copy_planes(h, h->wtg_hi, h->wtg_lo, h->won_hi, h->won_lo, h->K);
  if (rc) return rc;
  h->dense0_valid[1] = 0;
  return IDQN_OK;
}
// planes of externally modified arenas (NCCL / peer copies into idqn_arena_ptr memory) must be rebuilt
extern "C" int idqn_mark_planes_dirty(idqn_handle* h, int which) {
  REQUIRE(h && (which == IDQN_ONLINE || which == IDQN_TARGET), "bad argument");
  h->planes_dirty[which == IDQN_TARGET] = 1ull << 63;
  return IDQN_OK;
}
// the same for ONE head (the neighbour exchange of the sharded agent rewrites a single boundary head)
extern "C" int idqn_mark_head_planes_dirty(idqn_handle* h, int which, int head) {
  REQUIRE(h && (which == IDQN_ONLINE || which == IDQN_TARGET) && head >= 0 && head < h->K, "bad argument");
  h->planes_dirty[which == IDQN_TARGET] |= head < 63 ? 1ull << head : 1ull << 63;
  return IDQN_OK;
}

// network.apply of one head on n <= B inputs (already staged in h->s), result in h->q[0..n*A)
static int enqueue_apply(idqn_handle* h, int which, int head, int u8, int n) {
  int rc = refresh_planes(h);
  if (rc) return rc;
  rc = ensure_dense0_planes(h, which == IDQN_TARGET, head);
  if (rc) return rc;
  const bool tgt = which == IDQN_TARGET;
  const float* base = arena_of(h, which) + (int64_t)head * h->stride;
  const __nv_bfloat16* bh = (tgt ? h->wtg_hi : h->won_hi) + (int64_t)head * h->stride;
  const __nv_bfloat16* bl = (tgt ? h->wtg_lo : h->won_lo) + (int64_t)head * h->stride;
  if (use_tc(h) && (tc_conv_ok(h->layers[0]) || tc_dense_ok(h, h->layers[0]))) {
    if (((int64_t)n * h->in_elems) % 8 == 0) {
      rc = launch_input_planes(h, u8, n, 0);
      if (rc) return rc;
    }
  }
  for (int li = 0; li < h->n_layers; ++li) {
    FwdIO io;
    if (li == 0) {
      io.x = NetPtr{h->s, h->s, 0, 0, 1};
      io.xh = NetPtr{h->in_hi, h->in_hi, 0, 0, 1};
      io.xl = NetPtr{h->in_lo, h->in_lo, 0, 0, 1};
    } else {
      const int64_t o = h->layers[li - 1].act_off;
      io.x = NetPtr{h->act + o, h->act + o, 0, 0, 1};
      io.xh = NetPtr{h->act_hi + o, h->act_hi + o, 0, 0, 1};
      io.xl = NetPtr{h->act_lo + o, h->act_lo + o, 0, 0, 1};
    }
    io.w = NetPtr{base, base, 0, 0, 1};
    io.wh = NetPtr{bh, bh, 0, 0, 1};
    io.wl = NetPtr{bl, bl, 0, 0, 1};
    const bool last = li == h->n_layers - 1;
    const int64_t o = h->layers[li].act_off;
    io.y = last ? h->q : h->act + o;
    io.yh = last ? nullptr : h->act_hi + o;
    io.yl = last ? nullptr : h->act_lo + o;
    io.ystride = 0;
    if (h->layers[li].kind == IDQN_LAYER_POOL)
      rc = launch_pool_fwd(h, li, 1, n, h->act + h->layers[li - 1].act_off, h->act + o, 0);
    else
      rc = launch_fwd_layer(h, li, 1, 1, n, io, li == 0 ? u8 : 0, last ? 0 : h->layers[li].relu_out, false, nullptr, nullptr);
    if (rc) return rc;
  }
  return IDQN_OK;
}

// best_action fast path (idqn.py:126-131 at Atari shapes): the single uint8 state runs through the SAME image-resident conv
// kernels, weight-streaming Dense_0 kernel and head kernel as the learning step, as (online head, image 0) of the training
// layout -- the step's activation buffers are scratch between steps.  q[(head * B + 0) * A ..] receives the Q-values.
// idqn_select_actions runs the same kernels over images [0, imgs) of the online heads [head0, head0 + heads): every
// (net, image) unit is computed exactly as it is alone, so q[(head * B + i) * A ..] equals the single-state row.
static bool apply_fast_ok(const idqn_handle* h, int which, int u8) {
  if (!h->img_on || !h->img_host || which != IDQN_ONLINE || !u8 || h->n_layers != IDQN_IMG_LAYERS + 2) return false;
  const ImgHost* H = (const ImgHost*)h->img_host;
  return H->dense_on && H->dfwd.splits > 1 && !(h->cfg.flags & IDQN_F_SLOW_APPLY);
}
static int enqueue_apply_fast(idqn_handle* h, int head0, int heads = 1, int imgs = 1) {
  ImgHost* H = (ImgHost*)h->img_host;
  const int keep = h->n_launch, prof = h->prof_on;  // launch accounting / profiling belong to the learning step
  h->prof_on = 0;
  // units (net, image) of conv1/conv2 and (net, sample) pairs of the head: net-major, so the window from (head0, 0) to
  // (head0 + heads - 1, imgs - 1) also covers images >= imgs of the heads before the last (their results are not read)
  const int pairs = (heads - 1) * h->B + imgs, dunits = H->dfwd.tiles * H->dfwd.splits;
  int rc = refresh_planes(h);
  if (!rc) rc = img_launch_s2d(h, 1, imgs);
  if (!rc) rc = img_launch_taps(h, 0, false, 1, 0, imgs * H->fwd[0].n_hg);  // every online head group of images [0, imgs)
  for (int li = 1; li < IDQN_IMG_LAYERS && !rc; ++li) rc = img_launch_taps(h, li, false, 2, head0 * h->B, pairs);
  if (!rc) rc = dense_launch(h, false, false, head0 * dunits, heads * dunits);
  if (!rc) {
    const int L = h->n_layers;
    const Layer& l = h->layers[L - 1];
    HeadArgs a;
    memset(&a, 0, sizeof(a));
    const float* hid = h->act + h->layers[L - 2].act_off;
    a.hid = NetPtr{hid, hid, h->act_stride, h->act_stride, 2 * h->K};
    a.H = l.g.Kd, a.A = h->A, a.B = h->B, a.K = h->K;
    a.online = h->online, a.target = h->target;
    a.stride = h->stride, a.w_off = l.w_off, a.b_off = l.b_off;
    a.q = h->q;
    a.part = H->dfwd.part, a.ptiles = H->dfwd.tiles, a.psplits = H->dfwd.splits, a.pb_off = h->layers[L - 2].b_off;
    a.hbias_off = -1;
    a.tl_id = -1;
    a.cta0 = head0 * h->B;
    CK(launch_pdl(h->pdl, head_q_kernel, dim3(pairs), dim3(128), 0, h->stream, a));
  }
  h->n_launch = keep, h->prof_on = prof;
  return rc;
}

extern "C" int idqn_apply_host(idqn_handle* h, int which, int head, const void* x, int u8, int n, float* q) {
  REQUIRE(h && x && q && n >= 0, "bad argument");
  REQUIRE(which == IDQN_ONLINE || which == IDQN_TARGET, "apply needs the online or target arena");
  REQUIRE(head >= 0 && head < h->K, "bad head");
  CK(cudaSetDevice(h->cfg.device));
  const size_t esz = u8 ? 1 : 4;
  for (int done = 0; done < n; done += h->B) {
    const int m = std::min(h->B, n - done);
    CK(cudaMemcpyAsync(h->s, (const char*)x + (size_t)done * h->in_elems * esz, (size_t)m * h->in_elems * esz,
                       cudaMemcpyHostToDevice, h->stream));
    int rc = enqueue_apply(h, which, head, u8, m);
    if (rc) return rc;
    CK(cudaMemcpyAsync(q + (size_t)done * h->A, h->q, sizeof(float) * m * h->A, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
  }
  return IDQN_OK;
}

extern "C" int idqn_best_action(idqn_handle* h, int which, int head, const void* state, int u8, int32_t* action) {
  REQUIRE(h && state && action, "bad argument");
  REQUIRE(which == IDQN_ONLINE || which == IDQN_TARGET, "best_action needs the online or target arena");
  REQUIRE(head >= 0 && head < h->K, "bad head");
  CK(cudaSetDevice(h->cfg.device));
  const bool fast = apply_fast_ok(h, which, u8);
  if (fast && !(h->cfg.flags & IDQN_F_NO_GRAPH)) {
    // one graph launch per call: H2D of the state from pinned staging, the 7 kernels of the fast path, argmax, D2H of the
    // action (captured once per head; 9 API calls -> 1)
    int rc = refresh_planes(h);  // outside the capture: stale planes are a property of the moment, not of the graph
    if (rc) return rc;
    memcpy(h->h_state, state, (size_t)h->in_elems);
    cudaGraphExec_t& gx = h->act_graph[head];
    if (!gx) {
      cudaGraph_t g;
      CK(cudaStreamBeginCapture(h->stream, cudaStreamCaptureModeThreadLocal));
      cudaError_t e0 = cudaMemcpyAsync(h->s, h->h_state, (size_t)h->in_elems, cudaMemcpyHostToDevice, h->stream);
      rc = e0 == cudaSuccess ? enqueue_apply_fast(h, head) : IDQN_ECUDA;
      if (!rc) {
        argmax_kernel<<<1, 32, 0, h->stream>>>(h->q + (int64_t)head * h->B * h->A, h->A, (int32_t*)h->best_idx);
        if (cudaGetLastError() != cudaSuccess ||
            cudaMemcpyAsync(h->h_i32, h->best_idx, sizeof(int32_t), cudaMemcpyDeviceToHost, h->stream) != cudaSuccess)
          rc = IDQN_ECUDA;
      }
      cudaError_t e = cudaStreamEndCapture(h->stream, &g);
      if (rc || e != cudaSuccess) {
        if (e == cudaSuccess && g) cudaGraphDestroy(g);
        if (!rc) idqn_set_error("best_action: graph capture failed: %s", cudaGetErrorString(e));
        return rc ? rc : IDQN_ECUDA;
      }
      CK(cudaGraphInstantiate(&gx, g, 0));
      CK(cudaGraphDestroy(g));
    }
    CK(cudaGraphLaunch(gx, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    *action = h->h_i32[0];
    return IDQN_OK;
  }
  CK(cudaMemcpyAsync(h->s, state, (size_t)h->in_elems * (u8 ? 1 : 4), cudaMemcpyHostToDevice, h->stream));
  int rc = fast ? enqueue_apply_fast(h, head) : enqueue_apply(h, which, head, u8, 1);
  if (rc) return rc;
  // Q-values: q[0..A) (generic path) or the (head, sample 0) row of the step's layout; the index goes to the pinned word
  const float* qv = fast ? h->q + (int64_t)head * h->B * h->A : h->q;
  int32_t* d_out = (int32_t*)h->best_idx;
  argmax_kernel<<<1, 32, 0, h->stream>>>(qv, h->A, d_out);
  CK(cudaGetLastError());
  CK(cudaMemcpyAsync(h->h_i32, d_out, sizeof(int32_t), cudaMemcpyDeviceToHost, h->stream));
  CK(cudaStreamSynchronize(h->stream));
  *action = h->h_i32[0];
  return IDQN_OK;
}

// IDQN_F_TIMELINE: first-CTA-start / last-CTA-end global-timer stamps (ns) of every kernel of the most recent step,
// in launch order; resets the slots.  out: [2 * n] begin/end pairs, names: [32 * n]
extern "C" int idqn_kernel_timeline(idqn_handle* h, unsigned long long* out, char* names, int max_entries, int* n_out) {
  REQUIRE(h && out && names && n_out, "null argument");
  REQUIRE(h->cfg.flags & IDQN_F_TIMELINE, "the handle was created without IDQN_F_TIMELINE");
  CK(cudaSetDevice(h->cfg.device));
  CK(cudaStreamSynchronize(h->stream));
  const int n = std::min(std::min(h->n_launch, IDQN_KTL_MAX), max_entries);
  unsigned long long buf[2 * IDQN_KTL_MAX];
  CK(cudaMemcpyFromSymbol(buf, g_ktl, sizeof(buf)));
  memcpy(out, buf, sizeof(unsigned long long) * 2 * n);
  for (int i = 0; i < n; ++i) memcpy(names + 32 * i, h->tl_name[i], 32);
  for (int i = 0; i < IDQN_KTL_MAX; ++i) buf[2 * i] = ~0ull, buf[2 * i + 1] = 0;
  CK(cudaMemcpyToSymbol(g_ktl, buf, sizeof(buf)));
  *n_out = n;
  return IDQN_OK;
}

// ------------------------------------------------------------------------------------------
// Acting draw (slimdqn/sample_collection/utils.py:8-15 + idqn.py:126-131): jax's threefry2x32 PRNG restated on the host
// in C (the Python-int version cost 27 us per environment step).  Pinned against the values the JAX documentation prints
// for random.split / random.uniform (tests/test_cabi_and_host.py) and against the Random123 known answers.
static inline uint32_t tf_rotl(uint32_t x, int r) { return (x << r) | (x >> (32 - r)); }
static void threefry2x32(uint32_t k0, uint32_t k1, uint32_t x0, uint32_t x1, uint32_t* y0, uint32_t* y1) {
  static const int rot[2][4] = {{13, 15, 26, 6}, {17, 29, 16, 24}};
  const uint32_t ks[3] = {k0, k1, k0 ^ k1 ^ 0x1BD11BDAu};
  x0 += ks[0], x1 += ks[1];
  for (int i = 0; i < 5; ++i) {
    for (int j = 0; j < 4; ++j) {
      x0 += x1;
      x1 = tf_rotl(x1, rot[i % 2][j]) ^ x0;
    }
    x0 += ks[(i + 1) % 3];
    x1 += ks[(i + 2) % 3] + (uint32_t)(i + 1);
  }
  *y0 = x0, *y1 = x1;
}
// jax.random.split(key, num): counters arange(2 num) as (x0 = first half, x1 = second half); keys = concat(y0, y1).reshape(num, 2)
static void tf_split(uint32_t k0, uint32_t k1, int num, uint32_t* out /* [num][2] */) {
  std::vector<uint32_t> flat(2 * num);
  for (int i = 0; i < num; ++i) threefry2x32(k0, k1, (uint32_t)i, (uint32_t)(num + i), &flat[i], &flat[num + i]);
  for (int i = 0; i < 2 * num; ++i) out[i] = flat[i];
}
static uint32_t tf_bits32(uint32_t k0, uint32_t k1) {
  uint32_t a, b;
  threefry2x32(k0, k1, 0, 0, &a, &b);
  return a;
}
static float tf_uniform(uint32_t k0, uint32_t k1) {  // jax.random.uniform(key): mantissa bits | 1.0f, minus 1
  const uint32_t bits = (tf_bits32(k0, k1) >> 9) | 0x3F800000u;
  float f;
  memcpy(&f, &bits, 4);
  return f - 1.0f;
}
static int32_t tf_randint(uint32_t k0, uint32_t k1, int32_t minval, int32_t maxval) {  // jax.random.randint(key, (), lo, hi), int32
  uint32_t ks[4];
  tf_split(k0, k1, 2, ks);
  const uint32_t hi = tf_bits32(ks[0], ks[1]), lo = tf_bits32(ks[2], ks[3]);
  const uint32_t span = maxval > minval ? (uint32_t)(maxval - minval) : 1u;
  uint32_t mult = 65536u % span;
  mult = (uint32_t)(((uint64_t)mult * mult) % span);
  uint32_t off = (uint32_t)((uint64_t)(hi % span) * mult) + (lo % span);
  return minval + (int32_t)(off % span);
}

extern "C" int idqn_prng(int what, uint32_t key0, uint32_t key1, int32_t a, int32_t b, uint32_t* out) {
  REQUIRE(out, "null argument");
  switch (what) {
    case 0: tf_split(key0, key1, a, out); return IDQN_OK;                                 // split(key, a) -> out[2a]
    case 1: { float u = tf_uniform(key0, key1); memcpy(out, &u, 4); return IDQN_OK; }     // uniform(key) -> float bits
    case 2: out[0] = (uint32_t)tf_randint(key0, key1, a, b); return IDQN_OK;              // randint(key, (), a, b)
  }
  REQUIRE(false, "unknown draw %d", what);
}

// select_action (utils.py:8-15): uniform_key, action_key, kwargs_key = split(key, 3); explore if uniform(uniform_key) <= epsilon,
// else best_action(params, state, key=kwargs_key) whose head is randint(kwargs_key, (), 0, K) (idqn.py:128).
// info[0] = 1 if the random action was taken, info[1] = the head that was (or would have been) asked.
extern "C" int idqn_select_action(idqn_handle* h, const void* state, int u8, uint32_t key0, uint32_t key1, int n_actions,
                                  float epsilon, int32_t* action, int32_t* info) {
  REQUIRE(h && state && action, "null argument");
  uint32_t ks[6];
  tf_split(key0, key1, 3, ks);
  const bool explore = tf_uniform(ks[0], ks[1]) <= epsilon;
  const int32_t head = tf_randint(ks[4], ks[5], 0, h->K);
  if (info) info[0] = explore ? 1 : 0, info[1] = head;
  if (explore) {
    *action = tf_randint(ks[2], ks[3], 0, n_actions);
    return IDQN_OK;  // no device work at all on an exploring step
  }
  return idqn_best_action(h, IDQN_ONLINE, head, state, u8, action);
}

// ---- idqn_select_actions: the acting step of N environments ---------------------------------------------------------
// Staging block of one chunk (host and device alike): the B act codes of act_select_kernel, then the chunk's states.
static size_t vact_states_off(const idqn_handle* h) { return ((size_t)h->B * sizeof(int32_t) + 255) / 256 * 256; }
static size_t vact_block(const idqn_handle* h) {
  return (vact_states_off(h) + (size_t)h->B * h->in_elems * 4 + 255) / 256 * 256;
}

// pinned staging for `chunks` chunks (grown, never shrunk; nothing of ours is in flight between calls)
static int vact_reserve(idqn_handle* h, int64_t chunks) {
  if (!h->d_vact) {
    CK(cudaMalloc(&h->d_vact, vact_block(h)));
    CK(cudaMalloc(&h->d_vout, sizeof(int32_t) * h->B));
  }
  if (chunks <= h->vact_chunks) return IDQN_OK;
  if (h->h_vact) CK(cudaFreeHost(h->h_vact));
  if (h->h_vout) CK(cudaFreeHost(h->h_vout));
  h->h_vact = nullptr, h->h_vout = nullptr, h->vact_chunks = 0;
  CK(cudaMallocHost(&h->h_vact, (size_t)chunks * vact_block(h)));
  CK(cudaMallocHost(&h->h_vout, sizeof(int32_t) * chunks * h->B));
  h->vact_chunks = chunks;
  return IDQN_OK;
}

// the fast path's graph for a chunk of p (a power of two, or B) images: H2D of the staging block, the forward of every
// online head over images [0, p), act_select_kernel, D2H of the p actions.  Captured against chunk 0's pinned regions;
// vact_launch re-points the two copies at the chunk it runs.
static int vact_capture(idqn_handle* h, int slot, int p) {
  const size_t h2d = vact_states_off(h) + (size_t)p * h->in_elems;
  void* s0 = h->s;
  h->s = h->d_vact + vact_states_off(h);  // s2d_input_kernel reads the staged states in place
  cudaGraph_t g = nullptr;
  CK(cudaStreamBeginCapture(h->stream, cudaStreamCaptureModeThreadLocal));
  int rc = cudaMemcpyAsync(h->d_vact, h->h_vact, h2d, cudaMemcpyHostToDevice, h->stream) == cudaSuccess
               ? enqueue_apply_fast(h, 0, h->K, p) : IDQN_ECUDA;
  if (!rc) {
    act_select_kernel<<<(p + 3) / 4, 128, 0, h->stream>>>(h->q, h->A, (const int32_t*)h->d_vact, p, h->d_vout);
    if (cudaGetLastError() != cudaSuccess ||
        cudaMemcpyAsync(h->h_vout, h->d_vout, sizeof(int32_t) * p, cudaMemcpyDeviceToHost, h->stream) != cudaSuccess)
      rc = IDQN_ECUDA;
  }
  cudaError_t e = cudaStreamEndCapture(h->stream, &g);
  h->s = s0;
  if (rc || e != cudaSuccess) {
    if (e == cudaSuccess && g) cudaGraphDestroy(g);
    if (!rc) idqn_set_error("select_actions: graph capture failed: %s", cudaGetErrorString(e));
    return rc ? rc : IDQN_ECUDA;
  }
  size_t n_nodes = 0;
  CK(cudaGraphGetNodes(g, nullptr, &n_nodes));
  std::vector<cudaGraphNode_t> nodes(n_nodes);
  CK(cudaGraphGetNodes(g, nodes.data(), &n_nodes));
  h->vact_h2d[slot] = h->vact_d2h[slot] = nullptr;
  for (cudaGraphNode_t nd : nodes) {
    cudaGraphNodeType t;
    CK(cudaGraphNodeGetType(nd, &t));
    if (t != cudaGraphNodeTypeMemcpy) continue;
    cudaMemcpy3DParms mp;
    CK(cudaGraphMemcpyNodeGetParams(nd, &mp));
    (mp.dstPtr.ptr == h->d_vact ? h->vact_h2d : h->vact_d2h)[slot] = nd;
  }
  if (!h->vact_h2d[slot] || !h->vact_d2h[slot]) {
    cudaGraphDestroy(g);
    REQUIRE(false, "internal: select_actions graph without its two copies");
  }
  cudaError_t ei = cudaGraphInstantiate(&h->vact_exec[slot], g, 0);
  if (ei != cudaSuccess) {
    cudaGraphDestroy(g);
    CK(ei);
  }
  h->vact_graph[slot] = g;
  return IDQN_OK;
}

static int vact_launch(idqn_handle* h, int64_t chunk, int p) {
  int slot = 0;
  while ((1 << slot) < p) ++slot;
  if (!h->vact_exec[slot]) {
    int rc = vact_capture(h, slot, p);
    if (rc) return rc;
  }
  const size_t h2d = vact_states_off(h) + (size_t)p * h->in_elems;
  CK(cudaGraphExecMemcpyNodeSetParams1D(h->vact_exec[slot], h->vact_h2d[slot], h->d_vact,
                                        h->h_vact + chunk * vact_block(h), h2d, cudaMemcpyHostToDevice));
  CK(cudaGraphExecMemcpyNodeSetParams1D(h->vact_exec[slot], h->vact_d2h[slot], h->h_vout + chunk * h->B, h->d_vout,
                                        sizeof(int32_t) * p, cudaMemcpyDeviceToHost));
  CK(cudaGraphLaunch(h->vact_exec[slot], h->stream));
  return IDQN_OK;
}

// N x select_action (utils.py:8-15, idqn.py:126-131): env i draws with key (keys[2i], keys[2i+1]) exactly what
// idqn_select_action draws; the greedy ones are answered by one device pass per chunk of up to B environments.
extern "C" int idqn_select_actions(idqn_handle* h, const void* states, int u8, int n, const uint32_t* keys, int n_actions,
                                   float epsilon, int32_t* actions, int32_t* info) {
  REQUIRE(h, "null handle");
  REQUIRE(n >= 0, "select_actions: n = %d < 0", n);
  REQUIRE(n_actions > 0, "select_actions: n_actions = %d <= 0", n_actions);
  if (n == 0) return IDQN_OK;
  REQUIRE(states && keys && actions, "null argument");
  std::vector<int32_t> head(n), code(n);
  int n_greedy = 0;
  for (int i = 0; i < n; ++i) {
    uint32_t ks[6];
    tf_split(keys[2 * i], keys[2 * i + 1], 3, ks);
    const bool explore = tf_uniform(ks[0], ks[1]) <= epsilon;
    head[i] = tf_randint(ks[4], ks[5], 0, h->K);
    if (info) info[2 * i] = explore ? 1 : 0, info[2 * i + 1] = head[i];
    if (explore) actions[i] = tf_randint(ks[2], ks[3], 0, n_actions);
    code[i] = explore ? -1 - actions[i] : head[i];
    n_greedy += !explore;
  }
  if (!n_greedy) return IDQN_OK;  // no device work at all when every environment explores
  CK(cudaSetDevice(h->cfg.device));
  const size_t esz = u8 ? 1 : 4, sbytes = (size_t)h->in_elems * esz;
  const int B = h->B;
  int rc;
  if (apply_fast_ok(h, IDQN_ONLINE, u8) && !(h->cfg.flags & IDQN_F_NO_GRAPH)) {
    const int64_t chunks = (n + B - 1) / B;
    if ((rc = vact_reserve(h, chunks))) return rc;
    if ((rc = refresh_planes(h))) return rc;  // outside the capture, as in idqn_best_action
    for (int64_t c = 0; c < chunks; ++c) {
      const int i0 = (int)(c * B), m = std::min(B, n - i0);
      bool any = false;
      for (int j = 0; j < m; ++j) any |= code[i0 + j] >= 0;
      if (!any) continue;
      int p = 1;
      while (p < m) p <<= 1;
      p = std::min(p, B);
      uint8_t* blk = h->h_vact + c * vact_block(h);
      int32_t* bc = (int32_t*)blk;
      uint8_t* bs = blk + vact_states_off(h);
      for (int j = 0; j < p; ++j) bc[j] = j >= m ? -1 : code[i0 + j] >= 0 ? code[i0 + j] * B + j : code[i0 + j];
      memcpy(bs, (const uint8_t*)states + (size_t)i0 * sbytes, (size_t)m * sbytes);
      memset(bs + (size_t)m * sbytes, 0, (size_t)(p - m) * sbytes);  // padding: zero images
      if ((rc = vact_launch(h, c, p))) return rc;
    }
    CK(cudaStreamSynchronize(h->stream));
    for (int i = 0; i < n; ++i)
      if (code[i] >= 0) actions[i] = h->h_vout[i];  // chunk c's actions sit at h_vout + c * B
    return IDQN_OK;
  }
  // generic path: the greedy states grouped by head (pinned, in chunks of B), enqueue_apply of that head per chunk, then
  // act_select_kernel over its q rows
  std::vector<int> order;
  order.reserve(n_greedy);
  for (int k = 0; k < h->K; ++k)
    for (int i = 0; i < n; ++i)
      if (code[i] == k) order.push_back(i);
  const int64_t blocks = ((int64_t)n_greedy * sbytes + vact_block(h) - 1) / vact_block(h);
  if ((rc = vact_reserve(h, std::max<int64_t>(blocks, (n_greedy + B - 1) / B)))) return rc;
  for (int j = 0; j < n_greedy; ++j)
    memcpy(h->h_vact + (size_t)j * sbytes, (const uint8_t*)states + (size_t)order[j] * sbytes, sbytes);
  for (int j0 = 0; j0 < n_greedy;) {
    const int k = code[order[j0]];
    int m = 0;
    while (j0 + m < n_greedy && m < B && code[order[j0 + m]] == k) ++m;
    CK(cudaMemcpyAsync(h->s, h->h_vact + (size_t)j0 * sbytes, (size_t)m * sbytes, cudaMemcpyHostToDevice, h->stream));
    if ((rc = enqueue_apply(h, IDQN_ONLINE, k, u8, m))) return rc;
    act_select_kernel<<<(m + 3) / 4, 128, 0, h->stream>>>(h->q, h->A, nullptr, m, h->d_vout);
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(h->h_vout + j0, h->d_vout, sizeof(int32_t) * m, cudaMemcpyDeviceToHost, h->stream));
    j0 += m;
  }
  CK(cudaStreamSynchronize(h->stream));
  for (int j = 0; j < n_greedy; ++j) actions[order[j]] = h->h_vout[j];
  return IDQN_OK;
}

// IDQN_F_TIMELINE: per-CTA stamps (entry, first operand landed, last MMA committed, exit; ns) of the kernel in timeline slot
// `slot` during the steps run since the selection; slot < 0 turns the recording off.  out: [4 * n_ctas]
extern "C" int idqn_cta_timeline(idqn_handle* h, int slot, unsigned long long* out, int max_ctas, int* n_out) {
  REQUIRE(h, "null handle");
  CK(cudaSetDevice(h->cfg.device));
  CK(cudaStreamSynchronize(h->stream));
  if (out && n_out) {
    const int n = std::min(max_ctas, IDQN_CTL_MAX);
    static unsigned long long buf[IDQN_CTL_MAX * 4];
    CK(cudaMemcpyFromSymbol(buf, g_ctl, sizeof(buf)));
    memcpy(out, buf, sizeof(unsigned long long) * 4 * n);
    *n_out = n;
  }
  static unsigned long long zeros[IDQN_CTL_MAX * 4];
  CK(cudaMemcpyToSymbol(g_ctl, zeros, sizeof(zeros)));
  CK(cudaMemcpyToSymbol(g_ctl_sel, &slot, sizeof(int)));
  return IDQN_OK;
}

// CTAs the graph-replayed step gives the Dense_0 weight-gradient + Adam kernel next to the conv backward chain
// (0: the kernel runs after the chain on the whole machine)
extern "C" int idqn_dense_update_ctas(idqn_handle* h) { return h ? dense_update_ctas(h) : 0; }

// n > 0: the Dense_0 update runs on n CTAs next to the conv backward chain; 0: after the chain on every SM; < 0: automatic
// (58 + 6.5 K).  Call before the first learning step: captured graphs keep the schedule they were captured with.
extern "C" int idqn_set_dense_update_ctas(idqn_handle* h, int n) {
  REQUIRE(h, "null handle");
  h->update_ctas_set = n < 0 ? 0 : n + 1;
  return IDQN_OK;
}
