// Shared declarations of libidqn_b200 (internal; the public surface is include/idqn_b200.h).
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdarg.h>
#include <string.h>
#include <unordered_set>
#include <vector>

#include "../../include/idqn_b200.h"

void idqn_set_error(const char* fmt, ...);

#define CK(expr)                                                                               \
  do {                                                                                         \
    cudaError_t e_ = (expr);                                                                   \
    if (e_ != cudaSuccess) {                                                                   \
      idqn_set_error("%s:%d: %s -> %s", __FILE__, __LINE__, #expr, cudaGetErrorString(e_));    \
      return IDQN_ECUDA;                                                                       \
    }                                                                                          \
  } while (0)

#define REQUIRE(cond, ...)                                                                     \
  do {                                                                                         \
    if (!(cond)) {                                                                             \
      idqn_set_error(__VA_ARGS__);                                                             \
      return IDQN_EINVAL;                                                                      \
    }                                                                                          \
  } while (0)

// ---------------------------------------------------------------------------------------------
// Programmatic dependent launch.  Every kernel of the learning step calls pdl_trigger() first thing (the next
// kernel of the stream / graph may then be scheduled as SM resources free up and run its prologue: barrier init,
// TMEM allocation, tensor-map prefetch, weight tiles) and pdl_wait() before it touches anything the step produces
// (full completion + visibility of all earlier kernels).  Without the launch attribute both are no-ops.
// Measured on B200 (K = 5 step, CUDA graph): 0.353 ms with the attribute, 0.358 ms without -- on unless IDQN_F_NO_PDL
// (an earlier generation of the conv kernels measured 0.481 vs 0.458 ms the other way round).
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

// ---------------------------------------------------------------------------------------------
// In-graph kernel timeline (IDQN_F_TIMELINE): every kernel of the step stamps the global timer when its first CTA
// starts and when its last CTA ends, so the true schedule of the captured graph (branches, programmatic dependent
// launch overlap, gaps between kernels) can be read back -- ncu serialises kernels and events cannot be recorded inside a
// graph replay.  tl_id < 0: off (one predictable branch per CTA).
#define IDQN_KTL_MAX 64
static __device__ unsigned long long g_ktl[2 * IDQN_KTL_MAX];
__device__ __forceinline__ unsigned long long ktl_now() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}
__device__ __forceinline__ void ktl_begin(int id) {
  if (id >= 0 && threadIdx.x == 0) atomicMin(&g_ktl[2 * id], ktl_now());
}
// call where every thread of the CTA arrives (the timeline build syncs the CTA first)
__device__ __forceinline__ void ktl_end(int id) {
  if (id >= 0) {
    __syncthreads();
    if (threadIdx.x == 0) atomicMax(&g_ktl[2 * id + 1], ktl_now());
  }
}

// per-CTA stamps of ONE kernel of the step (the one whose timeline slot equals g_ctl_sel): [cta][0] entry, [1] first operand
// landed, [2] last MMA committed, [3] exit -- where inside a kernel's span its CTAs spend their time (tools/cta_timeline.py)
#define IDQN_CTL_MAX 160
static __device__ unsigned long long g_ctl[IDQN_CTL_MAX * 4];
static __device__ int g_ctl_sel = -1;
__device__ __forceinline__ void ctl_stamp(int id, int k) {
  if (id >= 0 && id == g_ctl_sel && blockIdx.x < IDQN_CTL_MAX) g_ctl[blockIdx.x * 4 + k] = ktl_now();
}

template <class... KArgs, class... Args>
static inline cudaError_t launch_pdl(bool pdl, void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st,
                                     Args&&... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid, cfg.blockDim = block, cfg.dynamicSmemBytes = smem, cfg.stream = st;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  at[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = at, cfg.numAttrs = pdl ? 1 : 0;
  return cudaLaunchKernelEx(&cfg, kern, static_cast<KArgs>(args)...);
}

// ---------------------------------------------------------------------------------------------
// division by a runtime constant with one mul.hi + shift (valid for 0 <= n < 2^31)
struct FastDiv {
  uint32_t d, mul, shr;
  __host__ __device__ FastDiv() : d(1), mul(0), shr(0) {}
  __host__ explicit FastDiv(uint32_t div) : d(div), mul(0), shr(0) {
    if (div > 1) {
      uint32_t lg = 0;
      while ((1ull << lg) < div) ++lg;
      uint32_t p = 31 + lg;
      mul = (uint32_t)(((1ull << p) + div - 1) / div);
      shr = p - 32;
    }
  }
  __host__ __device__ __forceinline__ uint32_t div(uint32_t n) const {
#ifdef __CUDA_ARCH__
    return d == 1 ? n : (__umulhi(n, mul) >> shr);
#else
    return d == 1 ? n : (uint32_t)((((uint64_t)n * mul) >> 32) >> shr);
#endif
  }
  __host__ __device__ __forceinline__ void divmod(uint32_t n, uint32_t& q, uint32_t& r) const {
    q = div(n);
    r = n - q * d;
  }
};

// ring slot of frame id `id` (>= 0) in a frame store of n_frames frames: 32-bit remainder while both fit (every id of a
// run shorter than 2^32 frames), the 64-bit one after
__host__ __device__ __forceinline__ int64_t frame_ring_slot(int64_t id, int64_t n_frames) {
  if ((((uint64_t)id | (uint64_t)n_frames) >> 32) == 0) return (int64_t)((uint32_t)id % (uint32_t)n_frames);
  return id % n_frames;
}

// ---------------------------------------------------------------------------------------------
// One layer of DQNNet seen as a convolution (Dense == 1x1 conv on a 1x1 image with IC = fan-in).
struct ConvGeom {
  int B;                // samples in the batch
  int IH, IW, IC;       // input  (NHWC)
  int OH, OW, OC;       // output (NHWC)
  int KH, KW, S;        // kernel, stride
  int PH, PW;           // low-side SAME padding (XLA: total//2)
  int Kd;               // KH*KW*IC  (rows of the flax kernel seen as a [Kd, OC] matrix)
  FastDiv d_ohow, d_ow, d_kwic, d_ic, d_oc;
};

#define IDQN_LAYER_GEMM 0  /* conv / dense: has a kernel and a bias */
#define IDQN_LAYER_POOL 1  /* max-pool (impala, architectures/dqn.py:20): no parameters */
struct Layer {
  ConvGeom g;           // with g.B == cfg.batch_size
  int is_conv;
  int kind;             // IDQN_LAYER_*
  // y = [relu_out] (conv([relu_in] x) + b) [+ output of layer skip_from].  cnn / fc: relu_out on every hidden layer; impala's
  // pre-activation residual blocks (architectures/dqn.py:22-27) use all three
  int relu_in, relu_out, skip_from;
  int64_t w_off, b_off; // float offsets inside a head's arena (b_off == w_off + Kd*OC)
  int64_t act_off;      // float offset of this layer's output inside one net's activation block (per sample count B)
  int64_t act_size;     // B*OH*OW*OC
  char name[16];
};

#define IDQN_MAX_LAYERS 32  /* impala: 3 x (5 convs + pool) + dense trunk */
#define IDQN_PROF_MAX 128
#define IDQN_IMG_LAYERS 3

// per conv layer state of the image-resident tensor-core path (conv_img.cuh): space-to-depth activation planes
// X2 (input of the layer), zero-embedded output-gradient planes dyZ, and the TMA tensor maps over them
struct ImgLayerState {
  alignas(64) CUtensorMap mapX[2], mapW[2], mapZ[2];  // hi, lo
  alignas(64) CUtensorMap mapXw[2], mapZw[2];         // the same X2 / dyZ planes with the part boxes of conv_wgrad_kernel
  __nv_bfloat16 *x2_hi, *x2_lo;   // [nets][B][XRa][C2]  (layer 0: nets = 2 inputs; else 2K nets)
  __nv_bfloat16 *dz_hi, *dz_lo;   // [K][B][ZRa][OC]
  int64_t x2_net_stride, dz_net_stride;  // elements
};

struct idqn_handle {
  idqn_config cfg;
  int n_layers;
  Layer layers[IDQN_MAX_LAYERS];
  int n_param_layers, param_layer[IDQN_MAX_LAYERS];  // layers that own a (kernel, bias) leaf pair, in flax creation order
  int64_t stride;       // floats per head in every arena
  int64_t in_elems;     // elements of one input sample
  int K, B, A;
  cudaStream_t stream;
  // SM partitions of the backward pass (sm_partition.cuh): conv chain | HBM-bound Dense_0 wgrad+Adam
  void* partition;      // smpart::Partition, null when green contexts are unavailable or disabled
  // impala: the max-pool forward of the learning step records which window element it took (one byte per output element of the
  // online nets, indexed like act); the backward reads it.  pool_arg_ok[li]: the last step forward of pool layer li recorded it
  uint8_t* pool_arg;
  unsigned char pool_arg_ok[IDQN_MAX_LAYERS];
  cudaEvent_t ev_fork, ev_join[2];
  // second branch of the step graph: the conv weight-gradient kernels run next to the conv data-gradient chain
  cudaStream_t side, side2;
  cudaEvent_t ev_fork2;
  cudaEvent_t ev_conv[IDQN_IMG_LAYERS], ev_side_done;
  float part_frac;      // share of the Dense_0 wgrad+Adam tiles that run inside the partition
  int wg_tile0, wg_tiles;  // tile range of the next Dense wgrad+Adam launch (wg_tiles == 0: all)
  int update_ctas_set;     // idqn_set_dense_update_ctas: 0 = automatic, n + 1 = n CTAs (n = 0: after the conv chain, every SM)
  int sm_avail;         // SMs of the stream the next launches go to
  // arenas [K][stride]
  float *online, *target, *mu, *nu, *grad;
  int32_t* count;       // [K]
  float* loss;          // [K] last step
  double* loss_sum;     // [K] cumulated (idqn.py:72)
  float* td_abs;        // [K][B] per-sample |TD error| of the last step (priorities of prioritised replay)
  cudaEvent_t ev_step;  // recorded behind a step when another stream has to order itself after it (sum-tree update)
  int32_t* loss_acc_on; // device word: 1 = steps add their losses to loss_sum (update_online_params), 0 = they do not
  int loss_acc_host;    // host mirror of that word
  // batch staging (device)
  void *s, *s2;         // [B][in_elems] u8 or f32 (allocated for f32)
  int32_t* action;
  float* reward;
  uint8_t* terminal;
  // activations: nets g in [0,2K): g<K online on s, g>=K target on s'
  float* act;           // [2K][act_stride]
  int64_t act_stride;
  float* dact;          // [K][act_stride]   gradients w.r.t. layer outputs
  float* q;             // [2K][B][A] final-layer outputs (debug / apply)
  // bf16 hi/lo planes of every tensor-core GEMM operand (gemm_tc.cuh), same element indexing as the fp32 master
  __nv_bfloat16 *won_hi, *won_lo, *wtg_hi, *wtg_lo;  // [K][stride]      online / target weights
  __nv_bfloat16 *act_hi, *act_lo;                    // [2K][act_stride]
  __nv_bfloat16 *dact_hi, *dact_lo;                  // [K][act_stride]
  __nv_bfloat16 *in_hi, *in_lo;                      // [2][B*in_elems]  state, next_state
  __nv_bfloat16* ones;                               // {1,0 x7 | 0 x8}: bias-gradient row of the wgrad GEMMs
  unsigned long long planes_dirty[2];                // online / target planes stale: bit k = head k (bit 63: every head)
  int fast_dense;                                    // the big Dense layer has NO maintained planes: arena range [d0_lo, d0_hi)
  int64_t d0_lo, d0_hi;                              //   is skipped by every plane producer (refresh, target events, Adam)
  unsigned long long dense0_valid[2];                // ... and rebuilt on demand for the generic kernels: bit k = head k valid
  __nv_bfloat16 *wpl_hi, *wpl_lo;                    // the allocation behind won_*/wtg_*: [2K][stride], online first
  // image-resident conv path (conv_img.cuh); img_on == 0 -> the generic kernels of gemm_tc.cuh run instead
  int img_on;
  int img_last;           // the most recent step ran the image path (conv activations live in planes only)
  int pdl;                // launch the step's kernels with programmatic stream serialization
  ImgLayerState il[IDQN_IMG_LAYERS];
  void* img_host;         // ImgHost (net.cu): geometry and kernel arguments of the three conv layers
  float* wpart;           // [K][wgroups][wspan] partial conv weight gradients in arena coordinates
  int wgroups;
  int64_t wspan;
  // split-K workspace
  float* part;
  int64_t part_floats;
  int* tickets;
  int n_tickets;
  // pipelined host path (idqn_submit_batch_host / idqn_wait_losses): two staging slots filled by the copy stream
  cudaStream_t copy_stream;
  void *alt_s[2], *alt_s2[2];
  int32_t* alt_action[2];
  float* alt_reward[2];
  uint8_t* alt_terminal[2];
  float* h_loss_ring;   // pinned [2][K]
  cudaEvent_t ev_h2d[2], ev_consumed[2], ev_done[2];
  int64_t next_ticket;
  int32_t* best_idx;     // device word receiving the argmax of best_action
  cudaGraphExec_t* act_graph;  // [K] best_action fast path of head k as ONE graph launch (H2D state, 7 kernels, D2H action)
  uint8_t* h_state;      // pinned staging of the acting state (source of the graphs' H2D node)
  // idqn_select_actions, allocated on its first call: per chunk of up to B environments, a pinned staging block (act
  // codes, then the states) and the actions it gets back; one device copy of a block and the chunk's actions
  uint8_t* h_vact;       // pinned [chunks][vact_block]
  int32_t* h_vout;       // pinned [chunks * B]
  size_t h_vact_bytes;
  int64_t vact_chunks;   // chunks h_vact / h_vout hold
  uint8_t* d_vact;       // [vact_block]
  int32_t* d_vout;       // [B]
  cudaGraph_t vact_graph[8];          // fast path, one per padded chunk size 2^i (kept: its memcpy nodes are re-pointed)
  cudaGraphExec_t vact_exec[8];
  cudaGraphNode_t vact_h2d[8], vact_d2h[8];
  // pinned host scratch
  float* h_loss;
  int32_t* h_i32;
  // CUDA graph of one learn step, per input dtype (0: f32, 1: u8)
  cudaGraphExec_t graph[8];  // [staging set: 0 = s/s2/..., 1 + i = pipelined slot i, 3 = replay slots in place][input dtype]
  // replay-direct input (idqn_learn_from_replay on the image path): the first kernel of the step reads the frames
  // straight from the replay slots and gathers the scalars -- no gather kernel, no staging copy
  struct {
    const uint8_t *state, *next_state;
    const int64_t* slots;
    int64_t state_bytes;
    const int32_t* action;
    const double* reward;
    const uint8_t* terminal;
    // frame store (idqn_replay_create_frames): state/next_state are null and image g of slot s is assembled from the
    // frames rows[(s * 2 + g) * stack + c] (id -1: a zero frame), frame id f at ring + (f % n_frames) * frame_bytes
    const uint8_t* ring;
    const int64_t* rows;
    int64_t n_frames, frame_bytes;
    int stack;
  } rsrc;
  int rsrc_on;
  int graph_set;             // staging set the next step reads (idqn_submit_batch_host points the step at its slot)
  int sm_count;
  // launch accounting / live per-kernel timing (idqn_profile_step)
  int n_launch;          // kernels enqueued by the last enqueue_learn_step
  char tl_name[IDQN_KTL_MAX][32];  // IDQN_F_TIMELINE: kernel names by timeline id (= launch index inside the step)
  int prof_on, prof_n;
  cudaEvent_t prof_ev[IDQN_PROF_MAX + 1];
  char prof_name[IDQN_PROF_MAX][32];
};

// replay store (replay.cu)
struct idqn_replay {
  int device;
  int64_t n_slots, state_bytes;
  uint8_t *state, *next_state;
  int32_t* action;
  double* reward;
  uint8_t *terminal, *episode_end;
  cudaStream_t stream;
  int64_t* d_slots;  // device copy of the LEARNER's gather indices (read by the step graph on the learner's stream)
  int64_t cap_slots; // capacity of d_slots
  int64_t* d_gslots; // index buffer of idqn_replay_gather_host (own buffer: the learner's graph may still read d_slots)
  int64_t cap_gslots;
  // the most recent learner step reads its sampled slots IN PLACE, asynchronously, on the learner's stream: a put into
  // one of those slots first waits for that step's event (every other slot is written without waiting)
  cudaEvent_t ev_learner;
  int learner_pending;
  std::vector<int64_t>* learner_slots;
  // frame store (idqn_replay_create_frames; state/next_state stay null): each observation once, in a ring of n_frames
  // frames of value_bytes-byte values; slot s holds 2*stack frame ids (state positions, then next_state positions; -1 = zero frame) in rows and its
  // host mirror h_rows.  state_bytes = frame_bytes * stack.  Unlike learner_slots, the element rows and ring slots of
  // the in-flight steps accumulate until ev_learner has completed: a write into any of them waits for it.
  int frames;
  int stack, value_bytes;
  int64_t frame_bytes, n_frames;
  uint8_t* ring;
  int64_t* rows;
  int64_t* h_rows;
  std::unordered_set<int64_t> *inflight_rows, *inflight_frames;
  // pinned staging for gather_host
  void* h_stage;
  size_t h_stage_bytes;
};

int idqn_learn_step_resident(idqn_handle* h, int state_is_u8, float* losses_host);

// SumTree (sumtree.cu); declared here so that the learner-side update can reach it
struct idqn_sumtree;
