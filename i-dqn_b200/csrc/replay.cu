// Device-resident replay store + batch gather (slimdqn/sample_collection/replay_buffer.py:202-230).
//
// The reference keeps snappy-compressed ReplayElements in a host OrderedDict and rebuilds a batch with
// dict lookups + decompress + np.stack + H2D every step.  Here elements live uncompressed in fixed HBM slots
// (1M Atari elements = 56.4 GB of the 180 GB) and `sample` is one coalesced 16-byte-vector gather straight
// into the learner's batch staging: no host round trip on the step path.
//
// The frame store (idqn_replay_create_frames) is the reference's ReplayBuffer(compress=True) in spirit
// (replay_buffer.py:36-57,204-205): consecutive elements share 2*stack - 1 of their frames, so it keeps each observation
// once in a ring of frames (1M Atari elements = 7.1 GB) and an element as 2*stack frame ids; the learning step and the
// gather assemble the stacks from the ring.
#include "common.cuh"

#include <algorithm>

struct GatherArgs {
  const uint8_t* state;
  const uint8_t* next_state;
  const int32_t* action;
  const double* reward;
  const uint8_t* terminal;
  const uint8_t* episode_end;
  const int64_t* slots;
  int64_t state_bytes;
  // frame store: the stacks are assembled from ring frames (see idqn_replay)
  const uint8_t* ring;
  const int64_t* rows;
  int64_t n_frames, frame_bytes;
  int stack, value_bytes;
  int n;
  uint8_t* o_state;
  uint8_t* o_next;
  int32_t* o_action;
  float* o_reward_f32;   // learner staging (f32, like the jit boundary of the reference) or null
  double* o_reward_f64;  // host-facing (np.stack of python floats) or null
  uint8_t* o_terminal;
  uint8_t* o_episode_end;  // may be null
};

__device__ __forceinline__ void gather_scalars(const GatherArgs& a, int i, int64_t slot) {
  a.o_action[i] = a.action[slot];
  if (a.o_reward_f32) a.o_reward_f32[i] = __double2float_rn(a.reward[slot]);
  if (a.o_reward_f64) a.o_reward_f64[i] = a.reward[slot];
  a.o_terminal[i] = a.terminal[slot];
  if (a.o_episode_end) a.o_episode_end[i] = a.episode_end[slot];
}

// grid: (chunks, 2n) — blockIdx.y < n copies state of sample y, otherwise next_state of sample y-n
__global__ void __launch_bounds__(256) replay_gather_kernel(const GatherArgs a) {
  const int which = blockIdx.y >= a.n;
  const int i = blockIdx.y - which * a.n;
  const int64_t slot = a.slots[i];
  const uint8_t* src = (which ? a.next_state : a.state) + slot * a.state_bytes;
  uint8_t* dst = (which ? a.o_next : a.o_state) + (int64_t)i * a.state_bytes;
  if ((a.state_bytes & 15) == 0) {
    const int64_t n16 = a.state_bytes >> 4;
    const int4* s4 = reinterpret_cast<const int4*>(src);
    int4* d4 = reinterpret_cast<int4*>(dst);
    for (int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; j < n16; j += (int64_t)gridDim.x * blockDim.x)
      d4[j] = __ldcs(s4 + j);  // streamed once: keep it out of the way of the weights in L2
  } else {
    for (int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; j < a.state_bytes;
         j += (int64_t)gridDim.x * blockDim.x)
      dst[j] = src[j];
  }
  if (blockIdx.x == 0 && which == 0 && threadIdx.x == 0) gather_scalars(a, i, slot);
}

// frame store: the same grid; value v * stack + p of the stack is value v of frame rows[(slot * 2 + which) * stack + p]
__global__ void __launch_bounds__(256) replay_gather_frames_kernel(const GatherArgs a) {
  const int which = blockIdx.y >= a.n;
  const int i = blockIdx.y - which * a.n;
  const int64_t slot = a.slots[i];
  const int64_t* row = a.rows + (slot * 2 + which) * a.stack;
  uint8_t* dst = (which ? a.o_next : a.o_state) + (int64_t)i * a.state_bytes;
  if (a.stack == 4 && a.value_bytes == 1 && (a.frame_bytes & 3) == 0) {
    // Atari: 16 output bytes = 4 bytes of each of the 4 frames, interleaved
    const uint8_t* f[4];
#pragma unroll
    for (int c = 0; c < 4; ++c) {
      const int64_t id = row[c];
      f[c] = id < 0 ? nullptr : a.ring + frame_ring_slot(id, a.n_frames) * a.frame_bytes;
    }
    const int64_t n16 = a.frame_bytes >> 2;
    int4* d4 = reinterpret_cast<int4*>(dst);
    for (int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; j < n16; j += (int64_t)gridDim.x * blockDim.x) {
      uint32_t p[4];
#pragma unroll
      for (int c = 0; c < 4; ++c) p[c] = f[c] ? __ldcs(reinterpret_cast<const unsigned int*>(f[c]) + j) : 0u;
      const uint32_t lo01 = __byte_perm(p[0], p[1], 0x5140), hi01 = __byte_perm(p[0], p[1], 0x7362);
      const uint32_t lo23 = __byte_perm(p[2], p[3], 0x5140), hi23 = __byte_perm(p[2], p[3], 0x7362);
      d4[j] = make_int4((int)__byte_perm(lo01, lo23, 0x5410), (int)__byte_perm(lo01, lo23, 0x7632),
                        (int)__byte_perm(hi01, hi23, 0x5410), (int)__byte_perm(hi01, hi23, 0x7632));
    }
  } else {
    for (int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; j < a.state_bytes;
         j += (int64_t)gridDim.x * blockDim.x) {
      const int64_t t = j / a.value_bytes, b = j - t * a.value_bytes;  // byte b of value t / stack of frame t % stack
      const int64_t id = row[t % a.stack];
      dst[j] = id < 0 ? 0 : a.ring[frame_ring_slot(id, a.n_frames) * a.frame_bytes + t / a.stack * a.value_bytes + b];
    }
  }
  if (blockIdx.x == 0 && which == 0 && threadIdx.x == 0) gather_scalars(a, i, slot);
}

static int ensure_slots(idqn_replay* r, int n) {
  if (n <= r->cap_slots) return IDQN_OK;
  if (r->d_slots) cudaFree(r->d_slots);
  r->cap_slots = std::max(n, 256);
  CK(cudaMalloc(&r->d_slots, sizeof(int64_t) * r->cap_slots));
  return IDQN_OK;
}

static int launch_gather(idqn_replay* r, GatherArgs& a, cudaStream_t st, const int64_t* d_slots) {
  a.state = r->state, a.next_state = r->next_state, a.action = r->action, a.reward = r->reward;
  a.terminal = r->terminal, a.episode_end = r->episode_end, a.slots = d_slots, a.state_bytes = r->state_bytes;
  a.ring = r->ring, a.rows = r->rows, a.n_frames = r->n_frames, a.frame_bytes = r->frame_bytes, a.stack = r->stack;
  a.value_bytes = r->value_bytes;
  int64_t per = (r->state_bytes & 15) == 0 ? r->state_bytes / 16 : r->state_bytes;
  if (r->frames) per = r->stack == 4 && r->value_bytes == 1 && (r->frame_bytes & 3) == 0 ? r->frame_bytes / 4 : r->state_bytes;
  int chunks = (int)std::min<int64_t>(std::max<int64_t>((per + 255) / 256, 1), 64);
  if (r->frames) replay_gather_frames_kernel<<<dim3(chunks, 2 * a.n), 256, 0, st>>>(a);
  else replay_gather_kernel<<<dim3(chunks, 2 * a.n), 256, 0, st>>>(a);
  CK(cudaGetLastError());
  return IDQN_OK;
}

static int enough_hbm(size_t need) {
  size_t free_b = 0, total_b = 0;
  CK(cudaMemGetInfo(&free_b, &total_b));
  if (need > free_b) {
    idqn_set_error("replay store needs %zu bytes of HBM, only %zu free", need, free_b);
    return IDQN_ENOMEM;
  }
  return IDQN_OK;
}

// the scalars, the stream and the learner bookkeeping of both kinds of store
static int replay_open(idqn_replay* r) {
  const int64_t n_slots = r->n_slots;
  CK(cudaStreamCreateWithFlags(&r->stream, cudaStreamNonBlocking));
  CK(cudaMalloc(&r->action, sizeof(int32_t) * n_slots));
  CK(cudaMalloc(&r->reward, sizeof(double) * n_slots));
  CK(cudaMalloc(&r->terminal, n_slots));
  CK(cudaMalloc(&r->episode_end, n_slots));
  int rc = ensure_slots(r, 256);
  if (rc) return rc;
  CK(cudaEventCreateWithFlags(&r->ev_learner, cudaEventDisableTiming));
  r->learner_slots = new std::vector<int64_t>();
  return IDQN_OK;
}

extern "C" int idqn_replay_create(int64_t n_slots, int64_t state_bytes, int device, idqn_replay** out) {
  REQUIRE(out && n_slots > 0 && state_bytes > 0, "bad argument");
  CK(cudaSetDevice(device));
  int rc = enough_hbm((size_t)n_slots * (2 * state_bytes + 16));
  if (rc) return rc;
  idqn_replay* r = new idqn_replay();
  memset(r, 0, sizeof(*r));
  r->device = device, r->n_slots = n_slots, r->state_bytes = state_bytes;
  rc = replay_open(r);
  if (rc) return rc;
  CK(cudaMalloc(&r->state, (size_t)n_slots * state_bytes));
  CK(cudaMalloc(&r->next_state, (size_t)n_slots * state_bytes));
  *out = r;
  return IDQN_OK;
}

extern "C" int idqn_replay_create_frames(int64_t n_slots, int64_t frame_bytes, int stack, int value_bytes,
                                         int64_t n_frames, int device, idqn_replay** out) {
  REQUIRE(out && n_slots > 0 && frame_bytes > 0 && stack > 0 && value_bytes > 0 && frame_bytes % value_bytes == 0 &&
              n_frames > 0, "bad argument");
  CK(cudaSetDevice(device));
  const int64_t row = 2 * (int64_t)stack;
  int rc = enough_hbm((size_t)n_frames * frame_bytes + (size_t)n_slots * (sizeof(int64_t) * row + 16));
  if (rc) return rc;
  idqn_replay* r = new idqn_replay();
  memset(r, 0, sizeof(*r));
  r->device = device, r->n_slots = n_slots, r->state_bytes = frame_bytes * stack;
  r->frames = 1, r->stack = stack, r->value_bytes = value_bytes, r->frame_bytes = frame_bytes, r->n_frames = n_frames;
  rc = replay_open(r);
  if (rc) return rc;
  CK(cudaMalloc(&r->ring, (size_t)n_frames * frame_bytes));
  CK(cudaMalloc(&r->rows, sizeof(int64_t) * row * n_slots));
  r->h_rows = new int64_t[(size_t)row * n_slots];
  r->inflight_rows = new std::unordered_set<int64_t>();
  r->inflight_frames = new std::unordered_set<int64_t>();
  *out = r;
  return IDQN_OK;
}

extern "C" int idqn_replay_destroy(idqn_replay* r) {
  if (!r) return IDQN_OK;
  cudaSetDevice(r->device);
  cudaStreamSynchronize(r->stream);
  if (r->ev_learner) {
    cudaEventSynchronize(r->ev_learner);
    cudaEventDestroy(r->ev_learner);
  }
  delete r->learner_slots;
  delete r->inflight_rows;
  delete r->inflight_frames;
  delete[] r->h_rows;
  void* ptrs[] = {r->state, r->next_state, r->action, r->reward, r->terminal, r->episode_end, r->d_slots, r->d_gslots,
                  r->ring, r->rows};
  for (void* p : ptrs)
    if (p) cudaFree(p);
  if (r->h_stage) cudaFreeHost(r->h_stage);
  cudaStreamDestroy(r->stream);
  delete r;
  return IDQN_OK;
}

extern "C" int idqn_replay_put(idqn_replay* r, int64_t slot, const void* state, const void* next_state, int32_t action,
                               double reward, uint8_t is_terminal, uint8_t episode_end) {
  REQUIRE(r && state && next_state && slot >= 0 && slot < r->n_slots, "bad argument");
  REQUIRE(!r->frames, "a frame store takes idqn_replay_put_frame / idqn_replay_put_element");
  CK(cudaSetDevice(r->device));
  if (r->learner_pending) {
    // a learner step enqueued by idqn_learn_from_replay may still be reading its sampled slots in place
    if (cudaEventQuery(r->ev_learner) == cudaSuccess) r->learner_pending = 0;
    else if (std::find(r->learner_slots->begin(), r->learner_slots->end(), slot) != r->learner_slots->end())
      CK(cudaStreamWaitEvent(r->stream, r->ev_learner, 0));
  }
  CK(cudaMemcpyAsync(r->state + slot * r->state_bytes, state, r->state_bytes, cudaMemcpyHostToDevice, r->stream));
  CK(cudaMemcpyAsync(r->next_state + slot * r->state_bytes, next_state, r->state_bytes, cudaMemcpyHostToDevice,
                     r->stream));
  CK(cudaMemcpyAsync(r->action + slot, &action, sizeof(int32_t), cudaMemcpyHostToDevice, r->stream));
  CK(cudaMemcpyAsync(r->reward + slot, &reward, sizeof(double), cudaMemcpyHostToDevice, r->stream));
  CK(cudaMemcpyAsync(r->terminal + slot, &is_terminal, 1, cudaMemcpyHostToDevice, r->stream));
  CK(cudaMemcpyAsync(r->episode_end + slot, &episode_end, 1, cudaMemcpyHostToDevice, r->stream));
  CK(cudaStreamSynchronize(r->stream));
  return IDQN_OK;
}

// frame store: a write into `key` of `inflight` (a ring slot or an element row that a step enqueued by
// idqn_learn_from_replay may still read) is ordered after every such step; once they have all completed the sets empty
static int order_after_learner(idqn_replay* r, const std::unordered_set<int64_t>* inflight, int64_t key) {
  if (!r->learner_pending) return IDQN_OK;
  if (cudaEventQuery(r->ev_learner) == cudaSuccess) {
    r->learner_pending = 0;
    r->inflight_rows->clear(), r->inflight_frames->clear();
  } else if (inflight->count(key)) {
    CK(cudaStreamWaitEvent(r->stream, r->ev_learner, 0));
  }
  return IDQN_OK;
}

extern "C" int idqn_replay_put_frame(idqn_replay* r, int64_t frame_id, const void* frame) {
  REQUIRE(r && r->frames && frame && frame_id >= 0, "bad argument");
  CK(cudaSetDevice(r->device));
  const int64_t fs = frame_ring_slot(frame_id, r->n_frames);
  int rc = order_after_learner(r, r->inflight_frames, fs);
  if (rc) return rc;
  CK(cudaMemcpyAsync(r->ring + fs * r->frame_bytes, frame, r->frame_bytes, cudaMemcpyHostToDevice, r->stream));
  CK(cudaStreamSynchronize(r->stream));
  return IDQN_OK;
}

extern "C" int idqn_replay_put_element(idqn_replay* r, int64_t slot, const int64_t* frame_ids, int32_t action,
                                       double reward, uint8_t is_terminal, uint8_t episode_end) {
  REQUIRE(r && r->frames && frame_ids && slot >= 0 && slot < r->n_slots, "bad argument");
  const int64_t w = 2 * (int64_t)r->stack;
  for (int64_t k = 0; k < w; ++k) REQUIRE(frame_ids[k] >= -1, "frame id %lld < -1", (long long)frame_ids[k]);
  CK(cudaSetDevice(r->device));
  int rc = order_after_learner(r, r->inflight_rows, slot);
  if (rc) return rc;
  int64_t* h_row = r->h_rows + slot * w;
  memcpy(h_row, frame_ids, sizeof(int64_t) * w);
  CK(cudaMemcpyAsync(r->rows + slot * w, h_row, sizeof(int64_t) * w, cudaMemcpyHostToDevice, r->stream));
  CK(cudaMemcpyAsync(r->action + slot, &action, sizeof(int32_t), cudaMemcpyHostToDevice, r->stream));
  CK(cudaMemcpyAsync(r->reward + slot, &reward, sizeof(double), cudaMemcpyHostToDevice, r->stream));
  CK(cudaMemcpyAsync(r->terminal + slot, &is_terminal, 1, cudaMemcpyHostToDevice, r->stream));
  CK(cudaMemcpyAsync(r->episode_end + slot, &episode_end, 1, cudaMemcpyHostToDevice, r->stream));
  CK(cudaStreamSynchronize(r->stream));
  return IDQN_OK;
}

extern "C" int idqn_replay_grow_frames(idqn_replay* r, int64_t n_frames, int64_t live_lo, int64_t live_hi) {
  REQUIRE(r && r->frames && n_frames > r->n_frames && live_lo >= 0 && live_lo <= live_hi &&
              live_hi - live_lo <= r->n_frames, "bad argument");
  CK(cudaSetDevice(r->device));
  int rc = enough_hbm((size_t)n_frames * r->frame_bytes);
  if (rc) return rc;
  uint8_t* ring = nullptr;
  CK(cudaMalloc(&ring, (size_t)n_frames * r->frame_bytes));
  // ids [live_lo, live_hi) move from id % F to id % F': runs that wrap in neither ring (at most four)
  for (int64_t id = live_lo; id < live_hi;) {
    const int64_t s = frame_ring_slot(id, r->n_frames), d = frame_ring_slot(id, n_frames);
    const int64_t len = std::min(live_hi - id, std::min(r->n_frames - s, n_frames - d));
    CK(cudaMemcpyAsync(ring + d * r->frame_bytes, r->ring + s * r->frame_bytes, len * r->frame_bytes,
                       cudaMemcpyDeviceToDevice, r->stream));
    id += len;
  }
  // every step still reading the old ring completes before it is freed
  if (r->learner_pending) CK(cudaEventSynchronize(r->ev_learner));
  r->learner_pending = 0;
  r->inflight_rows->clear(), r->inflight_frames->clear();
  CK(cudaStreamSynchronize(r->stream));
  CK(cudaFree(r->ring));
  r->ring = ring, r->n_frames = n_frames;
  return IDQN_OK;
}

extern "C" int idqn_replay_gather_host(idqn_replay* r, const int64_t* slots, int n, void* state, void* next_state,
                                       int32_t* action, double* reward, uint8_t* terminal, uint8_t* episode_end) {
  REQUIRE(r && slots && n > 0 && state && next_state && action && reward && terminal && episode_end, "bad argument");
  for (int i = 0; i < n; ++i) REQUIRE(slots[i] >= 0 && slots[i] < r->n_slots, "slot %lld out of range", (long long)slots[i]);
  CK(cudaSetDevice(r->device));
  if (n > r->cap_gslots) {
    if (r->d_gslots) CK(cudaFree(r->d_gslots));
    r->cap_gslots = std::max(n, 256);
    CK(cudaMalloc(&r->d_gslots, sizeof(int64_t) * r->cap_gslots));
  }
  int rc = IDQN_OK;
  // device-side staging for the packed batch
  const size_t sb = (size_t)n * r->state_bytes;
  const size_t off_next = (sb + 255) / 256 * 256;
  const size_t off_act = off_next + (sb + 255) / 256 * 256;
  const size_t off_rew = off_act + ((size_t)n * 4 + 255) / 256 * 256;
  const size_t off_term = off_rew + ((size_t)n * 8 + 255) / 256 * 256;
  const size_t off_end = off_term + ((size_t)n + 255) / 256 * 256;
  const size_t total = off_end + ((size_t)n + 255) / 256 * 256;
  uint8_t* d_stage = nullptr;
  CK(cudaMallocAsync((void**)&d_stage, total, r->stream));
  CK(cudaMemcpyAsync(r->d_gslots, slots, sizeof(int64_t) * n, cudaMemcpyHostToDevice, r->stream));
  GatherArgs a;
  memset(&a, 0, sizeof(a));
  a.n = n;
  a.o_state = d_stage, a.o_next = d_stage + off_next, a.o_action = (int32_t*)(d_stage + off_act);
  a.o_reward_f64 = (double*)(d_stage + off_rew), a.o_terminal = d_stage + off_term, a.o_episode_end = d_stage + off_end;
  rc = launch_gather(r, a, r->stream, r->d_gslots);
  if (rc) return rc;
  CK(cudaMemcpyAsync(state, a.o_state, sb, cudaMemcpyDeviceToHost, r->stream));
  CK(cudaMemcpyAsync(next_state, a.o_next, sb, cudaMemcpyDeviceToHost, r->stream));
  CK(cudaMemcpyAsync(action, a.o_action, sizeof(int32_t) * n, cudaMemcpyDeviceToHost, r->stream));
  CK(cudaMemcpyAsync(reward, a.o_reward_f64, sizeof(double) * n, cudaMemcpyDeviceToHost, r->stream));
  CK(cudaMemcpyAsync(terminal, a.o_terminal, n, cudaMemcpyDeviceToHost, r->stream));
  CK(cudaMemcpyAsync(episode_end, a.o_episode_end, n, cudaMemcpyDeviceToHost, r->stream));
  CK(cudaFreeAsync(d_stage, r->stream));
  CK(cudaStreamSynchronize(r->stream));
  return IDQN_OK;
}

// the step just enqueued on the learner's stream reads `slots` of the store asynchronously: remember them (and an event
// behind the step) so that idqn_replay_put orders a write into one of them after the read.  A frame store remembers the
// rows and ring slots of every step since the event last completed (the event is behind the newest of them).
static int note_learner_read(idqn_handle* h, idqn_replay* r, const int64_t* slots, int n) {
  if (r->frames) {
    if (!r->learner_pending || cudaEventQuery(r->ev_learner) == cudaSuccess)
      r->inflight_rows->clear(), r->inflight_frames->clear();
    const int64_t w = 2 * (int64_t)r->stack;
    for (int i = 0; i < n; ++i) {
      r->inflight_rows->insert(slots[i]);
      for (int64_t k = 0; k < w; ++k) {
        const int64_t id = r->h_rows[slots[i] * w + k];
        if (id >= 0) r->inflight_frames->insert(frame_ring_slot(id, r->n_frames));
      }
    }
  } else {
    r->learner_slots->assign(slots, slots + n);
  }
  CK(cudaEventRecord(r->ev_learner, h->stream));
  r->learner_pending = 1;
  return IDQN_OK;
}

extern "C" int idqn_learn_from_replay(idqn_handle* h, idqn_replay* r, const int64_t* slots, int n, int u8,
                                      float* losses) {
  REQUIRE(h && r && slots, "null argument");
  REQUIRE(n == h->B, "sample size %d != learner batch size %d", n, h->B);
  REQUIRE(r->device == h->cfg.device, "replay store and learner live on different devices");
  REQUIRE(r->state_bytes == h->in_elems * (u8 ? 1 : 4), "element size mismatch: store %lld bytes, learner %lld",
          (long long)r->state_bytes, (long long)(h->in_elems * (u8 ? 1 : 4)));
  REQUIRE(!r->frames || r->value_bytes == (u8 ? 1 : 4), "frame store of %d-byte values fed as %s", r->value_bytes,
          u8 ? "uint8" : "float32");
  for (int i = 0; i < n; ++i) REQUIRE(slots[i] >= 0 && slots[i] < r->n_slots, "slot %lld out of range", (long long)slots[i]);
  CK(cudaSetDevice(h->cfg.device));
  int rc = ensure_slots(r, n);
  if (rc) return rc;
  CK(cudaMemcpyAsync(r->d_slots, slots, sizeof(int64_t) * n, cudaMemcpyHostToDevice, h->stream));
  if (h->img_on && u8) {
    // image path: its first kernel (space-to-depth) reads the frames from the replay slots in place and gathers the
    // scalars; the graph of this staging set is re-captured if the store or its index buffer changed
    // (a frame store: also after its ring grew)
    if (h->rsrc.state != r->state || h->rsrc.slots != r->d_slots || h->rsrc.ring != r->ring ||
        h->rsrc.rows != r->rows || h->rsrc.n_frames != r->n_frames) {
      for (int i = 6; i < 8; ++i)
        if (h->graph[i]) {
          CK(cudaGraphExecDestroy(h->graph[i]));
          h->graph[i] = nullptr;
        }
    }
    h->rsrc.state = r->state, h->rsrc.next_state = r->next_state, h->rsrc.slots = r->d_slots;
    h->rsrc.state_bytes = r->state_bytes, h->rsrc.action = r->action, h->rsrc.reward = r->reward, h->rsrc.terminal = r->terminal;
    h->rsrc.ring = r->ring, h->rsrc.rows = r->rows, h->rsrc.n_frames = r->n_frames;
    h->rsrc.frame_bytes = r->frame_bytes, h->rsrc.stack = r->stack;
    h->rsrc_on = 1, h->graph_set = 3;
    rc = idqn_learn_step_resident(h, u8, losses);
    h->rsrc_on = 0, h->graph_set = 0;
    if (rc) return rc;
    return note_learner_read(h, r, slots, n);
  }
  GatherArgs a;
  memset(&a, 0, sizeof(a));
  a.n = n;
  a.o_state = (uint8_t*)h->s, a.o_next = (uint8_t*)h->s2, a.o_action = h->action, a.o_reward_f32 = h->reward;
  a.o_terminal = h->terminal;
  rc = launch_gather(r, a, h->stream, r->d_slots);
  if (rc) return rc;
  rc = idqn_learn_step_resident(h, u8, losses);
  if (rc) return rc;
  return note_learner_read(h, r, slots, n);
}
