// Checkpoint support of the replay store: bulk host <-> device transfer of the frame ring and of the element slots, and
// a digest of the store computed where it lives.
//
// The reference saves no replay buffer (its ReplayBuffer(checkpoint_duration=...) argument is stored and never used,
// replay_buffer.py:82,93); here the store lives in HBM behind this ABI, so saving and restoring it needs these calls.
// Every transfer first waits for the store's stream and for the learner steps that may still read the store, then
// moves the bytes in chunks through one pinned staging buffer owned by the store (the caller's buffers may be pageable).
//
// The digest of a logical byte stream of length L, zero-padded to N little-endian 64-bit words w_i, is
//   ( sum_i splitmix64(w_i + (i + 1) * 0x9E3779B97F4A7C15) ) mod 2^64  XOR  splitmix64(L)
// Integer addition is associative, so it does not depend on the grid or on the order in which blocks finish, and a
// ring is digested at the logical word offsets of its frames, so the value does not depend on the ring's size.
#include "common.cuh"

#include <algorithm>

#define CKPT_STAGE_BYTES ((size_t)64 << 20)
#define DIGEST_GOLDEN 0x9E3779B97F4A7C15ull

__host__ __device__ __forceinline__ unsigned long long splitmix64(unsigned long long z) {
  z ^= z >> 30;
  z *= 0xBF58476D1CE4E5B9ull;
  z ^= z >> 27;
  z *= 0x94D049BB133111EBull;
  z ^= z >> 31;
  return z;
}

// nothing enqueued on the store's stream and no learner step that may read the store is still running
static int quiesce(idqn_replay* r) {
  CK(cudaSetDevice(r->device));
  if (r->learner_pending) CK(cudaEventSynchronize(r->ev_learner));
  r->learner_pending = 0;
  r->learner_slots->clear();
  if (r->frames) r->inflight_rows->clear(), r->inflight_frames->clear();
  CK(cudaStreamSynchronize(r->stream));
  return IDQN_OK;
}

static int ensure_stage(idqn_replay* r) {
  if (r->h_stage_bytes >= CKPT_STAGE_BYTES) return IDQN_OK;
  if (r->h_stage) CK(cudaFreeHost(r->h_stage));
  r->h_stage = nullptr, r->h_stage_bytes = 0;
  CK(cudaMallocHost(&r->h_stage, CKPT_STAGE_BYTES));
  r->h_stage_bytes = CKPT_STAGE_BYTES;
  return IDQN_OK;
}

// n bytes between device memory and (pageable) host memory, through the staging buffer
static int copy_chunked(idqn_replay* r, void* dev, void* host, size_t n, bool to_host) {
  if (n == 0) return IDQN_OK;
  int rc = ensure_stage(r);
  if (rc) return rc;
  uint8_t* d = (uint8_t*)dev;
  uint8_t* hp = (uint8_t*)host;
  for (size_t off = 0; off < n; off += r->h_stage_bytes) {
    const size_t len = std::min(r->h_stage_bytes, n - off);
    if (to_host) {
      CK(cudaMemcpyAsync(r->h_stage, d + off, len, cudaMemcpyDeviceToHost, r->stream));
      CK(cudaStreamSynchronize(r->stream));
      memcpy(hp + off, r->h_stage, len);
    } else {
      memcpy(r->h_stage, hp + off, len);
      CK(cudaMemcpyAsync(d + off, r->h_stage, len, cudaMemcpyHostToDevice, r->stream));
      CK(cudaStreamSynchronize(r->stream));
    }
  }
  return IDQN_OK;
}

static int transfer_frames(idqn_replay* r, int64_t id_lo, int64_t id_hi, void* host, bool to_host) {
  REQUIRE(r && r->frames && host && id_lo >= 0 && id_lo <= id_hi, "bad argument");
  REQUIRE(id_hi - id_lo <= r->n_frames, "%lld frames requested from a ring of %lld", (long long)(id_hi - id_lo),
          (long long)r->n_frames);
  int rc = quiesce(r);
  if (rc) return rc;
  // at most two runs: [id_lo, end of the ring) and the wrapped rest from slot 0
  const int64_t n = id_hi - id_lo, s = frame_ring_slot(id_lo, r->n_frames);
  const int64_t first = std::min(n, r->n_frames - s);
  rc = copy_chunked(r, r->ring + s * r->frame_bytes, host, (size_t)(first * r->frame_bytes), to_host);
  if (rc) return rc;
  return copy_chunked(r, r->ring, (uint8_t*)host + first * r->frame_bytes, (size_t)((n - first) * r->frame_bytes),
                      to_host);
}

extern "C" int idqn_replay_read_frames(idqn_replay* r, int64_t id_lo, int64_t id_hi, void* dst) {
  return transfer_frames(r, id_lo, id_hi, dst, true);
}
extern "C" int idqn_replay_write_frames(idqn_replay* r, int64_t id_lo, int64_t id_hi, const void* src) {
  return transfer_frames(r, id_lo, id_hi, const_cast<void*>(src), false);
}

static int transfer_slots(idqn_replay* r, int64_t slot_lo, int64_t n, void* state_or_rows, void* next_state,
                          void* action, void* reward, void* terminal, void* episode_end, bool to_host) {
  REQUIRE(r && slot_lo >= 0 && n >= 0 && slot_lo + n <= r->n_slots, "slots [%lld, %lld) outside the store",
          (long long)slot_lo, (long long)(slot_lo + n));
  REQUIRE(state_or_rows && action && reward && terminal && episode_end, "null argument");
  REQUIRE(r->frames ? next_state == nullptr : next_state != nullptr,
          r->frames ? "a frame store has no next_state stacks: pass NULL" : "null next_state");
  int rc = quiesce(r);
  if (rc) return rc;
  if (r->frames) {
    const int64_t w = 2 * (int64_t)r->stack;
    rc = copy_chunked(r, r->rows + slot_lo * w, state_or_rows, sizeof(int64_t) * w * n, to_host);
    if (rc) return rc;
    if (!to_host) memcpy(r->h_rows + slot_lo * w, state_or_rows, sizeof(int64_t) * w * n);
  } else {
    const size_t sb = (size_t)r->state_bytes;
    rc = copy_chunked(r, r->state + slot_lo * sb, state_or_rows, sb * n, to_host);
    if (!rc) rc = copy_chunked(r, r->next_state + slot_lo * sb, next_state, sb * n, to_host);
    if (rc) return rc;
  }
  rc = copy_chunked(r, r->action + slot_lo, action, sizeof(int32_t) * n, to_host);
  if (!rc) rc = copy_chunked(r, r->reward + slot_lo, reward, sizeof(double) * n, to_host);
  if (!rc) rc = copy_chunked(r, r->terminal + slot_lo, terminal, n, to_host);
  if (!rc) rc = copy_chunked(r, r->episode_end + slot_lo, episode_end, n, to_host);
  return rc;
}

extern "C" int idqn_replay_read_slots(idqn_replay* r, int64_t slot_lo, int64_t n, void* state_or_rows,
                                      void* next_state, int32_t* action, double* reward, uint8_t* terminal,
                                      uint8_t* episode_end) {
  return transfer_slots(r, slot_lo, n, state_or_rows, next_state, action, reward, terminal, episode_end, true);
}
extern "C" int idqn_replay_write_slots(idqn_replay* r, int64_t slot_lo, int64_t n, const void* state_or_rows,
                                       const void* next_state, const int32_t* action, const double* reward,
                                       const uint8_t* terminal, const uint8_t* episode_end) {
  return transfer_slots(r, slot_lo, n, const_cast<void*>(state_or_rows), const_cast<void*>(next_state),
                        const_cast<int32_t*>(action), const_cast<double*>(reward), const_cast<uint8_t*>(terminal),
                        const_cast<uint8_t*>(episode_end), false);
}

// ---------------------------------------------------------------------------------------------
// One logical byte stream: either `bytes` contiguous bytes at `base`, or (ring != null) `n_ids` frames of frame_bytes
// starting at frame id id_lo, each padded with zeros to `words_per_frame` words.
struct DigestStream {
  const uint8_t* base;
  int64_t bytes;
  const uint8_t* ring;
  int64_t n_frames, frame_bytes, id_lo, n_ids, words_per_frame;
  int64_t n_words;
};
struct DigestArgs {
  DigestStream s[6];
  unsigned long long* out;  // [6] partial sums (splitmix64(L) is applied on the host)
};

// the little-endian word of bytes [0, avail) at p (avail < 8: zero-padded)
__device__ __forceinline__ unsigned long long load_word(const uint8_t* p, int64_t avail) {
  if (avail >= 8 && (reinterpret_cast<uintptr_t>(p) & 7) == 0) return __ldcs(reinterpret_cast<const unsigned long long*>(p));
  unsigned long long w = 0;
  const int n = (int)(avail < 8 ? avail : 8);
  for (int b = 0; b < n; ++b) w |= (unsigned long long)p[b] << (8 * b);
  return w;
}

// grid: (blocks, 6) -- blockIdx.y is the array; grid-stride loop over its words, one atomic add per block
__global__ void __launch_bounds__(256) replay_digest_kernel(const DigestArgs a) {
  const DigestStream& s = a.s[blockIdx.y];
  unsigned long long acc = 0;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < s.n_words; i += (int64_t)gridDim.x * blockDim.x) {
    unsigned long long w;
    if (s.ring) {
      const int64_t f = i / s.words_per_frame, o = (i - f * s.words_per_frame) * 8;
      const uint8_t* fp = s.ring + frame_ring_slot(s.id_lo + f, s.n_frames) * s.frame_bytes;
      w = load_word(fp + o, s.frame_bytes - o);
    } else {
      w = load_word(s.base + i * 8, s.bytes - i * 8);
    }
    acc += splitmix64(w + (unsigned long long)(i + 1) * DIGEST_GOLDEN);
  }
#pragma unroll
  for (int d = 16; d > 0; d >>= 1) acc += __shfl_down_sync(0xffffffffu, acc, d);
  __shared__ unsigned long long warp_sum[8];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (lane == 0) warp_sum[warp] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    unsigned long long t = 0;
    for (int k = 0; k < (int)(blockDim.x >> 5); ++k) t += warp_sum[k];
    if (t) atomicAdd(&a.out[blockIdx.y], t);
  }
}

static void contiguous(DigestStream& s, const void* base, int64_t bytes) {
  memset(&s, 0, sizeof(s));
  s.base = (const uint8_t*)base, s.bytes = bytes, s.n_words = (bytes + 7) / 8;
}

extern "C" int idqn_replay_digest(idqn_replay* r, int64_t n_live, int64_t id_lo, int64_t id_hi, uint64_t* out) {
  REQUIRE(r && out && n_live >= 0 && n_live <= r->n_slots, "bad argument");
  REQUIRE(!r->frames || (id_lo >= 0 && id_lo <= id_hi && id_hi - id_lo <= r->n_frames), "bad frame id range");
  CK(cudaSetDevice(r->device));
  DigestArgs a;
  memset(&a, 0, sizeof(a));
  int64_t len[6];
  if (r->frames) {
    DigestStream& f = a.s[0];
    f.ring = r->ring, f.n_frames = r->n_frames, f.frame_bytes = r->frame_bytes;
    f.id_lo = id_lo, f.n_ids = id_hi - id_lo, f.words_per_frame = (r->frame_bytes + 7) / 8;
    f.n_words = f.n_ids * f.words_per_frame;
    len[0] = f.n_words * 8;  // every frame padded to a multiple of 8 bytes
    contiguous(a.s[1], r->rows, (int64_t)sizeof(int64_t) * 2 * r->stack * n_live);
  } else {
    contiguous(a.s[0], r->state, r->state_bytes * n_live);
    contiguous(a.s[1], r->next_state, r->state_bytes * n_live);
    len[0] = a.s[0].bytes;
  }
  contiguous(a.s[2], r->action, (int64_t)sizeof(int32_t) * n_live);
  contiguous(a.s[3], r->reward, (int64_t)sizeof(double) * n_live);
  contiguous(a.s[4], r->terminal, n_live);
  contiguous(a.s[5], r->episode_end, n_live);
  for (int i = 1; i < 6; ++i) len[i] = a.s[i].bytes;
  int64_t most = 0;
  for (int i = 0; i < 6; ++i) most = std::max(most, a.s[i].n_words);
  unsigned long long* d_out = nullptr;
  CK(cudaMallocAsync((void**)&d_out, sizeof(unsigned long long) * 6, r->stream));
  CK(cudaMemsetAsync(d_out, 0, sizeof(unsigned long long) * 6, r->stream));
  a.out = d_out;
  const int blocks = (int)std::min<int64_t>(std::max<int64_t>((most + 255) / 256, 1), 4 * 148);
  replay_digest_kernel<<<dim3(blocks, 6), 256, 0, r->stream>>>(a);
  CK(cudaGetLastError());
  unsigned long long h_out[6];
  CK(cudaMemcpyAsync(h_out, d_out, sizeof(h_out), cudaMemcpyDeviceToHost, r->stream));
  CK(cudaFreeAsync(d_out, r->stream));
  CK(cudaStreamSynchronize(r->stream));
  for (int i = 0; i < 6; ++i) out[i] = (uint64_t)h_out[i] ^ splitmix64((unsigned long long)len[i]);
  return IDQN_OK;
}

extern "C" void* idqn_replay_stream(idqn_replay* r) { return r ? (void*)r->stream : nullptr; }
