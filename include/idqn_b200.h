/*
 * idqn_b200.h — C ABI of libidqn_b200.so, the B200 (sm_100a) implementation of the i-DQN
 * iterated-Bellman learning step and its data feed.
 *
 * The reference (theovincent/i-DQN) has no FFI layer: its boundary is the Python class API of
 * slimdqn/networks and slimdqn/sample_collection.  Each entry point below names the reference
 * interface (file:line under the reference tree) it replaces; the Python package `idqn_b200`
 * binds them with ctypes and re-exposes the reference's class API (see INTEGRATION.md).
 *
 * Conventions
 *   - every function returns 0 on success, a negative IDQN_E* code on failure and never throws;
 *     idqn_last_error() returns a thread-local message for the last failure;
 *   - pointers named *_host are host memory, *_dev are device memory of the handle's device;
 *     the caller keeps them alive for the duration of the call;
 *   - a handle owns all its device memory and one CUDA stream; one host thread drives one handle;
 *   - parameters cross the boundary as flat float32 arrays per head in the "arena" layout
 *     described by idqn_leaf_info(): layers in flax creation order, kernel then bias, kernel
 *     stored exactly as flax stores it ([kh,kw,in,out] / [in,out], row-major).
 */
#ifndef IDQN_B200_H
#define IDQN_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define IDQN_OK 0
#define IDQN_EINVAL (-1)   /* bad argument / unsupported configuration */
#define IDQN_ECUDA (-2)    /* a CUDA runtime call or kernel failed */
#define IDQN_ERANGE (-3)   /* sum-tree query target outside [0, root)  (sum_tree.py:73-74 ValueError) */
#define IDQN_EASSERT (-4)  /* reference assertion would fire (sum_tree.py:30-31,81) */
#define IDQN_ENOMEM (-5)

#define IDQN_ARCH_FC 0     /* architectures/dqn.py:61-63 */
#define IDQN_ARCH_CNN 1    /* architectures/dqn.py:39-53 */
#define IDQN_ARCH_IMPALA 2 /* architectures/dqn.py:7-29,54-60: three residual stacks (fp32 CUDA-core kernels; not a benchmark config) */
#define IDQN_MAX_FEATURES 8

/* which per-head arena a transfer addresses */
#define IDQN_ONLINE 0      /* iDQN.params          idqn.py:48 */
#define IDQN_TARGET 1      /* iDQN.target_params   idqn.py:56 */
#define IDQN_MU 2          /* ScaleByAdamState.mu  idqn.py:53 */
#define IDQN_NU 3          /* ScaleByAdamState.nu  idqn.py:53 */
#define IDQN_GRAD 4        /* d loss_k / d params[k] of the last step (read-only; debug/parity) */

typedef struct idqn_config {
  int32_t arch;                         /* IDQN_ARCH_* */
  int32_t obs[3];                       /* cnn: H,W,C (stack last); fc: {dim,1,1} */
  int32_t n_actions;
  int32_t n_heads;                      /* K heads held by THIS handle (idqn.py:44) */
  int32_t n_features;
  int32_t features[IDQN_MAX_FEATURES];  /* DQNNet.features (architectures/dqn.py:32) */
  int32_t batch_size;                   /* B of learn_on_batch (samples per step) */
  float learning_rate;                  /* optax.adam(lr, eps) idqn.py:52 */
  float adam_eps;
  float gamma_n;                        /* gamma ** update_horizon (idqn.py:122) rounded to f32 */
  int32_t device;                       /* CUDA device ordinal */
  int32_t flags;                        /* IDQN_F_* */
} idqn_config;

#define IDQN_F_NO_GRAPH 1   /* launch kernels directly instead of replaying the captured CUDA graph */
#define IDQN_F_SIMT_ONLY 2  /* force the fp32 CUDA-core GEMM path for every layer (cross-check mode) */
#define IDQN_F_NO_PDL 16    /* launch the step's kernels WITHOUT programmatic dependent launch (default on: 0.353 vs 0.358 ms/step) */
#define IDQN_F_NO_IMG 8     /* disable the image-resident TMA conv kernels (generic tcgen05 implicit GEMM instead) */
#define IDQN_F_KEEP_GRADS 4 /* materialise every gradient in the IDQN_GRAD arena (disables fused wgrad+Adam) */
#define IDQN_F_PARTITION 32 /* backward pass on two SM partitions (green contexts): conv chain | Dense_0 wgrad+Adam.  Measured slower than the single-stream order on B200 (both sides are per-SM latency bound): off by default */
#define IDQN_F_SLOW_APPLY 512 /* best_action through the generic batch-1 kernels instead of the step's own kernels */
#define IDQN_F_NO_DEFER 256 /* Dense_0 wgrad+Adam right after its data gradient instead of at the end of the backward pass */
#define IDQN_F_NO_FORK 128  /* keep the conv weight-gradient kernels on the main stream (no second graph branch) */
#define IDQN_F_CHAIN 2048 /* conv1 and conv2 forward as ONE kernel (conv_chain_fwd_kernel: a (net, image) unit goes through both layers in one CTA, the intermediate image stays in shared memory).  Bit-identical; measured not faster than the two launches: off by default */
#define IDQN_F_TIMELINE 1024 /* kernels stamp the global timer at first-CTA start / last-CTA end: idqn_kernel_timeline reads the true in-graph schedule */
#define IDQN_F_OLD_WGRAD 64 /* Dense_0 wgrad+Adam on the generic tcgen05 kernel (Adam in its epilogue) instead of the TMA pipeline */

typedef struct idqn_handle idqn_handle;

const char* idqn_last_error(void);
int idqn_version(void);

/* iDQN.__init__ / DQN.__init__ (idqn.py:28-63, dqn.py:14-39): allocates K online + K target arenas,
 * Adam state (count=0, mu=nu=0) and all workspaces.  Parameters start at zero; the host uploads them. */
int idqn_create(const idqn_config* cfg, idqn_handle** out);
int idqn_destroy(idqn_handle* h);

/* arena description: floats per head (padded), number of leaves, and per leaf its offset/shape.
 * Leaf 2*l is layer l's kernel, leaf 2*l+1 its bias; name is "Conv_i"/"Dense_i" (flax auto-naming). */
int64_t idqn_arena_stride(const idqn_handle* h);
int idqn_leaf_count(const idqn_handle* h);
int idqn_leaf_info(const idqn_handle* h, int leaf, int64_t* offset, int64_t* size, int32_t shape[4],
                   int32_t* ndim, char name[16]);

/* host <-> device transfer of n floats at `offset` of head `head` of arena `which` */
int idqn_upload(idqn_handle* h, int which, int head, int64_t offset, const float* src_host, int64_t n);
int idqn_download(idqn_handle* h, int which, int head, int64_t offset, float* dst_host, int64_t n);
/* debug/parity: hidden activations (relu outputs) of the last step; net in [0,K) = online head on `state`,
 * [K,2K) = target head on `next_state`; layer in [0, n_layers-1); n floats (<= B*OH*OW*OC) */
int idqn_download_activation(idqn_handle* h, int net, int layer, float* dst_host, int64_t n);
int idqn_set_count(idqn_handle* h, const int32_t* count_host);  /* ScaleByAdamState.count[K] */
int idqn_get_count(idqn_handle* h, int32_t* count_host);
/* raw device pointer of an arena ([K][stride] floats) for zero-copy interop (NCCL / peer copies) */
void* idqn_arena_ptr(idqn_handle* h, int which);
/* after writing an online/target arena through idqn_arena_ptr (NCCL recv, peer copy): its bf16 operand planes are
 * rebuilt before the next step */
int idqn_mark_planes_dirty(idqn_handle* h, int which);
int idqn_mark_head_planes_dirty(idqn_handle* h, int which, int head);  /* one head only (neighbour exchange of the sharded agent) */
void* idqn_stream(idqn_handle* h);

/* iDQN.learn_on_batch (idqn.py:96-109) / DQN.learn_on_batch (dqn.py:60-72) on the handle's resident state:
 * one gradient step of all K heads on one shared batch; per-head MSE TD loss written to losses_host[K]
 * (may be NULL: losses stay on the device and are accumulated, see idqn_read_cumulated_losses).
 * state/next_state: [B, obs...] uint8 (state_is_u8=1) or float32; action int32[B]; reward float32[B];
 * is_terminal uint8[B].  The *_host variant includes the H2D copies (end-to-end path). */
int idqn_learn_on_batch_host(idqn_handle* h, const void* state_host, const void* next_state_host,
                             int state_is_u8, const int32_t* action_host, const float* reward_host,
                             const uint8_t* is_terminal_host, float* losses_host);
int idqn_learn_on_batch_dev(idqn_handle* h, const void* state_dev, const void* next_state_dev, int state_is_u8,
                            const int32_t* action_dev, const float* reward_dev, const uint8_t* is_terminal_dev,
                            float* losses_host);
/* The same step as idqn_learn_on_batch_host, pipelined the way the reference's own call is (jax dispatches
 * learn_on_batch asynchronously and idqn.py:72 only accumulates device futures): submit returns as soon as the copies
 * and the step are enqueued -- the H2D copies of batch t+1 run on a copy stream while step t computes -- and
 * idqn_wait_losses blocks until the step of `ticket` has finished and returns its K losses.  At most two steps are in
 * flight (submit waits for ticket-2); host buffers must stay valid until idqn_wait_losses(ticket) returns (pinned
 * buffers make the copies truly asynchronous). */
int idqn_submit_batch_host(idqn_handle* h, const void* state_host, const void* next_state_host, int state_is_u8,
                           const int32_t* action_host, const float* reward_host, const uint8_t* is_terminal_host,
                           int64_t* ticket);
int idqn_wait_losses(idqn_handle* h, int64_t ticket, float* losses_host);
/* idqn.py:72: only update_online_params adds a step's losses to the running sums; a direct learn_on_batch call does not.
 * on = 0 makes the following steps leave the sums alone (stream-ordered; default on = 1) */
int idqn_set_loss_accumulation(idqn_handle* h, int on);
/* |Q(s_b,a_b) - y_b| per head and sample of the most recent step, float32 [K][B]: the priorities a prioritised replay buffer
 * is updated with (replay_buffer.py:232-237) */
int idqn_read_td_abs(idqn_handle* h, float* out_host);
/* idqn.py:72,82-87: device-side sum of the per-head losses since the last reset */
int idqn_read_cumulated_losses(idqn_handle* h, double* sums_host, int reset);
/* its inverse (restore of a checkpoint): the K sums become sums_host */
int idqn_write_cumulated_losses(idqn_handle* h, const double* sums_host);

/* measurement aids (no reference counterpart): kernels one step launches, and one un-graphed step with a CUDA
 * event after every launch -> ms[i] / names[32*i..] per kernel, in launch order.  It runs on the batch the LAST host-batch
 * learning call staged: call it only after at least one idqn_learn_on_batch_host (a never-fed handle's staging buffers are
 * uninitialised device memory, and like idqn_learn_on_batch_dev the step does not validate the action indices it is given) */
int idqn_kernels_per_step(idqn_handle* h);
int idqn_profile_step(idqn_handle* h, int state_is_u8, int max_entries, float* ms, char* names, int* n_out);
/* IDQN_F_TIMELINE handles: global-timer stamps (ns) of the kernels of the most recent step in launch order, out[2*i] =
 * start of the first CTA, out[2*i+1] = end of the last CTA, names[32*i..] the kernel tag; resets the slots */
int idqn_kernel_timeline(idqn_handle* h, unsigned long long* out, char* names, int max_entries, int* n_out);
/* IDQN_F_TIMELINE: per-CTA global-timer stamps {entry, first operand landed, last MMA committed, exit} of the conv kernel in
 * timeline slot `slot` (launch index inside the step), recorded by the steps that follow; reads back what was recorded since
 * the previous call (out may be NULL) */
int idqn_cta_timeline(idqn_handle* h, int slot, unsigned long long* out, int max_ctas, int* n_out);
/* CTAs the graph-replayed step gives the Dense_0 update kernel while it runs next to the conv backward chain (0: it runs
 * after the chain on every SM) -- bench.py reports the kernel's in-step bandwidth next to its stand-alone roofline */
int idqn_dense_update_ctas(idqn_handle* h);
/* n > 0: that many CTAs; 0: the update runs after the chain on every SM; < 0: automatic (min(80, 54 + 6 K) on 148 SMs).  Before the first step. */
int idqn_set_dense_update_ctas(idqn_handle* h, int n);
/* pipeline timeline of CTA 0 of the kernel named by the IDQN_TL environment variable (fwd0..2, dgrad1..2, wgrad0..2,
 * dfwd3, ddgrad3) during the most recent step: entries (clock64 << 16 | tag), 0 = unused; returns the entry count */
int idqn_debug_timeline(unsigned long long* out, int max_entries);

/* shift_params (idqn.py:13-17), sync_target_params (idqn.py:20-24), target_params = params.copy() (idqn.py:78) */
int idqn_shift_params(idqn_handle* h);
int idqn_sync_target(idqn_handle* h);
int idqn_copy_online_to_target(idqn_handle* h);

/* ------------------------------------------------------------------------------------------------
 * Head-sharded chain over the GPUs of one box (one process per GPU): shift_params / sync_target_params
 * (idqn.py:13-24) act on the GLOBAL head index, so at the target events of idqn.py:74-94 one boundary head crosses
 * to the neighbouring rank.  Each rank exports CUDA-IPC handles of its arenas (idqn_peer_create fills a blob of
 * idqn_peer_export_size() bytes; the host exchanges the blobs by any means), maps its neighbours'
 * (idqn_peer_connect; NULL at the ends of the chain) and from then on the events are enqueued on the handle's stream:
 * the boundary head is PUSHED into the neighbour's slot by a kernel storing to peer memory over NVLink, ordered by
 * flags in peer memory -- no host synchronisation, no collective library on the event path. */
typedef struct idqn_peer idqn_peer;
int idqn_peer_export_size(void);
int idqn_peer_create(idqn_handle* h, idqn_peer** out, void* export_blob);
int idqn_peer_connect(idqn_peer* p, const void* prev_blob, const void* next_blob);
int idqn_peer_destroy(idqn_peer* p);
int idqn_peer_sync_target(idqn_peer* p);   /* idqn.py:91-92 sync_target_params across the shards */
int idqn_peer_shift_params(idqn_peer* p);  /* idqn.py:75-80 target <- online, then shift_params across the shards */

/* network.apply (architectures/dqn.py:37-70) of head `head` of arena `which` on n inputs -> q_host[n, A] */
int idqn_apply_host(idqn_handle* h, int which, int head, const void* x_host, int x_is_u8, int n, float* q_host);
/* iDQN.best_action (idqn.py:126-131) / DQN.best_action (dqn.py:89-92) with the head index made explicit:
 * argmax_a Q(params[head], state) for ONE state (float32 holding 0..255 for Atari, atari.py:43-45, or uint8) */
int idqn_best_action(idqn_handle* h, int which, int head, const void* state_host, int state_is_u8, int32_t* action);

/* select_action (slimdqn/sample_collection/utils.py:8-15) in ONE call: the three jax.random draws of the step (threefry2x32,
 * restated on the host in C), and -- only on a greedy step -- best_action of the drawn head as one CUDA-graph launch.
 * key0/key1: the uint32[2] jax key; info (optional, int32[2]): {explored, head}. */
int idqn_select_action(idqn_handle* h, const void* state_host, int state_is_u8, uint32_t key0, uint32_t key1,
                       int n_actions, float epsilon, int32_t* action, int32_t* info);
/* N independent select_action draws (slimdqn/sample_collection/utils.py:8-15, head draw idqn.py:126-131) in ONE call:
 * env i makes exactly the draws of idqn_select_action with the key (keys[2i], keys[2i+1]).  states: n * in_elems values
 * (uint8 if state_is_u8, else float32); actions: [n]; info (optional): [n][2] = {explored, head}.  No device work when
 * every environment explores; otherwise, at Atari shapes with uint8 states, one CUDA-graph launch per chunk of up to
 * batch_size environments (the online heads' forward of the chunk's states and the per-environment argmax of the drawn
 * head's Q row) and one host synchronisation at the end.  Q rows are bit-identical to idqn_best_action's.  Ordered
 * after every learning step enqueued before it.  IDQN_EINVAL for n < 0 or n_actions <= 0. */
int idqn_select_actions(idqn_handle* h, const void* states_host, int state_is_u8, int n, const uint32_t* keys,
                        int n_actions, float epsilon, int32_t* actions, int32_t* info);
/* the draws themselves (tests / host mirrors): what = 0 split(key, a) -> out[2a]; 1 uniform(key) -> float32 bits in out[0];
 * 2 randint(key, (), a, b) -> out[0] */
int idqn_prng(int what, uint32_t key0, uint32_t key1, int32_t a, int32_t b, uint32_t* out);

/* ------------------------------------------------------------------------------------------------
 * SumTree (slimdqn/sample_collection/sum_tree.py:8-102): float64 nodes resident on the device.
 * set/query reproduce the reference's arithmetic bit for bit (ordered per-ancestor adds, strict <). */
typedef struct idqn_sumtree idqn_sumtree;
int idqn_sumtree_create(int64_t capacity, int device, idqn_sumtree** out);     /* sum_tree.py:11-18 */
int idqn_sumtree_destroy(idqn_sumtree* t);
int idqn_sumtree_depth(const idqn_sumtree* t);
int64_t idqn_sumtree_num_nodes(const idqn_sumtree* t);
/* sum_tree.py:20-47; indices need not be unique (first occurrence wins) nor sorted */
int idqn_sumtree_set(idqn_sumtree* t, const int32_t* indices_host, const double* values_host, int64_t n);
int idqn_sumtree_get(idqn_sumtree* t, const int32_t* indices_host, double* values_host, int64_t n); /* :49-51 */
int idqn_sumtree_root(idqn_sumtree* t, double* root_host);                                          /* :53-56 */
/* sum_tree.py:58-102; IDQN_ERANGE if any target is outside [0, root) */
int idqn_sumtree_query(idqn_sumtree* t, const double* targets_host, int32_t* indices_host, int64_t n);
/* samplers.py:110-111: targets = root * unit_uniforms (Generator.uniform(0, root)), then query */
int idqn_sumtree_sample(idqn_sumtree* t, const double* unit_uniforms_host, int32_t* indices_host, int64_t n);
int idqn_sumtree_read_nodes(idqn_sumtree* t, double* nodes_host);  /* whole _nodes array (tests) */
/* sum_tree.py:18,32 max_recorded_priority, tracked on the device (device-side updates never visit the host) */
int idqn_sumtree_max_recorded(idqn_sumtree* t, double* value_host);
/* set(leaf, max_recorded_priority): how a prioritised buffer inserts a NEW element (it is sampled at least once) */
int idqn_sumtree_set_at_max(idqn_sumtree* t, int32_t leaf);
/* PrioritizedSamplingDistribution.update(keys, priorities) (samplers.py:75-87) with the priorities taken straight from
 * the learner's last step on the device: priority_i = mean over the K heads of |TD_k,i| (float64), leaves_host[i] = the
 * sampler's leaf of sample i.  Ordered after that step, before any later query; nothing visits the host.
 * Only priority_exponent == 1 is served here (the reference's array power has to stay numpy's, bit for bit). */
int idqn_sumtree_update_from_learner(idqn_sumtree* t, idqn_handle* h, const int32_t* leaves_host, int n);
void* idqn_sumtree_nodes_ptr(idqn_sumtree* t);
/* restore of a checkpoint: the whole _nodes array (idqn_sumtree_num_nodes doubles, as idqn_sumtree_read_nodes returned
 * it) and max_recorded_priority, uploaded unchanged -- a node's f64 value depends on the order of the adds that built it,
 * so replaying `set` on the leaves would not reproduce it */
int idqn_sumtree_write_nodes(idqn_sumtree* t, const double* nodes_host, double max_recorded);

/* ------------------------------------------------------------------------------------------------
 * Device-resident replay store (slimdqn/sample_collection/replay_buffer.py:89,202-230): fixed slots of
 * raw (uncompressed) ReplayElements; `gather` is the np.stack of ReplayBuffer.sample (:222-230). */
typedef struct idqn_replay idqn_replay;
int idqn_replay_create(int64_t n_slots, int64_t state_bytes, int device, idqn_replay** out);
int idqn_replay_destroy(idqn_replay* r);
/* ReplayBuffer.add (:207-210): store one element into `slot` */
int idqn_replay_put(idqn_replay* r, int64_t slot, const void* state_host, const void* next_state_host,
                    int32_t action, double reward, uint8_t is_terminal, uint8_t episode_end);
/* ReplayBuffer.sample (:222-230) into caller buffers (host) ... */
int idqn_replay_gather_host(idqn_replay* r, const int64_t* slots_host, int n, void* state_host, void* next_state_host,
                            int32_t* action_host, double* reward_host, uint8_t* is_terminal_host,
                            uint8_t* episode_end_host);
/* ... or straight into the learner's batch staging followed by one learn step (update_online_params, idqn.py:65-72) */
int idqn_learn_from_replay(idqn_handle* h, idqn_replay* r, const int64_t* slots_host, int n, int state_is_u8,
                           float* losses_host);

/* ------------------------------------------------------------------------------------------------
 * Frame store: ReplayBuffer(compress=True) in spirit (replay_buffer.py:36-57,204-205) -- each observation once in HBM.
 * A ring of n_frames frames of frame_bytes each (frame id f at ring slot f % n_frames) and, per element slot, 2*stack
 * frame ids: the state's stack positions, then next_state's (-1 = a zero frame, replay_buffer.py:125,136).  Value
 * v * stack + p of a stack (value_bytes bytes each) is value v of the frame at position p (the stack is the last axis,
 * :168-171).  The same handle type as the element store; idqn_replay_destroy,
 * idqn_replay_gather_host and idqn_learn_from_replay take both (their element size is frame_bytes * stack), while
 * idqn_replay_put refuses a frame store with IDQN_EINVAL.  A write into a ring slot or element row that a step
 * enqueued by idqn_learn_from_replay (losses_host == NULL) may still read waits for that step. */
int idqn_replay_create_frames(int64_t n_slots, int64_t frame_bytes, int stack, int value_bytes, int64_t n_frames,
                              int device, idqn_replay** out);
/* ReplayBuffer.add (:207-210), the observation half: frame `frame_id` into ring slot frame_id % n_frames */
int idqn_replay_put_frame(idqn_replay* r, int64_t frame_id, const void* frame_host);
/* ReplayBuffer.add (:207-210), the element half: the frame ids and scalars of one element into `slot` */
int idqn_replay_put_element(idqn_replay* r, int64_t slot, const int64_t* frame_ids_host, int32_t action, double reward,
                            uint8_t is_terminal, uint8_t episode_end);
/* no reference counterpart (its store is a dict, replay_buffer.py:89): a ring of n_frames > the current count; the frames
 * of ids [live_lo, live_hi) (at most the current count) move to their new slots, the old ring is freed once every step
 * reading it has completed */
int idqn_replay_grow_frames(idqn_replay* r, int64_t n_frames, int64_t live_lo, int64_t live_hi);

/* ------------------------------------------------------------------------------------------------
 * Checkpoint of a replay store (no reference counterpart: its checkpoint_duration argument is never used,
 * replay_buffer.py:82,93).  Each transfer first waits for the store's stream and for every learner step that may
 * still read the store, then copies in chunks through a pinned staging buffer of the store; host buffers may be
 * pageable.  A restore re-creates the store at its saved size (idqn_replay_create_frames takes n_frames). */
/* frame ids [id_lo, id_hi) in id order (frame id f at ring slot f % n_frames; a range that wraps is two copies);
 * id_hi - id_lo <= n_frames, otherwise IDQN_EINVAL */
int idqn_replay_read_frames(idqn_replay* r, int64_t id_lo, int64_t id_hi, void* dst_host);
int idqn_replay_write_frames(idqn_replay* r, int64_t id_lo, int64_t id_hi, const void* src_host);
/* slots [slot_lo, slot_lo + n): element store: state_or_rows / next_state are the two stacks ([n][state_bytes]);
 * frame store: state_or_rows is the int64 [n][2*stack] frame-id rows and next_state must be NULL (write_slots also
 * sets the host mirror of the rows) */
int idqn_replay_read_slots(idqn_replay* r, int64_t slot_lo, int64_t n, void* state_or_rows_host,
                           void* next_state_host, int32_t* action_host, double* reward_host, uint8_t* is_terminal_host,
                           uint8_t* episode_end_host);
int idqn_replay_write_slots(idqn_replay* r, int64_t slot_lo, int64_t n, const void* state_or_rows_host,
                            const void* next_state_host, const int32_t* action_host, const double* reward_host,
                            const uint8_t* is_terminal_host, const uint8_t* episode_end_host);
/* one 64-bit digest per logical array of the store, computed on the device:
 *   out[0]: element store: state stacks of slots [0, n_live_slots); frame store: frames [id_lo, id_hi) in id order,
 *           each zero-padded to a multiple of 8 bytes (id_lo / id_hi are ignored by an element store)
 *   out[1]: next_state stacks / frame-id rows of the same slots;  out[2..5]: action, reward, terminal, episode_end
 * For a byte stream of length L zero-padded to N little-endian 64-bit words w_i:
 *   digest = (sum_i splitmix64(w_i + (i + 1) * 0x9E3779B97F4A7C15)) mod 2^64  XOR  splitmix64(L)
 * It depends neither on the grid nor on the ring's size. */
int idqn_replay_digest(idqn_replay* r, int64_t n_live_slots, int64_t id_lo, int64_t id_hi, uint64_t out[6]);
/* the store's CUDA stream (cudaStream_t): its transfers and the digest run on it (events around the digest) */
void* idqn_replay_stream(idqn_replay* r);

#ifdef __cplusplus
}
#endif
#endif /* IDQN_B200_H */
