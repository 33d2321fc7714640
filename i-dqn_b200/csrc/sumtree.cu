// SumTree on the device (slimdqn/sample_collection/sum_tree.py:8-102 of the reference), float64 nodes in HBM.
//
// Bit-exactness contract (SURVEY App. C): `set` de-duplicates (first occurrence wins), visits leaves in
// ascending order and gives every ancestor one separately rounded f64 add per leaf, in that order — the same
// sequence np.add.at produces.  Adds to different nodes are independent, so every (level, ancestor) pair is
// processed by its own thread walking its run of leaves sequentially: parallel across nodes, ordered within.
// `query` is a warp-per-target descent that prefetches a 5-level sub-tree per memory round trip; comparisons
// and subtractions are the reference's (strict <, t -= left), so indices match bit for bit.
#include "common.cuh"

#include <algorithm>
#include <numeric>

struct idqn_sumtree {
  int device;
  int64_t capacity;
  int depth;
  int64_t first_leaf, n_nodes;
  double* nodes;
  cudaStream_t stream;
  // device scratch (grown on demand)
  int64_t cap_n;
  int32_t* d_idx;
  double* d_val;   // values in, deltas after
  int32_t* d_out;
  int* d_err;
  double* d_maxrec;  // max_recorded_priority (sum_tree.py:18,32), tracked on the device
  // pinned host scratch
  int* h_err;
  double* h_root;
};

#define ST_SMALL 1024

// ------------------------------------------------------------------------------------------
// n <= 1024: one CTA sorts (leaf, position) pairs, keeps the first occurrence of each leaf, then propagates.
// val == nullptr: every listed leaf is set to *maxrec (insertion of a new element at max_recorded_priority)
__global__ void __launch_bounds__(1024) sumtree_set_small_kernel(double* __restrict__ nodes, int64_t first_leaf,
                                                                 int depth, const int32_t* __restrict__ idx,
                                                                 const double* __restrict__ val, int n,
                                                                 double* __restrict__ maxrec) {
  __shared__ unsigned long long keys[ST_SMALL];
  __shared__ int leaf_s[ST_SMALL];
  __shared__ double delta_s[ST_SMALL];
  __shared__ int m_s;
  const int tid = threadIdx.x;
  int np2 = 1;
  while (np2 < n) np2 <<= 1;
  for (int i = tid; i < np2; i += blockDim.x)
    keys[i] = i < n ? (((unsigned long long)(unsigned)idx[i] << 32) | (unsigned)i) : ~0ull;
  __syncthreads();
  for (int k = 2; k <= np2; k <<= 1)
    for (int j = k >> 1; j > 0; j >>= 1) {
      for (int i = tid; i < np2; i += blockDim.x) {
        int l = i ^ j;
        if (l > i) {
          unsigned long long a = keys[i], b = keys[l];
          bool up = (i & k) == 0;
          if ((a > b) == up) keys[i] = b, keys[l] = a;
        }
      }
      __syncthreads();
    }
  // unique leaves ascending; within equal leaves the smallest position (first occurrence) sorts first
  if (tid == 0) {
    int m = 0;
    for (int i = 0; i < n; ++i) {
      int leaf = (int)(keys[i] >> 32);
      if (i == 0 || leaf != (int)(keys[i - 1] >> 32)) {
        int pos = (int)(keys[i] & 0xffffffffu);
        leaf_s[m] = leaf;
        delta_s[m] = (val ? val[pos] : *maxrec) - nodes[first_leaf + leaf];  // sum_tree.py:34
        ++m;
      }
    }
    if (val) {  // sum_tree.py:32: max over ALL given values (duplicates included)
      double mx = *maxrec;
      for (int i = 0; i < n; ++i) mx = fmax(mx, val[i]);
      *maxrec = mx;
    }
    m_s = m;
  }
  __syncthreads();
  const int m = m_s;
  // (level, i) pairs: level 0 = leaves ... depth-1 = root
  for (int w = tid; w < depth * m; w += blockDim.x) {
    const int lev = w / m, i = w - lev * m;
    const long long node = ((first_leaf + leaf_s[i] + 1) >> lev) - 1;
    if (i > 0 && (((first_leaf + leaf_s[i - 1] + 1) >> lev) - 1) == node) continue;  // not the head of its run
    double x = nodes[node];
    for (int j = i; j < m && (((first_leaf + leaf_s[j] + 1) >> lev) - 1) == node; ++j) x = x + delta_s[j];
    nodes[node] = x;
  }
}

// large n: leaves arrive unique + ascending (host canonicalised the INDICES; all arithmetic stays here)
__global__ void sumtree_delta_kernel(const double* __restrict__ nodes, int64_t first_leaf,
                                     const int32_t* __restrict__ leaf, double* __restrict__ val, int64_t m) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < m) val[i] = val[i] - nodes[first_leaf + leaf[i]];
}
__global__ void sumtree_propagate_kernel(double* __restrict__ nodes, int64_t first_leaf, int depth,
                                         const int32_t* __restrict__ leaf, const double* __restrict__ delta,
                                         int64_t m) {
  const int lev = blockIdx.y;
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= m) return;
  const long long node = ((first_leaf + leaf[i] + 1) >> lev) - 1;
  if (i > 0 && (((first_leaf + leaf[i - 1] + 1) >> lev) - 1) == node) return;
  double x = nodes[node];
  for (int64_t j = i; j < m && (((first_leaf + leaf[j] + 1) >> lev) - 1) == node; ++j) x = x + delta[j];
  nodes[node] = x;
}

__global__ void sumtree_max_kernel(double* maxrec, double v) { *maxrec = fmax(*maxrec, v); }

// priorities of prioritised replay from the learner's per-head |TD| of its last step: val[i] = mean_k td[k][i] in float64
__global__ void sumtree_td_priority_kernel(const float* __restrict__ td, int K, int B, double* __restrict__ val) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= B) return;
  double s = 0.0;
  for (int k = 0; k < K; ++k) s += (double)td[k * B + i];  // fixed order
  val[i] = s / (double)K;
}

// ------------------------------------------------------------------------------------------
// one warp per target; each round loads the 62 descendants of the current node down 5 levels
template <bool SCALE_BY_ROOT>
__global__ void __launch_bounds__(128) sumtree_query_kernel(const double* __restrict__ nodes, int64_t first_leaf,
                                                            int depth, const double* __restrict__ targets,
                                                            int32_t* __restrict__ out, int n, int* __restrict__ err) {
  const int lane = threadIdx.x & 31;
  const int q = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (q >= n) return;
  const double root = nodes[0];
  double t = SCALE_BY_ROOT ? __dmul_rn(root, targets[q]) : targets[q];  // Generator.uniform(0, root): 0 + root*u
  if (!(t >= 0.0 && t < root)) {  // sum_tree.py:73-74
    if (lane == 0) {
      atomicOr(err, 1);
      out[q] = -1;
    }
    return;
  }
  long long node = 0;
  double cur = root;
  int level = 0;
  bool bad = false;
  while (level < depth - 1) {
    const int L = min(5, depth - 1 - level);
    const int nrel = 1 << (L + 1);  // relative heap indices 1..nrel-1, 1 = current node
    // relative r at relative depth d -> absolute (node+1)*2^d - 1 + (r - 2^d)
    double v0 = 0.0, v1 = 0.0;
    {
      int r = lane + 2;
      if (r < nrel) {
        int d = 31 - __clz(r);
        v0 = nodes[((node + 1) << d) - 1 + (r - (1 << d))];
      }
      r = lane + 34;
      if (r < nrel) {
        int d = 31 - __clz(r);
        v1 = nodes[((node + 1) << d) - 1 + (r - (1 << d))];
      }
    }
    int r = 1;
    for (int d = 0; d < L; ++d) {
      bad |= !(t < cur);  // sum_tree.py:81
      const int left = 2 * r;
      const double sl = left < 34 ? __shfl_sync(0xffffffffu, v0, left - 2) : __shfl_sync(0xffffffffu, v1, left - 34);
      const int right = left + 1;
      const double sr = right < 34 ? __shfl_sync(0xffffffffu, v0, right - 2) : __shfl_sync(0xffffffffu, v1, right - 34);
      if (t < sl) {  // strict: zero-priority leaves are never selected (:89-91)
        r = left;
        cur = sl;
      } else {
        r = right;
        t = t - sl;  // :96-100
        cur = sr;
      }
    }
    node = ((node + 1) << L) - 1 + (r - (1 << L));
    level += L;
  }
  if (lane == 0) {
    out[q] = (int32_t)(node - first_leaf);
    if (bad) atomicOr(err, 2);
  }
}

// ------------------------------------------------------------------------------------------
static int ensure_scratch(idqn_sumtree* t, int64_t n) {
  if (n <= t->cap_n) return IDQN_OK;
  int64_t cap = std::max<int64_t>(n, 1024);
  if (t->d_idx) cudaFree(t->d_idx);
  if (t->d_val) cudaFree(t->d_val);
  if (t->d_out) cudaFree(t->d_out);
  CK(cudaMalloc(&t->d_idx, sizeof(int32_t) * cap));
  CK(cudaMalloc(&t->d_val, sizeof(double) * cap));
  CK(cudaMalloc(&t->d_out, sizeof(int32_t) * cap));
  t->cap_n = cap;
  return IDQN_OK;
}

extern "C" int idqn_sumtree_create(int64_t capacity, int device, idqn_sumtree** out) {
  if (capacity <= 0) {  // sum_tree.py:12 assert
    idqn_set_error("Capacity to sum tree must be positive.");
    return IDQN_EASSERT;
  }
  REQUIRE(out, "null argument");
  REQUIRE(capacity <= (1ll << 30), "capacity too large");
  CK(cudaSetDevice(device));
  idqn_sumtree* t = new idqn_sumtree();
  memset(t, 0, sizeof(*t));
  t->device = device;
  t->capacity = capacity;
  int lg = 0;
  while ((1ll << lg) < capacity) ++lg;  // ceil(log2(capacity))
  t->depth = lg + 1;
  t->first_leaf = (1ll << (t->depth - 1)) - 1;
  t->n_nodes = (1ll << t->depth) - 1;
  CK(cudaStreamCreateWithFlags(&t->stream, cudaStreamNonBlocking));
  CK(cudaMalloc(&t->nodes, sizeof(double) * t->n_nodes));
  CK(cudaMemsetAsync(t->nodes, 0, sizeof(double) * t->n_nodes, t->stream));
  CK(cudaMalloc(&t->d_err, sizeof(int)));
  CK(cudaMemsetAsync(t->d_err, 0, sizeof(int), t->stream));
  CK(cudaMallocHost(&t->h_err, sizeof(int)));
  CK(cudaMallocHost(&t->h_root, sizeof(double)));
  CK(cudaMalloc(&t->d_maxrec, sizeof(double)));
  {
    const double one = 1.0;  // sum_tree.py:18
    CK(cudaMemcpyAsync(t->d_maxrec, &one, sizeof(double), cudaMemcpyHostToDevice, t->stream));
  }
  int rc = ensure_scratch(t, 1024);
  if (rc) return rc;
  CK(cudaStreamSynchronize(t->stream));
  *out = t;
  return IDQN_OK;
}

extern "C" int idqn_sumtree_destroy(idqn_sumtree* t) {
  if (!t) return IDQN_OK;
  cudaSetDevice(t->device);
  cudaStreamSynchronize(t->stream);
  void* ptrs[] = {t->nodes, t->d_idx, t->d_val, t->d_out, t->d_err, t->d_maxrec};
  for (void* p : ptrs)
    if (p) cudaFree(p);
  if (t->h_err) cudaFreeHost(t->h_err);
  if (t->h_root) cudaFreeHost(t->h_root);
  cudaStreamDestroy(t->stream);
  delete t;
  return IDQN_OK;
}

extern "C" int idqn_sumtree_depth(const idqn_sumtree* t) { return t ? t->depth : 0; }
extern "C" int64_t idqn_sumtree_num_nodes(const idqn_sumtree* t) { return t ? t->n_nodes : 0; }
extern "C" void* idqn_sumtree_nodes_ptr(idqn_sumtree* t) { return t ? t->nodes : nullptr; }

extern "C" int idqn_sumtree_set(idqn_sumtree* t, const int32_t* idx, const double* val, int64_t n) {
  REQUIRE(t && idx && val && n >= 0, "bad argument");
  if (n == 0) return IDQN_OK;
  for (int64_t i = 0; i < n; ++i) {
    if (!(val[i] >= 0.0)) {  // sum_tree.py:31
      idqn_set_error("Values must be positive.");
      return IDQN_EASSERT;
    }
    REQUIRE(idx[i] >= 0 && idx[i] < ((int64_t)1 << (t->depth - 1)), "leaf index %d outside the tree", idx[i]);
  }
  CK(cudaSetDevice(t->device));
  int rc = ensure_scratch(t, n);
  if (rc) return rc;
  if (n <= ST_SMALL) {
    CK(cudaMemcpyAsync(t->d_idx, idx, sizeof(int32_t) * n, cudaMemcpyHostToDevice, t->stream));
    CK(cudaMemcpyAsync(t->d_val, val, sizeof(double) * n, cudaMemcpyHostToDevice, t->stream));
    int threads = (int)std::min<int64_t>(1024, std::max<int64_t>(64, (n * t->depth + 31) / 32 * 32));
    sumtree_set_small_kernel<<<1, threads, 0, t->stream>>>(t->nodes, t->first_leaf, t->depth, t->d_idx, t->d_val,
                                                          (int)n, t->d_maxrec);
    CK(cudaGetLastError());
    CK(cudaStreamSynchronize(t->stream));  // the caller's host buffers may go away
    return IDQN_OK;
  }
  // bulk: canonicalise the index list on the host (stable sort by leaf => first occurrence leads its run)
  std::vector<int64_t> order(n);
  std::iota(order.begin(), order.end(), 0);
  std::stable_sort(order.begin(), order.end(), [&](int64_t a, int64_t b) { return idx[a] < idx[b]; });
  std::vector<int32_t> u;
  std::vector<double> v;
  u.reserve(n), v.reserve(n);
  for (int64_t i = 0; i < n; ++i) {
    if (i == 0 || idx[order[i]] != idx[order[i - 1]]) {
      u.push_back(idx[order[i]]);
      v.push_back(val[order[i]]);
    }
  }
  const int64_t m = (int64_t)u.size();
  sumtree_max_kernel<<<1, 1, 0, t->stream>>>(t->d_maxrec, *std::max_element(val, val + n));
  CK(cudaGetLastError());
  CK(cudaMemcpyAsync(t->d_idx, u.data(), sizeof(int32_t) * m, cudaMemcpyHostToDevice, t->stream));
  CK(cudaMemcpyAsync(t->d_val, v.data(), sizeof(double) * m, cudaMemcpyHostToDevice, t->stream));
  const int threads = 256;
  const unsigned blocks = (unsigned)((m + threads - 1) / threads);
  sumtree_delta_kernel<<<blocks, threads, 0, t->stream>>>(t->nodes, t->first_leaf, t->d_idx, t->d_val, m);
  CK(cudaGetLastError());
  sumtree_propagate_kernel<<<dim3(blocks, t->depth), threads, 0, t->stream>>>(t->nodes, t->first_leaf, t->depth,
                                                                             t->d_idx, t->d_val, m);
  CK(cudaGetLastError());
  CK(cudaStreamSynchronize(t->stream));
  return IDQN_OK;
}

extern "C" int idqn_sumtree_get(idqn_sumtree* t, const int32_t* idx, double* val, int64_t n) {
  REQUIRE(t && idx && val && n >= 0, "bad argument");
  CK(cudaSetDevice(t->device));
  for (int64_t i = 0; i < n; ++i) {
    REQUIRE(idx[i] >= 0 && t->first_leaf + idx[i] < t->n_nodes, "leaf index outside the tree");
    CK(cudaMemcpyAsync(val + i, t->nodes + t->first_leaf + idx[i], sizeof(double), cudaMemcpyDeviceToHost,
                       t->stream));
  }
  CK(cudaStreamSynchronize(t->stream));
  return IDQN_OK;
}

extern "C" int idqn_sumtree_root(idqn_sumtree* t, double* root) {
  REQUIRE(t && root, "bad argument");
  CK(cudaSetDevice(t->device));
  CK(cudaMemcpyAsync(t->h_root, t->nodes, sizeof(double), cudaMemcpyDeviceToHost, t->stream));
  CK(cudaStreamSynchronize(t->stream));
  *root = *t->h_root;
  return IDQN_OK;
}

extern "C" int idqn_sumtree_read_nodes(idqn_sumtree* t, double* nodes) {
  REQUIRE(t && nodes, "bad argument");
  CK(cudaSetDevice(t->device));
  CK(cudaMemcpyAsync(nodes, t->nodes, sizeof(double) * t->n_nodes, cudaMemcpyDeviceToHost, t->stream));
  CK(cudaStreamSynchronize(t->stream));
  return IDQN_OK;
}

// restore of a saved tree: the nodes are uploaded as they were read, not rebuilt through `set` (a node's f64 value
// depends on the order of the adds that made it)
extern "C" int idqn_sumtree_write_nodes(idqn_sumtree* t, const double* nodes, double max_recorded) {
  REQUIRE(t && nodes, "bad argument");
  CK(cudaSetDevice(t->device));
  CK(cudaMemcpyAsync(t->nodes, nodes, sizeof(double) * t->n_nodes, cudaMemcpyHostToDevice, t->stream));
  CK(cudaMemcpyAsync(t->d_maxrec, &max_recorded, sizeof(double), cudaMemcpyHostToDevice, t->stream));
  CK(cudaStreamSynchronize(t->stream));
  return IDQN_OK;
}

template <bool SCALE>
static int query_impl(idqn_sumtree* t, const double* targets, int32_t* out, int64_t n) {
  REQUIRE(t && targets && out && n >= 0, "bad argument");
  if (n == 0) return IDQN_OK;
  CK(cudaSetDevice(t->device));
  int rc = ensure_scratch(t, n);
  if (rc) return rc;
  CK(cudaMemcpyAsync(t->d_val, targets, sizeof(double) * n, cudaMemcpyHostToDevice, t->stream));
  const int threads = 128;
  const unsigned blocks = (unsigned)((n * 32 + threads - 1) / threads);
  sumtree_query_kernel<SCALE><<<blocks, threads, 0, t->stream>>>(t->nodes, t->first_leaf, t->depth, t->d_val,
                                                                 t->d_out, (int)n, t->d_err);
  CK(cudaGetLastError());
  CK(cudaMemcpyAsync(out, t->d_out, sizeof(int32_t) * n, cudaMemcpyDeviceToHost, t->stream));
  CK(cudaMemcpyAsync(t->h_err, t->d_err, sizeof(int), cudaMemcpyDeviceToHost, t->stream));
  CK(cudaStreamSynchronize(t->stream));
  if (*t->h_err) {
    int e = *t->h_err;
    CK(cudaMemsetAsync(t->d_err, 0, sizeof(int), t->stream));
    CK(cudaStreamSynchronize(t->stream));
    if (e & 1) {
      double root = 0;
      idqn_sumtree_root(t, &root);
      idqn_set_error("Targets must be in the interval [0.0, %.17g).", root);
      return IDQN_ERANGE;
    }
    idqn_set_error("sum tree traversal: intermediate target not below intermediate node (sum_tree.py:81)");
    return IDQN_EASSERT;
  }
  return IDQN_OK;
}

extern "C" int idqn_sumtree_query(idqn_sumtree* t, const double* targets, int32_t* out, int64_t n) {
  return query_impl<false>(t, targets, out, n);
}
extern "C" int idqn_sumtree_sample(idqn_sumtree* t, const double* unit_uniforms, int32_t* out, int64_t n) {
  return query_impl<true>(t, unit_uniforms, out, n);
}

extern "C" int idqn_sumtree_max_recorded(idqn_sumtree* t, double* value) {
  REQUIRE(t && value, "bad argument");
  CK(cudaSetDevice(t->device));
  CK(cudaMemcpyAsync(t->h_root, t->d_maxrec, sizeof(double), cudaMemcpyDeviceToHost, t->stream));
  CK(cudaStreamSynchronize(t->stream));
  *value = *t->h_root;
  return IDQN_OK;
}

extern "C" int idqn_sumtree_set_at_max(idqn_sumtree* t, int32_t leaf) {
  REQUIRE(t && leaf >= 0 && leaf < ((int64_t)1 << (t->depth - 1)), "leaf index %d outside the tree", leaf);
  CK(cudaSetDevice(t->device));
  CK(cudaMemcpyAsync(t->d_idx, &leaf, sizeof(int32_t), cudaMemcpyHostToDevice, t->stream));
  sumtree_set_small_kernel<<<1, 64, 0, t->stream>>>(t->nodes, t->first_leaf, t->depth, t->d_idx, nullptr, 1, t->d_maxrec);
  CK(cudaGetLastError());
  CK(cudaStreamSynchronize(t->stream));
  return IDQN_OK;
}

extern "C" int idqn_sumtree_update_from_learner(idqn_sumtree* t, idqn_handle* h, const int32_t* leaves, int n) {
  REQUIRE(t && h && leaves, "null argument");
  REQUIRE(n == h->B && n <= ST_SMALL, "%d leaves for a learner batch of %d", n, h->B);
  REQUIRE(t->device == h->cfg.device, "sum tree and learner live on different devices");
  for (int i = 0; i < n; ++i)
    REQUIRE(leaves[i] >= 0 && leaves[i] < ((int64_t)1 << (t->depth - 1)), "leaf index %d outside the tree", leaves[i]);
  CK(cudaSetDevice(t->device));
  // ordered behind the learner's step, on the tree's own stream (later queries follow on the same stream)
  CK(cudaEventRecord(h->ev_step, h->stream));
  CK(cudaStreamWaitEvent(t->stream, h->ev_step, 0));
  CK(cudaMemcpyAsync(t->d_idx, leaves, sizeof(int32_t) * n, cudaMemcpyHostToDevice, t->stream));
  sumtree_td_priority_kernel<<<(n + 127) / 128, 128, 0, t->stream>>>(h->td_abs, h->K, h->B, t->d_val);
  CK(cudaGetLastError());
  const int threads = (int)std::min<int64_t>(1024, std::max<int64_t>(64, ((int64_t)n * t->depth + 31) / 32 * 32));
  sumtree_set_small_kernel<<<1, threads, 0, t->stream>>>(t->nodes, t->first_leaf, t->depth, t->d_idx, t->d_val, n, t->d_maxrec);
  CK(cudaGetLastError());
  return IDQN_OK;  // no host synchronisation: the leaves were staged by the pageable copy before it returned
}
