// replay.cu -- the device-resident prioritized replay of the Ape-X learner behind drl_apex_replay_* (include/drl_b200.h):
// buffer_queue.Memory / SumTree (distributed_queue/buffer_queue.py:326-416) together with the object storage of the
// transitions, kept in the learner's GPU memory and connected to its step without a host round trip.
//
// Storage is field-major: state / next_state [cap, 84*84*4] u8, previous_action / action [cap] i32, reward [cap] f32,
// done [cap] u8, all byte offsets 64-bit (at capacity 1e5 a frame array is 2.8 GB).  The sum tree is the reference's
// array of 2*cap - 1 float64 nodes with the leaves last.  Three kernels do the work; the first two never look at the
// record layout, so a sequence replay can reuse them:
//   ordered_update_kernel  SumTree.update applied to a list of (leaf, priority) in call order, bit-identical to the
//                          sequential host loop: change_i = p_i - (leaf value at time i), then every touched internal node
//                          adds the changes of the updates whose path passes through it, in increasing i.  (Level-by-level
//                          passes would reorder those adds when the leaves sit at two depths, i.e. whenever cap is not a
//                          power of two.)
//   replay_sample_kernel   Memory.sample: one thread per stratum, Philox4x32-10 draws, the _retrieve walk, importance
//                          weights normalised by their block maximum; every double operation rounds like the host's.
//   replay_gather_kernel   the sampled rows into a training slot, in the layout drl_apex_stage produces (16-byte copies).
#include <math.h>

#include <algorithm>

#include "replay.cuh"

namespace drl {
namespace {

constexpr double kPerE = 0.001, kPerA = 0.6, kBetaInc = 0.001, kBeta0 = 0.4;   // buffer_queue.py:372-375
constexpr int kMaxReplayBatch = 1024;                                         // one CTA per kernel

struct ReplayWords {           // device state the captured step reads and advances
  int64_t n_entries;
  int64_t write;
  double beta;
  uint64_t draws;              // sample calls so far: the Philox counter's high words
};

// ------------------------------------------------------------------------------------------
// Philox4x32-10 (Salmon et al., SC'11; the Random123 constants).  Stratum i of draw call c uses counter
// (i, c lo, c hi, 0) and key (seed lo, seed hi); u = ((x0 << 32 | x1) >> 11) * 2^-53 is in [0, 1) and exact.
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ double philox_u01(uint32_t i, uint64_t c, uint64_t seed) {
  uint32_t x0 = i, x1 = (uint32_t)c, x2 = (uint32_t)(c >> 32), x3 = 0;
  uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32);
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    if (r) { k0 += 0x9E3779B9u; k1 += 0xBB67AE85u; }
    const uint32_t lo0 = 0xD2511F53u * x0, hi0 = __umulhi(0xD2511F53u, x0);
    const uint32_t lo1 = 0xCD9E8D57u * x2, hi1 = __umulhi(0xCD9E8D57u, x2);
    const uint32_t y0 = hi1 ^ x1 ^ k0, y2 = hi0 ^ x3 ^ k1;
    x0 = y0; x1 = lo1; x2 = y2; x3 = lo0;
  }
  const uint64_t bits = ((uint64_t)x0 << 32 | x1) >> 11;
  return (double)bits * 0x1.0p-53;
}

// priority of |td| (Memory._getPriority, buffer_queue.py:383-384): CUDA's double pow is not correctly rounded, so a leaf
// may differ from glibc's by a few ulp; everything downstream of the leaves is exact
__device__ __forceinline__ double priority_of(float td) { return pow(__dadd_rn((double)td, kPerE), kPerA); }

__device__ __forceinline__ bool on_path(int64_t leaf, int64_t node) {
  while (leaf > node) leaf = (leaf - 1) >> 1;
  return leaf == node;
}

// The leaves of one ordered update: leaf[i] (sampled tree indices), or the ring positions cap - 1 + (first + i) % cap
// (an add at the write cursor).  Priorities come from |td|.
struct LeafList {
  const int64_t* leaf;
  int64_t first;
  const float* td;
  int n;
};

__global__ void __launch_bounds__(kMaxReplayBatch) ordered_update_kernel(double* __restrict__ tree, int64_t cap,
                                                                         LeafList L, int64_t* __restrict__ log_leaf,
                                                                         double* __restrict__ log_p,
                                                                         ReplayWords* words, int64_t new_n,
                                                                         int64_t new_write) {
  pdl_prologue();
  __shared__ int64_t s_leaf[kMaxReplayBatch];
  __shared__ double s_p[kMaxReplayBatch], s_change[kMaxReplayBatch];
  const int i = threadIdx.x, n = L.n;
  if (i < n) {
    s_leaf[i] = L.leaf ? L.leaf[i] : cap - 1 + (L.first + i) % cap;
    s_p[i] = priority_of(L.td[i]);
  }
  __syncthreads();
  if (i < n) {                      // the leaf's value at time i: an earlier duplicate's priority, else the tree's
    const int64_t lf = s_leaf[i];
    double old = tree[lf];
    for (int j = i - 1; j >= 0; --j)
      if (s_leaf[j] == lf) { old = s_p[j]; break; }
    s_change[i] = __dsub_rn(s_p[i], old);
  }
  __syncthreads();                  // every leaf has been read: from here on each node has exactly one writer
  if (i < n) {
    const int64_t lf = s_leaf[i];
    bool last = true;
    for (int j = i + 1; j < n; ++j) last = last && s_leaf[j] != lf;
    if (last) tree[lf] = s_p[i];
    // internal nodes: thread i owns the ancestors no earlier update passes through, and folds the changes of every
    // update from i on whose path contains the node, in call order
    for (int64_t a = lf; a != 0;) {
      a = (a - 1) >> 1;
      bool owned = true;
      for (int j = 0; j < i && owned; ++j) owned = !on_path(s_leaf[j], a);
      if (!owned) break;            // an earlier update passes through a, hence through all its ancestors
      double acc = tree[a];
      for (int j = i; j < n; ++j)
        if (on_path(s_leaf[j], a)) acc = __dadd_rn(acc, s_change[j]);
      tree[a] = acc;
    }
    log_leaf[i] = lf;
    log_p[i] = s_p[i];
  }
  if (i == 0 && words && new_n >= 0) {
    words->n_entries = new_n;
    words->write = new_write;
  }
}

struct SampleOut {
  int64_t* tree_index;
  int64_t* data_index;
  double* priority;
  double* is_weight;
  float* slot_weight;          // [n] the training slot's float32 weights
};

// Memory.sample (buffer_queue.py:390-411) for n strata, one thread each
__global__ void __launch_bounds__(kMaxReplayBatch) replay_sample_kernel(const double* __restrict__ tree, int64_t cap,
                                                                        ReplayWords* words, uint64_t seed, int n,
                                                                        SampleOut o) {
  pdl_prologue();
  __shared__ double red[kMaxReplayBatch / 32];
  const int i = threadIdx.x;
  const double total = tree[0];
  const int64_t n_entries = words->n_entries;
  const uint64_t c = words->draws;
  const double beta = fmin(1.0, __dadd_rn(words->beta, kBetaInc));         // :395
  double w = 0.0;
  if (i < n) {
    const double segment = __ddiv_rn(total, (double)n);                    // :393
    const double a = __dmul_rn(segment, (double)i), b = __dmul_rn(segment, (double)(i + 1));
    double s = __dadd_rn(a, __dmul_rn(__dsub_rn(b, a), philox_u01((uint32_t)i, c, seed)));   // random.uniform(a, b)
    int64_t idx = 0;                                                       // SumTree._retrieve (:340-347)
    const int64_t len = 2 * cap - 1;
    for (;;) {
      const int64_t left = 2 * idx + 1;
      if (left >= len) break;
      const double tl = tree[left];
      if (s <= tl) {
        idx = left;
      } else {
        s = __dsub_rn(s, tl);
        idx = left + 1;
      }
    }
    const double p = tree[idx];
    const double prob = __ddiv_rn(p, total);                               // :406
    w = pow(__dmul_rn((double)n_entries, prob), -beta);                    // :407
    o.tree_index[i] = idx;
    o.data_index[i] = idx - cap + 1;
    o.priority[i] = p;
  }
  // max over the strata (the host's running `if (w > mx) mx = w` from 0)
  double m = w;
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) {
    const double x = __shfl_xor_sync(0xffffffffu, m, off);
    m = x > m ? x : m;
  }
  if ((i & 31) == 0) red[i >> 5] = m;
  __syncthreads();
  double mx = 0.0;
  for (int k = 0; k < (int)(blockDim.x >> 5); ++k) mx = red[k] > mx ? red[k] : mx;
  if (i < n) {
    const double wn = __ddiv_rn(w, mx);                                    // :408
    o.is_weight[i] = wn;
    o.slot_weight[i] = __double2float_rn(wn);
  }
  if (i == 0) {                     // every thread has read beta and the counter (the barrier above)
    words->beta = beta;
    words->draws = c + 1;
  }
}

// one row of one field per CTA: dst[r] = src[rows[r]]
struct GatherField {
  const uint8_t* src;
  uint8_t* dst;
  int64_t row_bytes;
};
constexpr int kMaxGatherFields = 8;
struct GatherArgs {
  const int64_t* rows;
  GatherField f[kMaxGatherFields];
};

__global__ void __launch_bounds__(256) replay_gather_kernel(GatherArgs g) {
  pdl_prologue();
  const int r = blockIdx.x;
  const GatherField f = g.f[blockIdx.y];
  const int64_t bytes = f.row_bytes;
  const uint8_t* src = f.src + g.rows[r] * bytes;
  uint8_t* dst = f.dst + (int64_t)r * bytes;
  if ((bytes & 15) == 0 && ((reinterpret_cast<uintptr_t>(src) | reinterpret_cast<uintptr_t>(dst)) & 15) == 0) {
    const uint4* s4 = reinterpret_cast<const uint4*>(src);
    uint4* d4 = reinterpret_cast<uint4*>(dst);
    for (int64_t k = threadIdx.x; k < bytes / 16; k += blockDim.x) d4[k] = __ldg(s4 + k);
  } else {
    for (int64_t k = threadIdx.x; k < bytes; k += blockDim.x) dst[k] = src[k];
  }
}

}  // namespace
}  // namespace drl

using namespace drl;

struct drl_apex_replay {
  drl_apex* h = nullptr;
  ApexReplayLink link{};
  int64_t cap = 0;
  uint64_t seed = 0;
  int64_t n_entries = 0, write = 0;     // host mirror of the device words (argument checks)
  int last_update = 0;                  // entries of the most recent ordered update
  uint8_t *state = nullptr, *next_state = nullptr, *done = nullptr;
  int32_t *previous_action = nullptr, *action = nullptr;
  float* reward = nullptr;
  double* tree = nullptr;
  ReplayWords* words = nullptr;
  int64_t *tree_index = nullptr, *data_index = nullptr, *log_leaf = nullptr;
  double *priority = nullptr, *is_weight = nullptr, *log_p = nullptr;
  std::vector<void*> allocs;
  std::vector<cudaGraphExec_t> graphs;  // one captured replay step per training slot
};

namespace {

template <class T>
int replay_alloc(drl_apex_replay* r, T** p, size_t count, const char* what) {
  const size_t bytes = count * sizeof(T);
  void* q = nullptr;
  const cudaError_t e = cudaMalloc(&q, bytes);
  if (e != cudaSuccess) {
    cudaGetLastError();
    set_error("replay_create: cudaMalloc of %zu bytes for %s failed: %s", bytes, what, cudaGetErrorString(e));
    return DRL_ERR_CUDA;
  }
  r->allocs.push_back(q);
  DRL_CUDA_CHECK(cudaMemset(q, 0, bytes));
  *p = static_cast<T*>(q);
  return DRL_OK;
}

void free_replay(drl_apex_replay* r) {
  for (auto g : r->graphs) if (g) cudaGraphExecDestroy(g);
  for (void* p : r->allocs) cudaFree(p);
  cudaGetLastError();
  delete r;
}

// SumTree.update over L.n leaves on the learner's compute stream; new_n >= 0 also stores the add's cursor words
int enqueue_ordered_update(drl_apex_replay* r, cudaStream_t s, const LeafList& L, int64_t new_n, int64_t new_write) {
  const int threads = (L.n + 31) / 32 * 32;
  pdl_break(s);
  DRL_CUDA_CHECK((launch_k(ordered_update_kernel, 1, threads, 0, s, r->tree, r->cap, L, r->log_leaf, r->log_p,
                           r->words, new_n, new_write)));
  pdl_break(s);
  return DRL_OK;
}

// sample B strata, then gather the B transitions into the slot (drl_apex_stage's layout)
int enqueue_sample_gather(drl_apex_replay* r, cudaStream_t s, const ApexRecordView& v) {
  const int B = r->link.B;
  pdl_break(s);
  prof_mark(s, "replay_sample");
  DRL_CUDA_CHECK((launch_k(replay_sample_kernel, 1, (B + 31) / 32 * 32, 0, s, r->tree, r->cap, r->words, r->seed, B,
                           SampleOut{r->tree_index, r->data_index, r->priority, r->is_weight, v.weight})));
  GatherArgs g{};
  g.rows = r->data_index;
  g.f[0] = {r->state, v.frames, (int64_t)Geo::FRAME};
  g.f[1] = {r->next_state, v.frames + (size_t)v.row2 * Geo::FRAME, (int64_t)Geo::FRAME};
  g.f[2] = {reinterpret_cast<const uint8_t*>(r->previous_action), reinterpret_cast<uint8_t*>(v.pa2), 4};
  g.f[3] = {reinterpret_cast<const uint8_t*>(r->action), reinterpret_cast<uint8_t*>(v.pa2 + v.row2), 4};
  g.f[4] = {reinterpret_cast<const uint8_t*>(r->reward), reinterpret_cast<uint8_t*>(v.reward), 4};
  g.f[5] = {r->done, v.done, 1};
  prof_mark(s, "replay_gather");
  DRL_CUDA_CHECK((launch_k(replay_gather_kernel, dim3(B, 6), 256, 0, s, g)));
  pdl_break(s);
  return DRL_OK;
}

// copies rows [0, n) of a scratch field to ring positions write, write + 1, ... (mod cap), in order: a batch longer
// than the ring overwrites its own first rows, as n sequential Memory.add calls do
int copy_to_ring(cudaStream_t s, uint8_t* dst, const uint8_t* src, size_t row_bytes, int64_t write, int64_t cap, int n) {
  for (int64_t i = 0; i < n;) {
    const int64_t pos = (write + i) % cap;
    const int64_t len = std::min<int64_t>(n - i, cap - pos);
    DRL_CUDA_CHECK(cudaMemcpyAsync(dst + (size_t)pos * row_bytes, src + (size_t)i * row_bytes, (size_t)len * row_bytes,
                                   cudaMemcpyDeviceToDevice, s));
    i += len;
  }
  return DRL_OK;
}

}  // namespace

#define DRL_REPLAY_ENTER(r)                                                       \
  if (!(r)) { ::drl::set_error("null replay handle"); return DRL_ERR_INVALID; }   \
  std::lock_guard<std::recursive_mutex> _drl_lock(*(r)->link.mu);                 \
  DRL_CUDA_CHECK(cudaSetDevice((r)->link.device))

extern "C" {

int drl_apex_replay_create(drl_apex* h, int64_t capacity, uint64_t seed, drl_apex_replay** out) {
  if (drl_device_count() < 1) { set_error("replay_create: no CUDA device (no CPU fallback)"); return DRL_ERR_CUDA; }
  if (!h || !out) { set_error("null argument"); return DRL_ERR_INVALID; }
  *out = nullptr;
  ApexReplayLink link{};
  DRL_TRY(apex_replay_link(h, &link));
  std::lock_guard<std::recursive_mutex> lock(*link.mu);
  DRL_CUDA_CHECK(cudaSetDevice(link.device));
  if (link.algo != 0) { set_error("replay_create: needs an Ape-X handle (an A3C handle has no target network)"); return DRL_ERR_INVALID; }
  if (capacity < 2) { set_error("replay_create: capacity must be >= 2"); return DRL_ERR_INVALID; }
  if (link.B > kMaxReplayBatch) { set_error("replay_create: batch must be <= %d", kMaxReplayBatch); return DRL_ERR_INVALID; }
  drl_apex_replay* r = new drl_apex_replay();
  r->h = h;
  r->link = link;
  r->cap = capacity;
  r->seed = seed;
  const size_t cap = (size_t)capacity, B = (size_t)link.B;
  const int rc = [&]() -> int {
    DRL_TRY(replay_alloc(r, &r->state, cap * Geo::FRAME, "state"));
    DRL_TRY(replay_alloc(r, &r->next_state, cap * Geo::FRAME, "next_state"));
    DRL_TRY(replay_alloc(r, &r->previous_action, cap, "previous_action"));
    DRL_TRY(replay_alloc(r, &r->action, cap, "action"));
    DRL_TRY(replay_alloc(r, &r->reward, cap, "reward"));
    DRL_TRY(replay_alloc(r, &r->done, cap, "done"));
    DRL_TRY(replay_alloc(r, &r->tree, 2 * cap - 1, "the sum tree"));
    DRL_TRY(replay_alloc(r, &r->words, 1, "the replay words"));
    DRL_TRY(replay_alloc(r, &r->tree_index, B, "the sample record"));
    DRL_TRY(replay_alloc(r, &r->data_index, B, "the sample record"));
    DRL_TRY(replay_alloc(r, &r->priority, B, "the sample record"));
    DRL_TRY(replay_alloc(r, &r->is_weight, B, "the sample record"));
    DRL_TRY(replay_alloc(r, &r->log_leaf, B, "the update record"));
    DRL_TRY(replay_alloc(r, &r->log_p, B, "the update record"));
    const ReplayWords w0{0, 0, kBeta0, 0};
    DRL_CUDA_CHECK(cudaMemcpy(r->words, &w0, sizeof(w0), cudaMemcpyHostToDevice));
    return DRL_OK;
  }();
  if (rc != DRL_OK) {
    std::string keep = get_error();
    free_replay(r);
    set_error("%s", keep.c_str());
    return rc;
  }
  apex_replay_attach(h, +1);
  *out = r;
  return DRL_OK;
}

int drl_apex_replay_destroy(drl_apex_replay* r) {
  if (!r) return DRL_OK;
  drl_apex* h = r->h;
  {
    std::lock_guard<std::recursive_mutex> lock(*r->link.mu);
    cudaSetDevice(r->link.device);
    cudaStreamSynchronize(r->link.compute);
    free_replay(r);
  }
  apex_replay_attach(h, -1);
  return DRL_OK;
}

int drl_apex_replay_add(drl_apex_replay* r, int32_t n, const uint8_t* state, const uint8_t* next_state,
                        const int32_t* previous_action, const int32_t* action, const float* reward,
                        const uint8_t* done) {
  DRL_REPLAY_ENTER(r);
  if (n < 1 || n > r->link.B) { set_error("replay_add: n must be in [1, %d]", r->link.B); return DRL_ERR_INVALID; }
  if (!state || !next_state || !previous_action || !action || !reward || !done) { set_error("replay_add: null pointer"); return DRL_ERR_INVALID; }
  ApexRecordView v{};
  DRL_TRY(apex_enqueue_td_error(r->h, n, state, next_state, previous_action, action, reward, done, &v));
  const cudaStream_t s = r->link.compute;
  const int64_t w = r->write, cap = r->cap;
  DRL_TRY(copy_to_ring(s, r->state, v.frames, Geo::FRAME, w, cap, n));
  DRL_TRY(copy_to_ring(s, r->next_state, v.frames + (size_t)v.row2 * Geo::FRAME, Geo::FRAME, w, cap, n));
  DRL_TRY(copy_to_ring(s, reinterpret_cast<uint8_t*>(r->previous_action), reinterpret_cast<const uint8_t*>(v.pa2), 4, w, cap, n));
  DRL_TRY(copy_to_ring(s, reinterpret_cast<uint8_t*>(r->action), reinterpret_cast<const uint8_t*>(v.pa2 + v.row2), 4, w, cap, n));
  DRL_TRY(copy_to_ring(s, reinterpret_cast<uint8_t*>(r->reward), reinterpret_cast<const uint8_t*>(v.reward), 4, w, cap, n));
  DRL_TRY(copy_to_ring(s, r->done, v.done, 1, w, cap, n));
  const int64_t new_n = std::min<int64_t>(r->n_entries + n, cap), new_write = (w + n) % cap;
  DRL_TRY(enqueue_ordered_update(r, s, LeafList{nullptr, w, r->link.td_dev, n}, new_n, new_write));
  DRL_CUDA_CHECK(cudaStreamSynchronize(s));
  r->n_entries = new_n;
  r->write = new_write;
  r->last_update = n;
  return DRL_OK;
}

int drl_apex_replay_step_async(drl_apex_replay* r, int32_t slot) {
  DRL_REPLAY_ENTER(r);
  if (r->n_entries < 1) { set_error("replay_step: the replay is empty"); return DRL_ERR_STATE; }
  const ApexSlotWork fill = [r](cudaStream_t s, const ApexRecordView& v) { return enqueue_sample_gather(r, s, v); };
  const ApexSlotWork after = [r](cudaStream_t s, const ApexRecordView&) {
    prof_mark(s, "replay_priority_update");
    return enqueue_ordered_update(r, s, LeafList{r->tree_index, 0, r->link.td_dev, r->link.B}, -1, 0);
  };
  DRL_TRY(apex_replay_step(r->h, slot, r->graphs, fill, after));
  r->last_update = r->link.B;
  return DRL_OK;
}

int drl_apex_replay_step(drl_apex_replay* r, int32_t slot, drl_apex_out* out, float* td_error) {
  DRL_TRY(drl_apex_replay_step_async(r, slot));
  return drl_apex_wait(r->h, out, td_error);
}

int drl_apex_replay_last_sample(drl_apex_replay* r, int64_t* tree_index, int64_t* data_index, double* priority,
                                double* is_weight) {
  DRL_REPLAY_ENTER(r);
  DRL_CUDA_CHECK(cudaStreamSynchronize(r->link.compute));
  const size_t B = r->link.B;
  if (tree_index) DRL_CUDA_CHECK(cudaMemcpy(tree_index, r->tree_index, B * 8, cudaMemcpyDeviceToHost));
  if (data_index) DRL_CUDA_CHECK(cudaMemcpy(data_index, r->data_index, B * 8, cudaMemcpyDeviceToHost));
  if (priority) DRL_CUDA_CHECK(cudaMemcpy(priority, r->priority, B * 8, cudaMemcpyDeviceToHost));
  if (is_weight) DRL_CUDA_CHECK(cudaMemcpy(is_weight, r->is_weight, B * 8, cudaMemcpyDeviceToHost));
  return DRL_OK;
}

int drl_apex_replay_last_update(drl_apex_replay* r, int64_t* leaf, double* priority, int32_t max_count,
                                int32_t* count) {
  DRL_REPLAY_ENTER(r);
  if (!count) { set_error("null argument"); return DRL_ERR_INVALID; }
  DRL_CUDA_CHECK(cudaStreamSynchronize(r->link.compute));
  *count = r->last_update;
  const size_t m = (size_t)std::max(0, std::min(max_count, r->last_update));
  if (leaf && m) DRL_CUDA_CHECK(cudaMemcpy(leaf, r->log_leaf, m * 8, cudaMemcpyDeviceToHost));
  if (priority && m) DRL_CUDA_CHECK(cudaMemcpy(priority, r->log_p, m * 8, cudaMemcpyDeviceToHost));
  return DRL_OK;
}

int drl_apex_replay_info(drl_apex_replay* r, int64_t* n_entries, int64_t* write, double* total, double* beta,
                         int64_t* draws) {
  DRL_REPLAY_ENTER(r);
  DRL_CUDA_CHECK(cudaStreamSynchronize(r->link.compute));
  ReplayWords w{};
  double t = 0.0;
  DRL_CUDA_CHECK(cudaMemcpy(&w, r->words, sizeof(w), cudaMemcpyDeviceToHost));
  DRL_CUDA_CHECK(cudaMemcpy(&t, r->tree, sizeof(t), cudaMemcpyDeviceToHost));
  if (n_entries) *n_entries = w.n_entries;
  if (write) *write = w.write;
  if (total) *total = t;
  if (beta) *beta = w.beta;
  if (draws) *draws = (int64_t)w.draws;
  return DRL_OK;
}

int drl_apex_replay_read_tree(drl_apex_replay* r, double* host_nodes, int64_t count) {
  DRL_REPLAY_ENTER(r);
  if (!host_nodes || count != 2 * r->cap - 1) { set_error("read_tree: expected %lld nodes", (long long)(2 * r->cap - 1)); return DRL_ERR_INVALID; }
  DRL_CUDA_CHECK(cudaStreamSynchronize(r->link.compute));
  DRL_CUDA_CHECK(cudaMemcpy(host_nodes, r->tree, (size_t)count * 8, cudaMemcpyDeviceToHost));
  return DRL_OK;
}

}  // extern "C"
