// per.cu -- prioritized replay index behind drl_per_* (include/drl_b200.h): the host-side sum tree of
// buffer_queue.SumTree / Memory (distributed_queue/buffer_queue.py:326-416).  Host code only: the transitions stay
// with the caller, as in the reference's loop, which this path serves unchanged (B tree walks and B leaf updates per
// step next to the Python loop).  A learner that keeps the transitions on the GPU uses the device replay instead
// (replay.cu, drl_apex_replay_*), whose tree kernels follow the same arithmetic.  The tree is float64 and every update adds
// the same `change` to the same ancestors in the same order as the reference's recursion, so totals, sampled
// indices and priorities are bit-identical to the NumPy implementation for the same uniform draws.
#include <math.h>

#include <vector>

#include "common.cuh"

struct drl_per {
  int64_t capacity = 0;
  std::vector<double> tree;      // 2 * capacity - 1 nodes, leaves at [capacity - 1, 2 * capacity - 1)
  int64_t write = 0;             // SumTree.write
  int64_t n_entries = 0;
  double beta = 0.4;             // Memory.beta (buffer_queue.py:375)
};

namespace {
constexpr double kE = 0.001, kA = 0.6, kBetaInc = 0.001;     // Memory.e / a / beta_increment_per_sampling (:373-376)

inline double priority_of(double error) { return pow(error + kE, kA); }    // Memory._getPriority (:383-384)

void tree_update(drl_per* p, int64_t idx, double pr) {       // SumTree.update + _propagate (:361-364, :334-338)
  const double change = pr - p->tree[idx];
  p->tree[idx] = pr;
  while (idx != 0) {
    idx = (idx - 1) / 2;
    p->tree[idx] += change;
  }
}

int64_t tree_retrieve(const drl_per* p, double s) {          // SumTree._retrieve (:340-347)
  int64_t idx = 0;
  const int64_t len = (int64_t)p->tree.size();
  for (;;) {
    const int64_t left = 2 * idx + 1;
    if (left >= len) return idx;
    if (s <= p->tree[left]) {
      idx = left;
    } else {
      s -= p->tree[left];
      idx = left + 1;
    }
  }
}
}  // namespace

extern "C" {

int drl_per_create(int64_t capacity, drl_per** out) {
  if (!out) { drl::set_error("null argument"); return DRL_ERR_INVALID; }
  *out = nullptr;
  if (capacity < 2) { drl::set_error("per: capacity must be >= 2"); return DRL_ERR_INVALID; }
  drl_per* p = new drl_per();
  p->capacity = capacity;
  p->tree.assign((size_t)(2 * capacity - 1), 0.0);
  *out = p;
  return DRL_OK;
}

int drl_per_destroy(drl_per* p) {
  delete p;
  return DRL_OK;
}

int drl_per_add(drl_per* p, double error, int64_t* data_index) {
  if (!p) { drl::set_error("null per handle"); return DRL_ERR_INVALID; }
  const int64_t w = p->write;
  tree_update(p, w + p->capacity - 1, priority_of(error));      // SumTree.add (:351-359)
  if (data_index) *data_index = w;
  p->write = (w + 1 >= p->capacity) ? 0 : w + 1;
  if (p->n_entries < p->capacity) ++p->n_entries;
  return DRL_OK;
}

int drl_per_sample(drl_per* p, int32_t n, const double* u01, int64_t* tree_index, int64_t* data_index, double* priority,
                   double* is_weight) {
  if (!p) { drl::set_error("null per handle"); return DRL_ERR_INVALID; }
  if (n < 1 || !u01 || !tree_index || !data_index || !priority || !is_weight) { drl::set_error("per_sample: bad argument"); return DRL_ERR_INVALID; }
  if (p->n_entries < 1) { drl::set_error("per_sample: the memory is empty"); return DRL_ERR_STATE; }
  const double total = p->tree[0];
  const double segment = total / n;                              // :393
  p->beta = fmin(1.0, p->beta + kBetaInc);                       // :395
  double mx = 0.0;
  for (int32_t i = 0; i < n; ++i) {
    const double a = segment * i, b = segment * (i + 1);         // :398
    const double s = a + (b - a) * u01[i];                       // random.uniform(a, b)
    const int64_t idx = tree_retrieve(p, s);                     // SumTree.get (:366-369)
    tree_index[i] = idx;
    data_index[i] = idx - p->capacity + 1;
    priority[i] = p->tree[idx];
    const double prob = priority[i] / total;                     // :406
    is_weight[i] = pow((double)p->n_entries * prob, -p->beta);   // :407
    if (is_weight[i] > mx) mx = is_weight[i];
  }
  for (int32_t i = 0; i < n; ++i) is_weight[i] /= mx;            // :408
  return DRL_OK;
}

int drl_per_update(drl_per* p, int64_t tree_index, double error) {
  if (!p) { drl::set_error("null per handle"); return DRL_ERR_INVALID; }
  if (tree_index < p->capacity - 1 || tree_index >= 2 * p->capacity - 1) { drl::set_error("per_update: %lld is not a leaf index", (long long)tree_index); return DRL_ERR_INVALID; }
  tree_update(p, tree_index, priority_of(error));                // Memory.update (:413-415)
  return DRL_OK;
}

int drl_per_total(const drl_per* p, double* total) {
  if (!p || !total) { drl::set_error("null argument"); return DRL_ERR_INVALID; }
  *total = p->tree[0];
  return DRL_OK;
}
int drl_per_size(const drl_per* p, int64_t* n_entries) {
  if (!p || !n_entries) { drl::set_error("null argument"); return DRL_ERR_INVALID; }
  *n_entries = p->n_entries;
  return DRL_OK;
}
int drl_per_beta(const drl_per* p, double* beta) {
  if (!p || !beta) { drl::set_error("null argument"); return DRL_ERR_INVALID; }
  *beta = p->beta;
  return DRL_OK;
}

}  // extern "C"
