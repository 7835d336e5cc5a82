// kernels.h -- internal interface between the learner orchestration (learner.cu) and the kernel
// launchers (layers.cu, elementwise.cu, vtrace.cu, optimizer.cu).  Not part of the C-ABI.
#pragma once
#include <string.h>

#include <mutex>
#include <vector>

#include "common.cuh"

namespace drl {

// Offsets (in floats) of each tensor inside the padded flat parameter / gradient / slot vectors.
// Order = TF1 variable-creation order (SURVEY.md App. A.6); every bias directly follows its
// kernel (kernel sizes are multiples of 4) and is padded up to a multiple of 4 floats so that all
// kernels start 16-byte aligned.  [w ; b] therefore forms one contiguous [(K+1), N] matrix, which
// is what the weight-gradient GEMMs write (bias gradient = column sum of dY in row K).
// The IMPALA, Ape-X and R2D2 layouts extend this with their named offsets.
template <int N>
struct FlatLayout {
  static constexpr int kNumTensors = N;
  int64_t padded_total;   // floats in the padded vector (multiple of 4)
  int64_t packed_total;   // floats in the TF-flat (API) vector
  int64_t packed_off[N], padded_off[N], count[N];
  // tensor i has sizes[i] floats; *fields[i] receives its padded offset
  void place(const int64_t (&sizes)[N], int64_t* const (&fields)[N]) {
    int64_t po = 0, pk = 0;
    for (int i = 0; i < N; ++i) {
      count[i] = sizes[i];
      packed_off[i] = pk;
      padded_off[i] = po;
      *fields[i] = po;
      pk += sizes[i];
      po += sizes[i];
      if (i & 1) po = (po + 3) / 4 * 4;   // pad after each bias (all kernel sizes are multiples of 4)
    }
    packed_total = pk;
    padded_total = (po + 3) / 4 * 4;
  }
};

struct ParamLayout : FlatLayout<24> {
  int A;
  int64_t conv1_w, conv1_b, conv2_w, conv2_b, conv3_w, conv3_b;
  int64_t emb1_w, emb1_b, emb2_w, emb2_b;
  int64_t lstm_w, lstm_b;
  int64_t actor1_w, actor1_b, actor2_w, actor2_b, actor3_w, actor3_b;
  int64_t critic1_w, critic1_b, critic2_w, critic2_b, critic3_w, critic3_b;
  void init(int num_action);
};

struct Inputs {          // one device staging slot, caller's batch-major layout
  const uint8_t* frames; // [B,T,84,84,4]
  const float* reward;   // [B,T]
  const int32_t* action; // [B,T]
  const uint8_t* done;   // [B,T]
  const float* mu;       // [B,T,A]
  const int32_t* pa;     // [B,T]
  const float* h0;       // [B,T,256]
  const float* c0;       // [B,T,256]
};

struct Acts {            // forward activations, time-major rows m = t*B + b, M = B*T rows
  float* a1;             // [M,20,20,32]
  float* a1_lo;          // tf32 remainder plane of a1 (same shape), allocated right behind a1: TMA operand of conv2
  float* a2;             // [M,9,9,64]
  float* a2_lo;          // same for a2 (conv3)
  float* a3;             // [M,3136]
  float* e1;             // [A,256]  relu(emb1)
  float* table;          // [A,256]  action-embedding table
  float* zpart;          // [SPLITS][M,1024] LSTM pre-activation partial sums
  float* gates;          // [M,4,256] sigmoid(i), tanh(j), sigmoid(f+1), sigmoid(o)
  float* c1;             // [M,256]
  float* tc1;            // [M,256] tanh(c1)
  float* h1;             // [M,256]
  float* hid1;           // [2][M,256] actor/critic hidden 1
  float* hid2;           // [2][M,256] actor/critic hidden 2
  float* logits;         // [M,A]
  float* policy;         // [M,A]
  float* value;          // [M]
  // math mode 5, bulk-fed lstm_wgrad (gemm_bulk16.cuh): x^T = [a3|emb|h0]^T as a 16-bit operand image, nullptr = gather path
  uint8_t* img_xt = nullptr;   // x^T : rows = features (3648) x K = Mb rows -- A operand of lstm_wgrad
  int img_rows = 0;            // M the images were sized for
};

struct Bwd {             // backward workspace, Mb = B*(T-2) rows
  float* dlogits;        // [Mb,32] (columns >= A stay zero)
  float* dv;             // [Mb,32] (column 0 = dL/dV, others stay zero)
  float* dhid2;          // [2][Mb,256]
  float* dhid1;          // [2][Mb,256]
  float* dh_part;        // [2][Mb,256] actor and critic contributions to dL/dh1
  float* dz;             // [Mb,1024]
  uint8_t* img_dzt = nullptr;  // dz^T : rows n (1024) x K = Mb rows  -- B operand of the bulk-fed lstm_wgrad (see Acts::img_xt)
  float* da3;            // [Mb,3136]
  float* du;             // [Mb,256]
  float* dpre2;          // [A,256]
  float* dpre1;          // [A,256]
  float* da2;            // [Mb,9,9,64]
  float* da1;            // [Mb,20,20,32]
  float* wg_part;        // split-K partial slabs for the conv3/conv2 weight gradients (side stream) + emb scratch
  float* wg_part2;       // split-K partial slabs for the conv1 weight gradient (main stream)
  float* dcol;           // [Mb*81, 512] (conv2) / [Mb*49, 576] (conv3): per-output-pixel tap gradients before col2im
  size_t wg_part_floats;
  float* emb_scratch = nullptr;   // own scratch of emb_backward (16 * 32 * 256 floats): lets it run on the second side lane
                                  // beside the conv weight gradients; nullptr: it borrows wg_part on `side`
};

struct VtraceOut {       // parity taps, batch-major [B, T-2]
  float *vs, *clipped_rho, *vs_plus_1, *pg_adv;
  float* loss_partials;  // [nblk,3]
  unsigned int* ticket;  // last-block counter
  float* loss_sums;      // [4] pi, baseline, entropy, (pad) -- tail of the gradient bucket
};

constexpr int kLstmSplits = 8;   // slabs allocated for the LSTM split-K partial sums (4 or 7 are used)

// math_mode 0 in drl_learner_config resolves to this (1 = FP32 FFMA, 2 = tcgen05 3xTF32)
#ifndef DRL_DEFAULT_PDL_LEVEL
#define DRL_DEFAULT_PDL_LEVEL 0   // programmatic dependent launch (common.cuh); see DESIGN.md for the measurements
#endif
#ifndef DRL_DEFAULT_MATH_MODE
#define DRL_DEFAULT_MATH_MODE 2          // Ape-X / A3C / R2D2 handles
#endif
#ifndef DRL_DEFAULT_MATH_MODE_IMPALA
#define DRL_DEFAULT_MATH_MODE_IMPALA 5   // IMPALA handle: tcgen05 kind::f16 with 16-bit split operands (gemm_umma16.cuh)
#endif

// Per-kernel device timing (learner.cu): when a profile run is active, prof_mark records a CUDA event
// on the launching stream before each named launch; otherwise it is a no-op.
void prof_mark(cudaStream_t s, const char* name);
// profile run bracket (shared by the IMPALA and the Ape-X learner): prof_begin arms prof_mark; prof_end synchronises
// `s`, converts the recorded events into per-launch times (names joined by '\n') and disarms it.
void prof_begin();
int prof_end(cudaStream_t s, int rc, char* names, int64_t names_len, float* ms, int32_t max_kernels, int32_t* count);

// Pre-split (hi/lo tf32), pre-tiled, pre-swizzled global copies of the weights that serve as B operands of the
// tensor-core GEMMs (gemm_umma.cuh: PretiledB / retile_b_kernel); refreshed after every parameter update.
struct WeightImages {
  static constexpr int kCount = 7;
  uint8_t* img[kCount];   // 0 conv1 fwd, 1 conv2 fwd, 2 conv3 fwd, 3 lstm fwd, 4 lstm dgrad, 5 conv3 dCol, 6 conv2 dCol
};
void weight_image_sizes(size_t (&bytes)[WeightImages::kCount]);
int net_retile(cudaStream_t s_conv, cudaStream_t s_rest, const ParamLayout& pl, const float* params,
               const WeightImages& wi);

// ---- layers.cu ----------------------------------------------------------------------------
// main = critical path; side = kernels off the critical path (fork/join through ev[]); par = false runs
// everything on main (used by the per-kernel profile so that event times are per-kernel).
struct Streams {
  cudaStream_t main, side;
  cudaEvent_t ev[8];
  bool par;
  // optional second side lane (IMPALA handle): the four small, latency-bound head weight gradients run here so that they
  // do not sit in front of lstm_wgrad / the conv weight gradients on `side` (tools/timeline.py, profiles/r02_timeline_*).
  // nullptr: everything stays on `side`.
  cudaStream_t side2 = nullptr;
  cudaEvent_t ev2[4] = {nullptr, nullptr, nullptr, nullptr};
  cudaEvent_t ev_lstm_grads = nullptr;   // backward: recorded on the side stream once the head and LSTM weight gradients
                                         // are in the bucket (the early part of the peer exchange waits for it)
};
// mode: 1 = FP32-FFMA gather-GEMM, 2 = tcgen05 3xTF32 gather-GEMM for the large contractions
int net_forward(const Streams& st, const ParamLayout& pl, const float* params, const WeightImages& wi, const Inputs& in,
                const Acts& act, int B, int T, int mode, bool retile);
int net_backward(const Streams& st, const ParamLayout& pl, const float* params, const WeightImages& wi, float* grads,
                 const Inputs& in, const Acts& act, const Bwd& bwd, int B, int T, int mode);
size_t wgrad_partial_floats(int B, int T);
// bytes of the operand images of the bulk-fed lstm_wgrad: which = 1 x^T (K = Mb), 3 dz^T (K = Mb)
size_t lstm_image_bytes(int which, int M, int Mb);
int forward_launch_count();
int backward_launch_count();

// ---- elementwise.cu -----------------------------------------------------------------------
int emb_forward(cudaStream_t s, const float* w1, const float* b1, const float* w2, const float* b2, float* e1,
                float* table, int A);
int lstm_gates_forward(cudaStream_t s, const float* zpart, int nsplit, const float* bias, const float* c0,
                       float* gates, float* c1, float* tc1, float* h1, int M, int B, int T);
int heads_out_forward(cudaStream_t s, const float* hid2_actor, const float* hid2_critic, const float* w5,
                      const float* b5, const float* w8, const float* b8, float* logits, float* policy,
                      float* value, int M, int A);
int heads_out_backward(cudaStream_t s, const float* dlogits, const float* dv, const float* w5, const float* w8,
                       const float* hid2_actor, const float* hid2_critic, float* dhid2_actor, float* dhid2_critic,
                       int Mb, int A);
int lstm_gates_backward(cudaStream_t s, const float* dh_part, size_t part_stride, const float* gates,
                        const float* tc1, const float* c0, float* dz, int Mb, int B, int T);
int emb_backward(cudaStream_t s, const float* du, const int32_t* pa, const float* e1, const float* table,
                 const float* w2, float* dpre2, float* dpre1, float* g_w1, float* g_b1, float* g_w2, float* g_b2,
                 float* scratch, int Mb, int B, int T, int A);
int splitk_reduce(cudaStream_t s, const float* part, size_t slab, int nsplit, float* out, size_t n);
// second half of the "dCol" form of the conv data gradients (gather of <= 9 / 4 taps + ReLU mask)
int col2im_conv3(cudaStream_t s, const float* dcol, const float* a2, float* da2, int nimg);
int col2im_conv2(cudaStream_t s, const float* dcol, const float* a1, float* da1, int nimg);

// ---- vtrace.cu ----------------------------------------------------------------------------
struct VtraceCfg {
  float discount, baseline_coef, entropy_coef;
  int reward_clipping;
};
int vtrace_losses(cudaStream_t s, const VtraceCfg& cfg, const float* policy, const float* value, const Inputs& in,
                  const VtraceOut& out, float* dlogits, float* dv, int B, int T, int A);

// ---- optimizer.cu -------------------------------------------------------------------------
struct OptState {
  float* params; float* ms; float* grads;   // padded flat vectors
  int64_t n;                                 // padded_total (multiple of 4)
  float* norm_partials; int nblk;            // partial sums of squares; grid size of the two optimizer kernels
  int npart;                                 // how many partials the update kernel sums (nblk, or world * nblk_r)
  // peer exchange (peer.cu): the update kernel first waits for the peers' barrier-1 flags (null: single replica)
  const uint32_t* wait_flags; const uint32_t* wait_epoch; int wait_world;
  uint32_t* wait_err; uint32_t* wait_err_host; unsigned long long wait_timeout_ns;   // peer_sync.cuh::PeerErr
  int wait_parts;                            // exchange instances to wait for
  long long* step;                           // device global_step
  float* lr_cur;                             // device scalar
  float* out;                                // device [8]: pi, baseline, entropy, lr, grad_norm, total, step_lo, step_hi
  const float* loss_sums;                    // bucket tail
  float start_lr, end_lr; double learning_frame;
  float clip_norm, baseline_coef, entropy_coef;
};
int optimizer_apply(cudaStream_t s, const OptState& o);
int optimizer_update_only(cudaStream_t s, const OptState& o);   // clip + RMSProp from already reduced partials

// TF1 Adam (the Ape-X, A3C and R2D2 learners)
// clip_norm <= 0: no clipping (optimizer.minimize, agent/r2d2.py:92); start_lr == end_lr: constant learning rate
struct AdamState {
  float* params; float* m; float* v; const float* grads; int64_t n;
  float* norm_partials; int nblk;
  long long* step; float* lr_cur; float* alpha; float* b1p; float* b2p;
  float* out;               // [8] mapped pinned: loss, lr, grad_norm, -, -, -, step_lo, step_hi
  const float* loss;
  float start_lr, end_lr; double learning_frame; float clip_norm;
  float grad_scale;         // data parallel: the bucket holds the SUM over ranks of per-rank MEAN-loss gradients -> 1/world
                            // (1 for a single replica); applied to the gradient, its norm and the logged losses
};
int adam_step(cudaStream_t s, const AdamState& o);   // 2 launches: partial norms + scalars, then the update
constexpr float kAdamBeta1 = 0.9f, kAdamBeta2 = 0.999f;

// ---- peer.cu: gradient exchange over NVLink peer memory (CUDA IPC), fused with the norm ------------------------
constexpr int kMaxPeers = 16;
constexpr int kPeerParts = 2;      // exchange instances per step: part 0 = [lstm .. end) of the bucket (96 % of the bytes, complete when
                                   // the LSTM weight gradient is, ~230 us before the backward pass ends) on its own stream with a small
                                   // grid; part 1 = [conv1 .. emb2] after the backward pass (see DESIGN.md section 5)
struct PeerTable {                 // device pointers into every rank's buffers (index = rank; own entries are local)
  float* bucket[kMaxPeers];        // [padded grads | 4 loss sums]
  float* reduced[kMaxPeers];       // same shape: the summed bucket, delivered by the owners of the slices
  float* partials[kMaxPeers];      // [world * nblk_r] partial squared norms
  uint32_t* flags[kMaxPeers];      // [2 * kPeerParts][kMaxPeers] barrier epochs (phase = 2 * part + {ready, delivered})
  uint32_t* epoch[kMaxPeers];      // per part 4 words: epochs completed (x2), CTA ticket counter (own entry only)
  uint32_t* err[kMaxPeers];        // barrier time-out word in device memory (only the own entry is used)
  uint32_t* err_host;              // its mapped pinned copy for the host
  unsigned long long timeout_ns;   // barrier time-out (DRL_B200_PEER_TIMEOUT_S)
};
struct PeerPlan {
  PeerTable t;
  OptState o;                      // the update's state (lr / step live here)
  int rank, world, nblk;
};
// one exchange instance over float4 range [beg4, end4) of the bucket; do_lr: also lr / global_step (last instance)
int peer_exchange(cudaStream_t s, const PeerPlan& pp, int part, int64_t beg4, int64_t end4, bool do_lr, int grid = 0);

// ---- host-side handle helpers (learner.cu, apex.cu, r2d2.cu) ----------------------------------------------------
// Prologue of every C-ABI entry point that takes a handle: null check, the handle's recursive lock (actor threads call
// parameter_sync -> get_params on the learner's handle while the learner thread trains; ctypes drops the GIL), and
// the handle's device.
#define DRL_ENTER(h)                                                                  \
  if (!(h)) { ::drl::set_error("null handle"); return DRL_ERR_INVALID; }             \
  std::lock_guard<std::recursive_mutex> _drl_lock((h)->mu);                           \
  DRL_CUDA_CHECK(cudaSetDevice((h)->cfg.device))

// zeroed (or fill_byte) device buffer of count T plus 256 bytes of slack, freed with the handle (h->allocs)
template <class H, class T>
int dev_alloc(H* h, T** p, size_t count, int fill_byte = 0) {
  void* q = nullptr;
  DRL_CUDA_CHECK(cudaMalloc(&q, count * sizeof(T) + 256));
  DRL_CUDA_CHECK(cudaMemset(q, fill_byte, count * sizeof(T) + 256));
  h->allocs.push_back(q);
  *p = static_cast<T*>(q);
  return DRL_OK;
}
inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

// packed (TF-flat, API) <-> padded (device) copies on stream s through the pinned scratch h_flat (padded_total floats)
template <class L>
int upload_flat(const L& pl, float* h_flat, cudaStream_t s, float* dev_padded, const float* host_packed,
                float pad_value = 0.0f) {
  for (int64_t i = 0; i < pl.padded_total; ++i) h_flat[i] = pad_value;
  for (int i = 0; i < L::kNumTensors; ++i)
    memcpy(h_flat + pl.padded_off[i], host_packed + pl.packed_off[i], pl.count[i] * sizeof(float));
  DRL_CUDA_CHECK(cudaStreamSynchronize(s));
  DRL_CUDA_CHECK(cudaMemcpyAsync(dev_padded, h_flat, pl.padded_total * sizeof(float), cudaMemcpyHostToDevice, s));
  DRL_CUDA_CHECK(cudaStreamSynchronize(s));
  return DRL_OK;
}
template <class L>
int download_flat(const L& pl, float* h_flat, cudaStream_t s, const float* dev_padded, float* host_packed) {
  DRL_CUDA_CHECK(cudaMemcpyAsync(h_flat, dev_padded, pl.padded_total * sizeof(float), cudaMemcpyDeviceToHost, s));
  DRL_CUDA_CHECK(cudaStreamSynchronize(s));
  for (int i = 0; i < L::kNumTensors; ++i)
    memcpy(host_packed + pl.packed_off[i], h_flat + pl.padded_off[i], pl.count[i] * sizeof(float));
  return DRL_OK;
}

// captures what enqueue() puts on stream s (and the streams it forks to) and instantiates it into *exec
template <class F>
int capture_graph(cudaStream_t s, cudaGraphExec_t* exec, F&& enqueue) {
  cudaGraph_t g = nullptr;
  DRL_CUDA_CHECK(cudaStreamBeginCapture(s, cudaStreamCaptureModeThreadLocal));
  const int r = enqueue();
  const cudaError_t e = cudaStreamEndCapture(s, &g);
  if (r != DRL_OK) { if (g) cudaGraphDestroy(g); return r; }
  if (e != cudaSuccess) { set_error("graph capture failed: %s", cudaGetErrorString(e)); return DRL_ERR_CUDA; }
  DRL_CUDA_CHECK(cudaGraphInstantiate(exec, g, 0));
  cudaGraphDestroy(g);
  return DRL_OK;
}

// read_buffer: copies the named device buffer of tab[0, n) to host_dst once compute has drained
struct NamedBuffer { const char* name; const float* p; size_t count; };
inline int read_named_buffer(cudaStream_t compute, const NamedBuffer* tab, size_t n, const char* name, float* host_dst,
                             int64_t count) {
  for (size_t i = 0; i < n; ++i) {
    const NamedBuffer& e = tab[i];
    if (strcmp(e.name, name) != 0) continue;
    if ((size_t)count != e.count) { set_error("read_buffer(%s): expected %zu floats, got %lld", name, e.count, (long long)count); return DRL_ERR_INVALID; }
    DRL_CUDA_CHECK(cudaStreamSynchronize(compute));
    DRL_CUDA_CHECK(cudaMemcpy(host_dst, e.p, e.count * sizeof(float), cudaMemcpyDeviceToHost));
    return DRL_OK;
  }
  set_error("read_buffer: unknown buffer '%s'", name);
  return DRL_ERR_INVALID;
}

// global_step of a result row: the update kernel stores it as two int32 bit patterns in r[6] (low) and r[7] (high)
inline int64_t result_row_step(const float* r) {
  uint32_t lo, hi;
  memcpy(&lo, &r[6], 4);
  memcpy(&hi, &r[7], 4);
  return (int64_t)(((uint64_t)hi << 32) | lo);
}

}  // namespace drl
