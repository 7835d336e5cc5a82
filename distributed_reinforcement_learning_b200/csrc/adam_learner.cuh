// adam_learner.cuh -- the host-side handle shell of the learners that train with TF1 Adam and keep a target network:
// Ape-X and A3C (apex.cu) and R2D2 (r2d2.cu).  It owns the streams and events, the main / target parameters, the Adam
// state, the gradient bucket, the mapped pinned result rows, the staging-slot handshake and the step lifecycle with its
// CUDA graph cache (run_step; run_filled_step for slots filled on the device).  A family handle derives from
// AdamLearner and adds its layout `pl`, its `cfg` (device, num_slots, use_cuda_graph), its slot payloads and its
// forward + loss + backward enqueue (FwdBwd); the shell appends the update.
#pragma once
#include <string>

#include "layer_defs.cuh"

namespace drl {

struct SlotSync {
  cudaEvent_t staged = nullptr;     // H2D of this slot finished (copy stream)
  cudaEvent_t consumed = nullptr;   // last compute that read this slot finished (compute stream)
  bool has_data = false;
};

struct AdamLearner {
  mutable std::recursive_mutex mu;   // taken by every C-ABI entry point (DRL_ENTER)
  int B = 0, mode = 2;
  cudaStream_t compute = nullptr, copy = nullptr, side = nullptr;
  cudaEvent_t ev_start = nullptr, ev_stop = nullptr, ev_done = nullptr;
  cudaEvent_t fj[8] = {};
  // the target scope's forward is independent of the main scope's: it runs on its own stream pair beside it
  cudaStream_t tmain = nullptr, tside = nullptr;
  cudaEvent_t tfj[8] = {}, ev_tfork = nullptr, ev_tjoin = nullptr;
  bool par = true;
  float *params = nullptr, *target = nullptr, *adam_m = nullptr, *adam_v = nullptr, *grads = nullptr;
  float* loss = nullptr;                        // the loss scalars ride in the tail of the gradient bucket
  WeightImages wi{}, twi{};
  bool main_images_stale = true, target_images_stale = true;
  int last_rows = 0;                            // rows of the most recent step / td_error call (taps, read_buffer)
  AdamState opt{};
  long long* d_step = nullptr;
  float *d_lr = nullptr, *d_alpha = nullptr, *d_b1p = nullptr, *d_b2p = nullptr;
  float *h_out = nullptr, *d_out = nullptr;     // mapped pinned [num_slots][8]
  float *h_td = nullptr, *d_td = nullptr;       // mapped pinned [num_slots][B]
  float* h_flat = nullptr;
  float* h_ones = nullptr;                      // pinned 1.0f (unit importance weights)
  std::vector<SlotSync> sync;                   // num_slots training slots + 1 scratch slot for the synchronous calls
  std::vector<void*> allocs;
  std::vector<cudaGraphExec_t> graph_step;
  bool pending = false;
  int last_slot = 0;
  int launches = 0;
};

// the family's forward passes, loss kernel and backward pass over training slot `slot` (launches: count or null)
template <class H>
using FwdBwd = int (*)(H* h, int slot, int* launches);

inline Streams streams_of(const AdamLearner* h) {
  Streams st;
  st.main = h->compute;
  st.side = h->side;
  for (int i = 0; i < 8; ++i) st.ev[i] = h->fj[i];
  st.par = h->par;
  return st;
}

// stream pair of the target scope: its own pair when the step runs parallel, otherwise the main pair (serial)
inline Streams target_streams_of(const AdamLearner* h) {
  Streams st = streams_of(h);
  if (h->par) {
    st.main = h->tmain;
    st.side = h->tside;
    for (int i = 0; i < 8; ++i) st.ev[i] = h->tfj[i];
  }
  return st;
}

// the target forward has no dependence on the main forward: fork it onto its own stream pair first and join before the
// loss kernel (inside a captured step these become parallel branches of the graph)
inline int fork_target(AdamLearner* h) {
  if (h->par) {
    DRL_CUDA_CHECK(cudaEventRecord(h->ev_tfork, h->compute));
    DRL_CUDA_CHECK(cudaStreamWaitEvent(h->tmain, h->ev_tfork, 0));
    pdl_break(h->tmain);
    pdl_break(h->tside);
  }
  return DRL_OK;
}
inline int target_done(AdamLearner* h) {
  if (h->par) DRL_CUDA_CHECK(cudaEventRecord(h->ev_tjoin, h->tmain));
  return DRL_OK;
}
inline int join_target(AdamLearner* h) {
  if (h->par) {
    DRL_CUDA_CHECK(cudaStreamWaitEvent(h->compute, h->ev_tjoin, 0));
    pdl_break(h->compute);
  }
  return DRL_OK;
}

struct AdamSchedule { float start_lr, end_lr; double learning_frame; float clip_norm; };

// create-time setup shared by the families: streams, events, parameters / target / Adam state / bucket, the pinned
// result rows, `ones` unit weights, the Adam state wiring and the events of num_slots + 1 slots.  After h->cfg, h->B
// and h->pl are set.
template <class H>
int create_shell(H* h, size_t ones, const AdamSchedule& sch) {
  DRL_CUDA_CHECK(cudaSetDevice(h->cfg.device));
  DRL_CUDA_CHECK(cudaStreamCreateWithFlags(&h->compute, cudaStreamNonBlocking));
  DRL_CUDA_CHECK(cudaStreamCreateWithFlags(&h->copy, cudaStreamNonBlocking));
  DRL_CUDA_CHECK(cudaStreamCreateWithFlags(&h->side, cudaStreamNonBlocking));
  for (int i = 0; i < 8; ++i) DRL_CUDA_CHECK(cudaEventCreateWithFlags(&h->fj[i], cudaEventDisableTiming));
  DRL_CUDA_CHECK(cudaStreamCreateWithFlags(&h->tmain, cudaStreamNonBlocking));
  DRL_CUDA_CHECK(cudaStreamCreateWithFlags(&h->tside, cudaStreamNonBlocking));
  for (int i = 0; i < 8; ++i) DRL_CUDA_CHECK(cudaEventCreateWithFlags(&h->tfj[i], cudaEventDisableTiming));
  DRL_CUDA_CHECK(cudaEventCreateWithFlags(&h->ev_tfork, cudaEventDisableTiming));
  DRL_CUDA_CHECK(cudaEventCreateWithFlags(&h->ev_tjoin, cudaEventDisableTiming));
  DRL_CUDA_CHECK(cudaEventCreate(&h->ev_start));
  DRL_CUDA_CHECK(cudaEventCreate(&h->ev_stop));
  DRL_CUDA_CHECK(cudaEventCreateWithFlags(&h->ev_done, cudaEventDisableTiming));
  const size_t B = h->B, NP = h->pl.padded_total;
  DRL_TRY(dev_alloc(h, &h->params, NP));
  DRL_TRY(dev_alloc(h, &h->target, NP));
  DRL_TRY(dev_alloc(h, &h->adam_m, NP));
  DRL_TRY(dev_alloc(h, &h->adam_v, NP));
  DRL_TRY(dev_alloc(h, &h->grads, NP + 4));
  h->loss = h->grads + NP;     // one all-reduce of the bucket covers the gradients and the loss scalars
  {
    size_t wb[WeightImages::kCount];
    weight_image_sizes(wb);
    for (int i : {1, 2, 5, 6}) DRL_TRY(dev_alloc(h, &h->wi.img[i], wb[i]));
    for (int i : {1, 2}) DRL_TRY(dev_alloc(h, &h->twi.img[i], wb[i]));
  }
  DRL_TRY(dev_alloc(h, &h->d_step, 1));
  DRL_TRY(dev_alloc(h, &h->d_lr, 1));
  DRL_TRY(dev_alloc(h, &h->d_alpha, 1));
  DRL_TRY(dev_alloc(h, &h->d_b1p, 1));
  DRL_TRY(dev_alloc(h, &h->d_b2p, 1));
  DRL_CUDA_CHECK(cudaMemcpy(h->d_b1p, &kAdamBeta1, 4, cudaMemcpyHostToDevice));
  DRL_CUDA_CHECK(cudaMemcpy(h->d_b2p, &kAdamBeta2, 4, cudaMemcpyHostToDevice));
  const size_t ns = h->cfg.num_slots;
  DRL_CUDA_CHECK(cudaHostAlloc((void**)&h->h_out, ns * 8 * sizeof(float), cudaHostAllocMapped));
  DRL_CUDA_CHECK(cudaHostGetDevicePointer((void**)&h->d_out, h->h_out, 0));
  memset(h->h_out, 0, ns * 8 * sizeof(float));
  DRL_CUDA_CHECK(cudaHostAlloc((void**)&h->h_td, ns * B * sizeof(float), cudaHostAllocMapped));
  DRL_CUDA_CHECK(cudaHostGetDevicePointer((void**)&h->d_td, h->h_td, 0));
  memset(h->h_td, 0, ns * B * sizeof(float));
  DRL_CUDA_CHECK(cudaHostAlloc((void**)&h->h_flat, NP * sizeof(float), cudaHostAllocDefault));
  DRL_CUDA_CHECK(cudaHostAlloc((void**)&h->h_ones, ones * sizeof(float), cudaHostAllocDefault));
  for (size_t i = 0; i < ones; ++i) h->h_ones[i] = 1.0f;
  AdamState& o = h->opt;
  o.params = h->params; o.m = h->adam_m; o.v = h->adam_v; o.grads = h->grads; o.n = (int64_t)NP;
  o.nblk = 148 * 4;
  DRL_TRY(dev_alloc(h, &o.norm_partials, o.nblk));
  o.step = h->d_step; o.lr_cur = h->d_lr; o.alpha = h->d_alpha; o.b1p = h->d_b1p; o.b2p = h->d_b2p;
  o.out = h->d_out; o.loss = h->loss;
  o.start_lr = sch.start_lr; o.end_lr = sch.end_lr; o.learning_frame = sch.learning_frame;
  o.clip_norm = sch.clip_norm;
  o.grad_scale = 1.0f;
  h->sync.resize(ns + 1);
  h->graph_step.assign(ns, nullptr);
  for (SlotSync& s : h->sync) {
    DRL_CUDA_CHECK(cudaEventCreateWithFlags(&s.staged, cudaEventDisableTiming));
    DRL_CUDA_CHECK(cudaEventCreateWithFlags(&s.consumed, cudaEventDisableTiming));
  }
  return DRL_OK;
}

template <class H>
int destroy_shell(H* h) {
  if (!h) return DRL_OK;
  cudaSetDevice(h->cfg.device);
  cudaDeviceSynchronize();
  for (auto g : h->graph_step) if (g) cudaGraphExecDestroy(g);
  for (SlotSync& s : h->sync) {
    if (s.staged) cudaEventDestroy(s.staged);
    if (s.consumed) cudaEventDestroy(s.consumed);
  }
  for (void* p : h->allocs) cudaFree(p);
  float* pinned[] = {h->h_out, h->h_td, h->h_flat, h->h_ones};
  for (float* p : pinned) if (p) cudaFreeHost(p);
  cudaEvent_t events[] = {h->ev_start, h->ev_stop, h->ev_done, h->ev_tfork, h->ev_tjoin};
  for (cudaEvent_t e : events) if (e) cudaEventDestroy(e);
  for (int i = 0; i < 8; ++i) if (h->fj[i]) cudaEventDestroy(h->fj[i]);
  for (int i = 0; i < 8; ++i) if (h->tfj[i]) cudaEventDestroy(h->tfj[i]);
  cudaStream_t streams[] = {h->tmain, h->tside, h->side, h->compute, h->copy};
  for (cudaStream_t s : streams) if (s) cudaStreamDestroy(s);
  cudaGetLastError();
  delete h;
  return DRL_OK;
}

// end of a create call: hands the handle out, or destroys it keeping the error text of the failed step
template <class H>
int finish_create(H* h, int rc, H** out) {
  if (rc != DRL_OK) {
    std::string keep = get_error();
    destroy_shell(h);
    set_error("%s", keep.c_str());
    return rc;
  }
  *out = h;
  return DRL_OK;
}

// ---- parameters and optimizer state (packed TF-flat vectors on the host) ----------------------------------------
template <class H>
int check_count(const H* h, int64_t n, const char* what) {
  if (n == h->pl.packed_total) return DRL_OK;
  set_error("%s: expected %lld floats, got %lld", what, (long long)h->pl.packed_total, (long long)n);
  return DRL_ERR_INVALID;
}
// which: 0 = main network, 1 = target network (DRL_APEX_MAIN / DRL_APEX_TARGET)
inline int check_which(int32_t which) {
  if (which == 0 || which == 1) return DRL_OK;
  set_error("which must be 0 (main) or 1 (target)");
  return DRL_ERR_INVALID;
}

template <class H>
int set_params(H* h, int32_t which, const float* host_flat, int64_t n) {
  DRL_TRY(check_which(which));
  if (!host_flat) { set_error("set_params: null argument"); return DRL_ERR_INVALID; }
  DRL_TRY(check_count(h, n, "set_params"));
  DRL_TRY(upload_flat(h->pl, h->h_flat, h->compute, which == 0 ? h->params : h->target, host_flat));
  if (which == 0) h->main_images_stale = true; else h->target_images_stale = true;
  return DRL_OK;
}
template <class H>
int get_params(H* h, int32_t which, float* host_flat, int64_t n) {
  DRL_TRY(check_which(which));
  if (!host_flat) { set_error("get_params: null argument"); return DRL_ERR_INVALID; }
  DRL_TRY(check_count(h, n, "get_params"));
  return download_flat(h->pl, h->h_flat, h->compute, which == 0 ? h->params : h->target, host_flat);
}
template <class H>
int get_grads(H* h, float* host_flat, int64_t n) {
  if (!host_flat) { set_error("get_grads: null argument"); return DRL_ERR_INVALID; }
  DRL_TRY(check_count(h, n, "get_grads"));
  return download_flat(h->pl, h->h_flat, h->compute, h->grads, host_flat);
}
template <class H>
int set_opt_state(H* h, const float* host_m, const float* host_v, int64_t n, int64_t step, float beta1_power,
                  float beta2_power) {
  if (!host_m || !host_v) { set_error("set_opt_state: null argument"); return DRL_ERR_INVALID; }
  DRL_TRY(check_count(h, n, "set_opt_state"));
  DRL_TRY(upload_flat(h->pl, h->h_flat, h->compute, h->adam_m, host_m));
  DRL_TRY(upload_flat(h->pl, h->h_flat, h->compute, h->adam_v, host_v));
  long long st = step;
  DRL_CUDA_CHECK(cudaMemcpy(h->d_step, &st, sizeof(st), cudaMemcpyHostToDevice));
  DRL_CUDA_CHECK(cudaMemcpy(h->d_b1p, &beta1_power, 4, cudaMemcpyHostToDevice));
  DRL_CUDA_CHECK(cudaMemcpy(h->d_b2p, &beta2_power, 4, cudaMemcpyHostToDevice));
  return DRL_OK;
}
template <class H>
int get_opt_state(H* h, float* host_m, float* host_v, int64_t n, int64_t* step, float* beta1_power,
                  float* beta2_power) {
  DRL_TRY(check_count(h, n, "get_opt_state"));
  if (host_m) DRL_TRY(download_flat(h->pl, h->h_flat, h->compute, h->adam_m, host_m));
  if (host_v) DRL_TRY(download_flat(h->pl, h->h_flat, h->compute, h->adam_v, host_v));
  DRL_CUDA_CHECK(cudaStreamSynchronize(h->compute));
  if (step) {
    long long st = 0;
    DRL_CUDA_CHECK(cudaMemcpy(&st, h->d_step, sizeof(st), cudaMemcpyDeviceToHost));
    *step = st;
  }
  if (beta1_power) DRL_CUDA_CHECK(cudaMemcpy(beta1_power, h->d_b1p, 4, cudaMemcpyDeviceToHost));
  if (beta2_power) DRL_CUDA_CHECK(cudaMemcpy(beta2_power, h->d_b2p, 4, cudaMemcpyDeviceToHost));
  return DRL_OK;
}
// target <- main, in stream order
template <class H>
int copy_main_to_target(H* h) {
  DRL_CUDA_CHECK(cudaMemcpyAsync(h->target, h->params, h->pl.padded_total * sizeof(float), cudaMemcpyDeviceToDevice,
                                 h->compute));
  pdl_break(h->compute);
  h->target_images_stale = true;
  return DRL_OK;
}
template <class H>
int grad_bucket(H* h, void** dev_ptr, int64_t* count) {
  if (dev_ptr) *dev_ptr = h->grads;
  if (count) *count = h->pl.padded_total + 4;
  return DRL_OK;
}

// ---- the step ----------------------------------------------------------------------------------------------------
template <class H>
int check_slot(const H* h, int slot) {
  if (slot >= 0 && slot < h->cfg.num_slots) return DRL_OK;
  set_error("slot %d out of range", slot);
  return DRL_ERR_INVALID;
}

// the staged/consumed handshake around the family's H2D copies, copy(stream), into training slot `slot`
template <class H, class F>
int stage_slot(H* h, int slot, F&& copy) {
  DRL_TRY(check_slot(h, slot));
  SlotSync& s = h->sync[slot];
  DRL_CUDA_CHECK(cudaStreamWaitEvent(h->copy, s.consumed, 0));
  DRL_TRY(copy(h->copy));
  DRL_CUDA_CHECK(cudaEventRecord(s.staged, h->copy));
  s.has_data = true;
  return DRL_OK;
}

// compute waits for the staged slot
inline int wait_staged(AdamLearner* h, int slot) {
  const SlotSync& s = h->sync[slot];
  if (!s.has_data) { set_error("slot %d has not been staged", slot); return DRL_ERR_STATE; }
  DRL_CUDA_CHECK(cudaStreamWaitEvent(h->compute, s.staged, 0));
  return DRL_OK;
}

// the whole step: the family's forward + loss + backward, then clip + Adam writing result row `slot`
template <class H>
int enqueue_step(H* h, int slot, FwdBwd<H> fwd_bwd, int* launches) {
  DRL_TRY(fwd_bwd(h, slot, launches));
  pdl_break(h->compute);
  AdamState o = h->opt;
  o.out = h->d_out + 8 * slot;
  prof_mark(h->compute, "optimizer(norm+adam)");
  DRL_TRY(adam_step(h->compute, o));
  prof_mark(h->compute, "end");
  if (launches) *launches += 2;
  return DRL_OK;
}

// the weight images of the main network follow its parameters, which change every step; the target images only change
// with main_to_target / set_params.  A captured step always retiles the main images and never the target ones, so
// these are refreshed here, outside of the graph.
template <class H>
int refresh_target_images(H* h) {
  if (h->target_images_stale && h->mode >= 2) {
    DRL_TRY((launch_retile_b<64>(h->compute, PlainB{h->target + h->pl.conv2_w, 64, 0}, 64, 512, h->twi.img[1])));
    DRL_TRY((launch_retile_b<64>(h->compute, PlainB{h->target + h->pl.conv3_w, 64, 0}, 64, 576, h->twi.img[2])));
  }
  h->target_images_stale = false;
  return DRL_OK;
}

inline int record_step_end(AdamLearner* h) {
  DRL_CUDA_CHECK(cudaEventRecord(h->ev_stop, h->compute));
  DRL_CUDA_CHECK(cudaEventRecord(h->ev_done, h->compute));
  h->pending = true;
  return DRL_OK;
}

template <class H>
int run_step(H* h, int slot, FwdBwd<H> fwd_bwd) {
  DRL_TRY(check_slot(h, slot));
  DRL_TRY(wait_staged(h, slot));
  if (h->cfg.use_cuda_graph) DRL_TRY(refresh_target_images(h));
  DRL_CUDA_CHECK(cudaEventRecord(h->ev_start, h->compute));
  h->main_images_stale = true;
  int cnt = 0;
  if (h->cfg.use_cuda_graph) {
    if (!h->graph_step[slot]) {
      // eager pass of forward + loss + backward first: it sets the per-kernel attributes outside of capture and does
      // not change any state the captured pass depends on (parameters and optimizer state only change in the update)
      DRL_TRY(fwd_bwd(h, slot, nullptr));
      h->main_images_stale = true;
      DRL_TRY(capture_graph(h->compute, &h->graph_step[slot], [&] { return enqueue_step(h, slot, fwd_bwd, &cnt); }));
      h->launches = cnt;
    }
    DRL_CUDA_CHECK(cudaGraphLaunch(h->graph_step[slot], h->compute));
  } else {
    DRL_TRY(enqueue_step(h, slot, fwd_bwd, &cnt));
    h->launches = cnt;
  }
  h->main_images_stale = true;      // the update changed the main parameters
  h->last_rows = h->B;
  h->last_slot = slot;
  DRL_CUDA_CHECK(cudaEventRecord(h->sync[slot].consumed, h->compute));
  return record_step_end(h);
}

// run_step for a slot that device work fills instead of an H2D copy (the device replay, replay.cu): fill() runs on the
// compute stream after any pending H2D into the slot, then the step, then after().  With use_cuda_graph all three are
// captured into graphs[slot], a cache the caller owns.  The eager pass before capture is forward + loss + backward
// only, so fill() and after() -- which advance the caller's state -- run exactly once per step, captured or not.  The
// slot is left "not staged": a plain step on it needs a new stage first.
template <class H, class Fill, class After>
int run_filled_step(H* h, int slot, FwdBwd<H> fwd_bwd, std::vector<cudaGraphExec_t>& graphs, Fill&& fill,
                    After&& after) {
  DRL_TRY(check_slot(h, slot));
  if ((int)graphs.size() < h->cfg.num_slots) graphs.resize(h->cfg.num_slots, nullptr);
  SlotSync& s = h->sync[slot];
  DRL_CUDA_CHECK(cudaStreamWaitEvent(h->compute, s.staged, 0));
  pdl_break(h->compute);
  if (h->cfg.use_cuda_graph) DRL_TRY(refresh_target_images(h));
  DRL_CUDA_CHECK(cudaEventRecord(h->ev_start, h->compute));
  h->main_images_stale = true;
  int cnt = 0;
  auto whole = [&]() -> int {
    DRL_TRY(fill());
    DRL_TRY(enqueue_step(h, slot, fwd_bwd, &cnt));
    return after();
  };
  if (h->cfg.use_cuda_graph) {
    if (!graphs[slot]) {
      DRL_TRY(fwd_bwd(h, slot, nullptr));
      h->main_images_stale = true;
      DRL_TRY(capture_graph(h->compute, &graphs[slot], whole));
      h->launches = cnt;
    }
    DRL_CUDA_CHECK(cudaGraphLaunch(graphs[slot], h->compute));
  } else {
    DRL_TRY(whole());
    h->launches = cnt;
  }
  h->main_images_stale = true;
  h->last_rows = h->B;
  h->last_slot = slot;
  DRL_CUDA_CHECK(cudaEventRecord(s.consumed, h->compute));
  s.has_data = false;
  return record_step_end(h);
}

// data parallel: the step in two halves around the caller's all-reduce of the bucket (eager launches)
template <class H>
int run_forward_backward(H* h, int slot, FwdBwd<H> fwd_bwd) {
  DRL_TRY(check_slot(h, slot));
  DRL_TRY(wait_staged(h, slot));
  DRL_CUDA_CHECK(cudaEventRecord(h->ev_start, h->compute));
  h->main_images_stale = true;
  int cnt = 0;
  DRL_TRY(fwd_bwd(h, slot, &cnt));
  h->launches = cnt + 2;
  h->last_rows = h->B;
  h->last_slot = slot;
  DRL_CUDA_CHECK(cudaEventRecord(h->sync[slot].consumed, h->compute));
  return DRL_OK;
}
inline int run_apply(AdamLearner* h, float grad_scale) {
  if (!(grad_scale > 0.f)) { set_error("apply: grad_scale must be > 0"); return DRL_ERR_INVALID; }
  pdl_break(h->compute);
  AdamState o = h->opt;
  o.out = h->d_out + 8 * h->last_slot;
  o.grad_scale = grad_scale;
  DRL_TRY(adam_step(h->compute, o));
  h->main_images_stale = true;
  return record_step_end(h);
}

// waits for the step in flight; *row = its result row (loss, lr, grad_norm, A3C baseline loss, A3C entropy, -, step),
// td_error (or null) receives its B priorities
inline int wait_step(AdamLearner* h, float* td_error, const float** row) {
  if (!h->pending) { set_error("wait: no step in flight"); return DRL_ERR_STATE; }
  h->pending = false;
  DRL_CUDA_CHECK(cudaEventSynchronize(h->ev_done));
  *row = h->h_out + 8 * h->last_slot;
  if (td_error) memcpy(td_error, h->h_td + (size_t)h->last_slot * h->B, (size_t)h->B * sizeof(float));
  return DRL_OK;
}

// one serial step (no side streams) with a device event before every launch
template <class H>
int profile_step(H* h, int slot, FwdBwd<H> fwd_bwd, char* names, int64_t names_len, float* ms, int32_t max_kernels,
                 int32_t* count) {
  DRL_TRY(check_slot(h, slot));
  if (!names || !ms || !count) { set_error("null argument"); return DRL_ERR_INVALID; }
  DRL_TRY(wait_staged(h, slot));
  DRL_CUDA_CHECK(cudaStreamSynchronize(h->compute));
  prof_begin();
  const bool par_saved = h->par;
  h->par = false;
  h->main_images_stale = true;
  int rc = enqueue_step(h, slot, fwd_bwd, nullptr);
  h->par = par_saved;
  h->main_images_stale = true;
  h->last_rows = h->B;
  DRL_TRY(prof_end(h->compute, rc, names, names_len, ms, max_kernels, count));
  h->pending = false;
  return DRL_OK;
}

inline int last_step_ms(AdamLearner* h, float* ms) {
  if (!ms) { set_error("null argument"); return DRL_ERR_INVALID; }
  DRL_CUDA_CHECK(cudaEventSynchronize(h->ev_stop));
  DRL_CUDA_CHECK(cudaEventElapsedTime(ms, h->ev_start, h->ev_stop));
  return DRL_OK;
}

}  // namespace drl
