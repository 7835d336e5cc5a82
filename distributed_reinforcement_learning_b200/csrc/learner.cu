// learner.cu -- the learner handle behind the C-ABI (include/drl_b200.h): owns parameters, RMSProp
// slots, the gradient bucket, activations, device staging slots, a compute and a copy stream.
// Replaces impala.Agent's learner graph and Agent.train (agent/impala.py:11-103,132-148).
#include <stdarg.h>
#include <string.h>

#include <stdlib.h>

#include <mutex>
#include <string>
#include <unordered_map>
#include <vector>

#include <nvtx3/nvToolsExt.h>   // header-only NVTX v3: no link dependency, a no-op unless a profiler injects itself

#include "kernels.h"

namespace drl {

// NVTX ranges (SURVEY.md section 5: the reference has no tracing at all) around the host-side phases of a step:
// stage (H2D enqueue), forward, vtrace_losses, backward, exchange, update.  Inside a CUDA-graph replay the phases are
// one cudaGraphLaunch, so the ranges mark the capture / eager enqueue and the replay as a whole ("step(graph)").
struct NvtxRange {
  explicit NvtxRange(const char* name) { nvtxRangePushA(name); }
  ~NvtxRange() { nvtxRangePop(); }
};

static thread_local char g_err[1024] = {0};
void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}
const char* get_error() { return g_err; }

// programmatic-dependent-launch bookkeeping (common.cuh): per thread, per stream
bool& pdl_chain_ok(cudaStream_t s) {
  static thread_local std::unordered_map<cudaStream_t, bool> chain;
  return chain[s];
}
int pdl_level() {
  static const int level = [] {
    const char* e = getenv("DRL_B200_PDL");
    return e ? atoi(e) : DRL_DEFAULT_PDL_LEVEL;
  }();
  return level;
}
static std::vector<TraceSetter>& trace_setters() {
  static std::vector<TraceSetter> v;
  return v;
}
int register_trace_setter(TraceSetter f) {
  trace_setters().push_back(f);
  return (int)trace_setters().size();
}
bool& pdl_region_on() {
  static thread_local bool on = true;
  return on;
}

// ---- per-kernel profiler -------------------------------------------------------------------
struct Profiler {
  bool on = false;
  std::vector<cudaEvent_t> ev;
  std::vector<const char*> names;
};
static Profiler g_prof;
void prof_mark(cudaStream_t s, const char* name) {
  if (!g_prof.on) return;
  cudaEvent_t e = nullptr;
  if (cudaEventCreate(&e) != cudaSuccess) return;
  cudaEventRecord(e, s);
  pdl_break(s);
  g_prof.ev.push_back(e);
  g_prof.names.push_back(name);
}

void prof_begin() {
  g_prof.on = true;
  g_prof.ev.clear();
  g_prof.names.clear();
}
int prof_end(cudaStream_t s, int rc, char* names, int64_t names_len, float* ms, int32_t max_kernels, int32_t* count) {
  g_prof.on = false;
  cudaError_t e = cudaStreamSynchronize(s);
  int n = 0;
  std::string joined;
  if (rc == DRL_OK && e == cudaSuccess) {
    for (size_t i = 0; i + 1 < g_prof.ev.size() && n < max_kernels; ++i) {
      float t = 0.f;
      cudaEventElapsedTime(&t, g_prof.ev[i], g_prof.ev[i + 1]);
      ms[n++] = t;
      if (!joined.empty()) joined += "\n";
      joined += g_prof.names[i];
    }
  }
  for (cudaEvent_t ev : g_prof.ev) cudaEventDestroy(ev);
  g_prof.ev.clear();
  g_prof.names.clear();
  if (rc != DRL_OK) return rc;
  if (e != cudaSuccess) { set_error("profile step failed: %s", cudaGetErrorString(e)); return DRL_ERR_CUDA; }
  if ((int64_t)joined.size() + 1 > names_len) { set_error("profile: names buffer too small"); return DRL_ERR_INVALID; }
  memcpy(names, joined.c_str(), joined.size() + 1);
  *count = n;
  return DRL_OK;
}

struct Slot {
  uint8_t* base = nullptr;   // one allocation, fields at 256-byte aligned offsets
  Inputs in{};
  cudaEvent_t staged = nullptr;     // H2D of this slot finished (copy stream)
  cudaEvent_t consumed = nullptr;   // last compute that read this slot finished (compute stream)
  bool has_data = false;
};

}  // namespace drl

using namespace drl;

struct drl_learner {
  drl_learner_config cfg{};
  int B = 0, T = 0, A = 0, M = 0, Mb = 0, mode = 1;
  ParamLayout pl{};
  cudaStream_t compute = nullptr, copy = nullptr, side = nullptr, xchg = nullptr;
  cudaEvent_t ev_lstm_grads = nullptr, ev_xchg_done = nullptr;   // early part of the peer exchange (stream xchg)
  int peer_early_ctas = 64;   // grid of the early exchange instance (DRL_B200_PEER_EARLY_CTAS; 0 = no early part)
  cudaEvent_t ev_start = nullptr, ev_stop = nullptr, ev_done = nullptr;
  cudaEvent_t fj[8] = {};    // fork/join events between the compute and the side stream
  cudaStream_t side2 = nullptr;   // second side lane (small head weight gradients), DRL_B200_SIDE2=0 disables
  cudaEvent_t fj2[4] = {};
  bool par = true;           // run off-critical-path kernels on the side stream
  bool images_stale = true;  // weight images do not match the parameters (forward-only entry points rebuild them)
  float* params = nullptr;
  float* ms = nullptr;
  float* bucket = nullptr;   // [padded_total grads | 4 loss sums]
  Acts act{};
  Bwd bwd{};
  WeightImages wimg{};
  VtraceOut vt{};
  OptState opt{};
  long long* d_step = nullptr;
  float* d_lr = nullptr;
  float* d_out = nullptr;    // device alias of h_out (mapped pinned memory)
  float* h_out = nullptr;    // pinned [num_slots + 1][8]: the steps' scalars, written by the update kernel itself
                             // (zero-copy); row = slot for drl_learner_step*, row num_slots for drl_learner_apply
  std::vector<cudaEvent_t> ev_done_slot;   // per result row
  int last_out = 0;          // result row of the most recently enqueued update
  float* h_flat = nullptr;   // pinned scratch for set/get params (padded_total floats)
  std::vector<Slot> slots;
  std::vector<void*> allocs;
  bool pending = false;      // a step was enqueued and its scalars not yet collected
  int launches = 0;
  // CUDA graphs (one per slot) for forward+backward and for apply
  std::vector<cudaGraphExec_t> graph_fb;
  cudaGraphExec_t graph_apply = nullptr;
  std::vector<cudaGraphExec_t> graph_step;   // forward+backward+[exchange]+apply in one graph
  // gradient exchange over NVLink peer memory (peer.cu); off until drl_learner_peer_import
  bool peer_on = false;
  int peer_nblk = 148 * 4;
  uint8_t* comm = nullptr;                   // [reduced | partials | flags | epochs | err], own cudaMalloc (IPC-exported)
  size_t comm_bytes = 0, off_partials = 0, off_flags = 0, off_epoch = 0, off_err = 0;
  PeerPlan plan{};                           // peer table + the update's OptState on the reduced buffer
  std::vector<void*> peer_opened;            // bases returned by cudaIpcOpenMemHandle
  uint32_t* h_peer_err = nullptr;            // pinned copy of the barrier time-out word
  bool failed = false;                       // a peer barrier timed out: the replica is out of step with its peers and
                                             // refuses every further step / state read (drl_learner_wait reported it)
  // One handle is used by one host thread at a time (include/drl_b200.h); the documented in-process mode of the
  // reference's launchers nevertheless has actor threads call parameter_sync() -> get_params on the learner's handle
  // while the learner thread trains, and ctypes drops the GIL.  Every entry point therefore takes this lock (the
  // pinned staging buffer h_flat, `pending`, `last_out` and the graph caches are all guarded by it).
  mutable std::recursive_mutex mu;
};

namespace {

int check_not_failed(const drl_learner* h) {
  if (h->failed) {
    set_error("learner handle is in the failed state (a peer-exchange barrier timed out): parameters and optimizer "
              "state are not readable and no further step can run");
    return DRL_ERR_STATE;
  }
  return DRL_OK;
}

Streams streams_of(const drl_learner* h) {
  Streams st;
  st.main = h->compute;
  st.side = h->side;
  for (int i = 0; i < 8; ++i) st.ev[i] = h->fj[i];
  st.par = h->par;
  st.side2 = h->side2;
  for (int i = 0; i < 4; ++i) st.ev2[i] = h->fj2[i];
  st.ev_lstm_grads = (h->peer_on && h->peer_early_ctas > 0) ? h->ev_lstm_grads : nullptr;
  return st;
}

// retile = true: (re)build the weight images first.  A training step always does (the parameters changed in the
// previous apply); the forward-only entry points only when the images are stale.
int enqueue_forward(drl_learner* h, const Inputs& in, int B, int T, bool retile) {
  pdl_break(h->compute);   // whatever precedes (event waits, copies) is not a pdl-aware kernel
  pdl_break(h->side);
  return net_forward(streams_of(h), h->pl, h->params, h->wimg, in, h->act, B, T, h->mode, retile);
}

int enqueue_forward_backward(drl_learner* h, int slot) {
  const Inputs& in = h->slots[slot].in;
  {
    NvtxRange r("drl:forward");
    DRL_TRY(enqueue_forward(h, in, h->B, h->T, true));
  }
  VtraceCfg vc{h->cfg.discount_factor, h->cfg.baseline_loss_coef, h->cfg.entropy_coef, h->cfg.reward_clipping};
  prof_mark(h->compute, "vtrace_losses");
  {
    NvtxRange r("drl:vtrace_losses");
    DRL_TRY(vtrace_losses(h->compute, vc, h->act.policy, h->act.value, in, h->vt, h->bwd.dlogits, h->bwd.dv, h->B,
                          h->T, h->A));
  }
  NvtxRange r("drl:backward");
  DRL_TRY(net_backward(streams_of(h), h->pl, h->params, h->wimg, h->bucket, in, h->act, h->bwd, h->B, h->T, h->mode));
  return DRL_OK;
}

// local_only: the single-replica update on the local bucket even when the peer exchange is on (profiling on one rank)
// early: the backward pass of THIS enqueue recorded ev_lstm_grads (one-graph step): part 0 of the exchange overlaps it
int enqueue_apply(drl_learner* h, int out_row, bool local_only = false, bool early = false) {
  pdl_break(h->compute);
  OptState o_local = h->opt, o_peer = h->plan.o;
  o_local.out = o_peer.out = h->d_out + 8 * out_row;
  if (h->peer_on && !local_only) {
    prof_mark(h->compute, "peer_exchange");
    {
      NvtxRange r("drl:exchange");
      // part 0: [lstm_w .. end) incl. the loss sums -- 96 % of the bucket.  In the one-graph step it runs on its own stream
      // behind the LSTM weight gradient (ev_lstm_grads), i.e. under the rest of the backward pass, with a small grid so that
      // the convolution kernels never queue behind it; otherwise right here.  part 1: [0 .. lstm_w), after the backward pass.
      const int64_t split4 = h->pl.lstm_w / 4, end4 = h->pl.padded_total / 4 + 1;
      if (early) {
        DRL_CUDA_CHECK(cudaStreamWaitEvent(h->xchg, h->ev_lstm_grads, 0));
        DRL_TRY(peer_exchange(h->xchg, h->plan, 0, split4, end4, false, h->peer_early_ctas));
        DRL_CUDA_CHECK(cudaEventRecord(h->ev_xchg_done, h->xchg));
        DRL_CUDA_CHECK(cudaStreamWaitEvent(h->compute, h->ev_xchg_done, 0));
      } else {
        DRL_TRY(peer_exchange(h->compute, h->plan, 0, split4, end4, false, h->peer_early_ctas));
      }
      DRL_TRY(peer_exchange(h->compute, h->plan, 1, 0, split4, true, 148));
    }
    prof_mark(h->compute, "optimizer(rmsprop)");
    NvtxRange r("drl:update");
    DRL_TRY(optimizer_update_only(h->compute, o_peer));
    prof_mark(h->compute, "end");
  } else {
    prof_mark(h->compute, "optimizer(norm+rmsprop)");
    NvtxRange r("drl:update");
    DRL_TRY(optimizer_apply(h->compute, o_local));
    prof_mark(h->compute, "end");
  }
  // no D2H copy node: the update kernel stores the 8 scalars straight into mapped pinned memory (h_out); a memcpy
  // at the end of the graph sat in the ~20 us gap between two steps (tools/timeline.py --back-to-back)
  return DRL_OK;
}

int run_forward_backward(drl_learner* h, int slot) {
  Slot& sl = h->slots[slot];
  if (!sl.has_data) { set_error("slot %d has not been staged", slot); return DRL_ERR_STATE; }
  DRL_CUDA_CHECK(cudaStreamWaitEvent(h->compute, sl.staged, 0));
  DRL_CUDA_CHECK(cudaEventRecord(h->ev_start, h->compute));
  if (h->cfg.use_cuda_graph) {
    if (!h->graph_fb[slot]) {
      // one eager pass first: sets the per-kernel shared-memory attributes outside of stream capture
      // (idempotent: every buffer it writes is fully overwritten by the captured pass)
      DRL_TRY(enqueue_forward_backward(h, slot));
      DRL_TRY(capture_graph(h->compute, &h->graph_fb[slot], [&] { return enqueue_forward_backward(h, slot); }));
    }
    DRL_CUDA_CHECK(cudaGraphLaunch(h->graph_fb[slot], h->compute));
  } else {
    DRL_TRY(enqueue_forward_backward(h, slot));
  }
  DRL_CUDA_CHECK(cudaEventRecord(sl.consumed, h->compute));
  return DRL_OK;
}

int run_apply(drl_learner* h) {
  if (h->cfg.use_cuda_graph) {
    if (!h->graph_apply) {
      DRL_TRY(capture_graph(h->compute, &h->graph_apply, [&] { return enqueue_apply(h, (int)h->slots.size()); }));
    }
    DRL_CUDA_CHECK(cudaGraphLaunch(h->graph_apply, h->compute));
  } else {
    DRL_TRY(enqueue_apply(h, (int)h->slots.size()));
  }
  h->last_out = (int)h->slots.size();
  DRL_CUDA_CHECK(cudaEventRecord(h->ev_stop, h->compute));
  DRL_CUDA_CHECK(cudaEventRecord(h->ev_done, h->compute));
  DRL_CUDA_CHECK(cudaEventRecord(h->ev_done_slot[h->last_out], h->compute));
  h->pending = true;
  h->images_stale = true;
  return DRL_OK;
}

// drl_learner_step*: nothing on the host runs between the backward pass and the update (at N > 1 the peer exchange
// is part of the update), so both go into ONE graph per slot; the scalars land in the slot's own result row.
int run_step(drl_learner* h, int slot) {
  Slot& sl = h->slots[slot];
  if (!sl.has_data) { set_error("slot %d has not been staged", slot); return DRL_ERR_STATE; }
  DRL_CUDA_CHECK(cudaStreamWaitEvent(h->compute, sl.staged, 0));
  DRL_CUDA_CHECK(cudaEventRecord(h->ev_start, h->compute));
  if (h->cfg.use_cuda_graph) {
    if (!h->graph_step[slot]) {
      DRL_TRY(enqueue_forward_backward(h, slot));   // eager pass: per-kernel attributes are set outside of capture
      DRL_TRY(capture_graph(h->compute, &h->graph_step[slot], [&] {
        const int r = enqueue_forward_backward(h, slot);
        return r != DRL_OK ? r : enqueue_apply(h, slot, false, h->peer_on && h->par && h->peer_early_ctas > 0);
      }));
    }
    NvtxRange r("drl:step(graph)");
    DRL_CUDA_CHECK(cudaGraphLaunch(h->graph_step[slot], h->compute));
  } else {
    DRL_TRY(enqueue_forward_backward(h, slot));
    DRL_TRY(enqueue_apply(h, slot, false, h->peer_on && h->par && h->peer_early_ctas > 0));
  }
  h->last_out = slot;
  DRL_CUDA_CHECK(cudaEventRecord(sl.consumed, h->compute));
  DRL_CUDA_CHECK(cudaEventRecord(h->ev_stop, h->compute));
  DRL_CUDA_CHECK(cudaEventRecord(h->ev_done, h->compute));
  DRL_CUDA_CHECK(cudaEventRecord(h->ev_done_slot[slot], h->compute));
  h->pending = true;
  h->images_stale = true;
  return DRL_OK;
}

}  // namespace

extern "C" {

const char* drl_last_error(void) { return get_error(); }

// debug: arm (dev_buf = device buffer of >= 8001 uint64, word 0 = entry counter) or disarm (NULL) the kernel
// start-time trace of common.cuh::pdl_prologue
int drl_debug_trace(void* dev_buf) {
  if (drl_device_count() < 1) { set_error("CUDA device not available (no CPU fallback)"); return DRL_ERR_CUDA; }
  DRL_CUDA_CHECK(cudaDeviceSynchronize());
  for (TraceSetter f : trace_setters()) f(static_cast<unsigned long long*>(dev_buf));
  DRL_CUDA_CHECK(cudaDeviceSynchronize());
  return DRL_OK;
}
const char* drl_version(void) { return "drl_b200 0.4 (sm_100a; tcgen05 kind::f16 split-16 / 3xTF32 gather-GEMMs, FP32-FFMA core, NVLink peer exchange; IMPALA, Ape-X, R2D2, A3C learners)"; }

int drl_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
  return n;
}

int drl_learner_create(const drl_learner_config* cfg, drl_learner** out) {
  if (!cfg || !out) { set_error("null argument"); return DRL_ERR_INVALID; }
  *out = nullptr;
  if (cfg->height != Geo::IH || cfg->width != Geo::IW || cfg->channels != Geo::IC) {
    set_error("only the reference input geometry 84x84x4 is supported (got %dx%dx%d)", cfg->height, cfg->width,
              cfg->channels);
    return DRL_ERR_INVALID;
  }
  if (cfg->lstm_size != Geo::L) { set_error("only lstm_size 256 is supported (got %d)", cfg->lstm_size); return DRL_ERR_INVALID; }
  if (cfg->trajectory < 3 || cfg->trajectory > 32) { set_error("trajectory must be in [3,32]"); return DRL_ERR_INVALID; }
  if (cfg->num_action < 2 || cfg->num_action > 32) { set_error("num_action must be in [2,32]"); return DRL_ERR_INVALID; }
  if (cfg->batch < 1) { set_error("batch must be >= 1"); return DRL_ERR_INVALID; }
  if (cfg->reward_clipping != DRL_REWARD_ABS_ONE && cfg->reward_clipping != DRL_REWARD_SOFT_ASYMMETRIC) {
    set_error("reward_clipping must be DRL_REWARD_ABS_ONE or DRL_REWARD_SOFT_ASYMMETRIC");   // utils.py:45
    return DRL_ERR_INVALID;
  }
  if (cfg->math_mode < 0 || cfg->math_mode > 5) {
    set_error("math_mode must be 0 (default), 1 (FP32 FFMA), 2 (tcgen05 3xTF32), 3 (same, persistent kernels), "
              "4 (same as 2 with TMA-fed conv2/conv3 forward) or 5 (tcgen05 kind::f16 with 16-bit split operands)");
    return DRL_ERR_INVALID;
  }
  if (drl_device_count() <= cfg->device) { set_error("CUDA device %d not available (no CPU fallback)", cfg->device); return DRL_ERR_CUDA; }

  drl_learner* h = new drl_learner();
  h->cfg = *cfg;
  h->mode = (cfg->math_mode == 0) ? DRL_DEFAULT_MATH_MODE_IMPALA : cfg->math_mode;
  if (h->cfg.num_slots < 1) h->cfg.num_slots = 2;
  h->B = cfg->batch; h->T = cfg->trajectory; h->A = cfg->num_action;
  h->M = h->B * h->T; h->Mb = h->B * (h->T - 2);
  h->pl.init(h->A);
  int rc = [&]() -> int {
    DRL_CUDA_CHECK(cudaSetDevice(h->cfg.device));
    DRL_CUDA_CHECK(cudaStreamCreateWithFlags(&h->compute, cudaStreamNonBlocking));
    DRL_CUDA_CHECK(cudaStreamCreateWithFlags(&h->copy, cudaStreamNonBlocking));
    DRL_CUDA_CHECK(cudaStreamCreateWithFlags(&h->side, cudaStreamNonBlocking));
    DRL_CUDA_CHECK(cudaStreamCreateWithFlags(&h->xchg, cudaStreamNonBlocking));
    DRL_CUDA_CHECK(cudaEventCreateWithFlags(&h->ev_lstm_grads, cudaEventDisableTiming));
    DRL_CUDA_CHECK(cudaEventCreateWithFlags(&h->ev_xchg_done, cudaEventDisableTiming));
    if (const char* e = getenv("DRL_B200_PEER_EARLY_CTAS")) h->peer_early_ctas = atoi(e);
    for (int i = 0; i < 8; ++i) DRL_CUDA_CHECK(cudaEventCreateWithFlags(&h->fj[i], cudaEventDisableTiming));
    {
      const char* e = getenv("DRL_B200_SIDE2");
      if (!(e && atoi(e) == 0)) {
        DRL_CUDA_CHECK(cudaStreamCreateWithFlags(&h->side2, cudaStreamNonBlocking));
        for (int i = 0; i < 4; ++i) DRL_CUDA_CHECK(cudaEventCreateWithFlags(&h->fj2[i], cudaEventDisableTiming));
      }
    }
    DRL_CUDA_CHECK(cudaEventCreate(&h->ev_start));
    DRL_CUDA_CHECK(cudaEventCreate(&h->ev_stop));
    DRL_CUDA_CHECK(cudaEventCreateWithFlags(&h->ev_done, cudaEventDisableTiming));
    const size_t M = h->M, Mb = h->Mb, A = h->A, NP = h->pl.padded_total;
    DRL_TRY(dev_alloc(h, &h->params, NP));
    DRL_TRY(dev_alloc(h, &h->ms, NP));
    DRL_TRY(dev_alloc(h, &h->bucket, NP + 4));
    {  // RMSProp slots start at ONE (TF1 RMSPropOptimizer._create_slots)
      std::vector<float> ones(NP, 1.0f);
      DRL_CUDA_CHECK(cudaMemcpy(h->ms, ones.data(), NP * sizeof(float), cudaMemcpyHostToDevice));
    }
    Acts& a = h->act;
    const size_t planes = (h->mode == 4) ? 2 : 1;      // math mode 4: [value plane | tf32 remainder plane]
    DRL_TRY(dev_alloc(h, &a.a1, planes * M * 400 * 32));
    a.a1_lo = (planes == 2) ? a.a1 + M * 400 * 32 : nullptr;
    DRL_TRY(dev_alloc(h, &a.a2, planes * M * 81 * 64));
    a.a2_lo = (planes == 2) ? a.a2 + M * 81 * 64 : nullptr;
    DRL_TRY(dev_alloc(h, &a.a3, M * Geo::FLAT));
    DRL_TRY(dev_alloc(h, &a.e1, A * Geo::EMB));
    DRL_TRY(dev_alloc(h, &a.table, A * Geo::EMB));
    DRL_TRY(dev_alloc(h, &a.zpart, (size_t)kLstmSplits * M * Geo::G4));
    DRL_TRY(dev_alloc(h, &a.gates, M * Geo::G4));
    DRL_TRY(dev_alloc(h, &a.c1, M * Geo::L));
    DRL_TRY(dev_alloc(h, &a.tc1, M * Geo::L));
    DRL_TRY(dev_alloc(h, &a.h1, M * Geo::L));
    DRL_TRY(dev_alloc(h, &a.hid1, 2 * M * Geo::HID));
    DRL_TRY(dev_alloc(h, &a.hid2, 2 * M * Geo::HID));
    DRL_TRY(dev_alloc(h, &a.logits, M * A));
    DRL_TRY(dev_alloc(h, &a.policy, M * A));
    DRL_TRY(dev_alloc(h, &a.value, M));
    if (h->mode == 5 && !(getenv("DRL_B200_LSTM_BULK") && atoi(getenv("DRL_B200_LSTM_BULK")) == 0)) {
      const size_t Mbr = (size_t)h->B * (h->T - 2);
      DRL_TRY(dev_alloc(h, &a.img_xt, lstm_image_bytes(1, (int)M, (int)Mbr)));
      DRL_TRY(dev_alloc(h, &h->bwd.img_dzt, lstm_image_bytes(3, (int)M, (int)Mbr)));
      a.img_rows = (int)M;
    }
    Bwd& b = h->bwd;
    DRL_TRY(dev_alloc(h, &b.dlogits, Mb * 32));
    DRL_TRY(dev_alloc(h, &b.dv, Mb * 32));
    DRL_TRY(dev_alloc(h, &b.dhid2, 2 * Mb * Geo::HID));
    DRL_TRY(dev_alloc(h, &b.dhid1, 2 * Mb * Geo::HID));
    DRL_TRY(dev_alloc(h, &b.dh_part, 2 * Mb * Geo::L));
    DRL_TRY(dev_alloc(h, &b.dz, Mb * Geo::G4));
    DRL_TRY(dev_alloc(h, &b.da3, Mb * Geo::FLAT));
    DRL_TRY(dev_alloc(h, &b.du, Mb * Geo::EMB));
    DRL_TRY(dev_alloc(h, &b.dpre2, A * Geo::EMB));
    DRL_TRY(dev_alloc(h, &b.dpre1, A * Geo::EMB));
    DRL_TRY(dev_alloc(h, &b.da2, Mb * 81 * 64));
    DRL_TRY(dev_alloc(h, &b.da1, Mb * 400 * 32));
    b.wg_part_floats = wgrad_partial_floats(h->B, h->T);
    DRL_TRY(dev_alloc(h, &b.wg_part, b.wg_part_floats));
    DRL_TRY(dev_alloc(h, &b.wg_part2, b.wg_part_floats));
    DRL_TRY(dev_alloc(h, &b.emb_scratch, (size_t)16 * 32 * 256));
    DRL_TRY(dev_alloc(h, &b.dcol, Mb * 81 * 512));
    {
      size_t wb[WeightImages::kCount];
      weight_image_sizes(wb);
      for (int i = 0; i < WeightImages::kCount; ++i) DRL_TRY(dev_alloc(h, &h->wimg.img[i], wb[i]));
    }
    VtraceOut& v = h->vt;
    const size_t nt = (size_t)h->B * (h->T - 2);
    DRL_TRY(dev_alloc(h, &v.vs, nt));
    DRL_TRY(dev_alloc(h, &v.clipped_rho, nt));
    DRL_TRY(dev_alloc(h, &v.vs_plus_1, nt));
    DRL_TRY(dev_alloc(h, &v.pg_adv, nt));
    DRL_TRY(dev_alloc(h, &v.loss_partials, (size_t)cdiv(h->B, 4) * 3));
    DRL_TRY(dev_alloc(h, &v.ticket, 1));
    v.loss_sums = h->bucket + NP;
    DRL_TRY(dev_alloc(h, &h->d_step, 1));
    DRL_TRY(dev_alloc(h, &h->d_lr, 1));
    const size_t out_rows = (size_t)h->cfg.num_slots + 1;
    DRL_CUDA_CHECK(cudaHostAlloc((void**)&h->h_out, out_rows * 8 * sizeof(float), cudaHostAllocMapped));
    h->ev_done_slot.resize(out_rows, nullptr);
    for (auto& e : h->ev_done_slot) DRL_CUDA_CHECK(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    DRL_CUDA_CHECK(cudaHostGetDevicePointer((void**)&h->d_out, h->h_out, 0));
    DRL_CUDA_CHECK(cudaHostAlloc((void**)&h->h_flat, NP * sizeof(float), cudaHostAllocDefault));
    memset(h->h_out, 0, out_rows * 8 * sizeof(float));
    OptState& o = h->opt;
    o.params = h->params; o.ms = h->ms; o.grads = h->bucket; o.n = (int64_t)NP;
    o.nblk = 148 * 4;
    o.npart = o.nblk;
    o.wait_flags = nullptr; o.wait_epoch = nullptr; o.wait_world = 0; o.wait_err = nullptr; o.wait_parts = 0;
    o.wait_err_host = nullptr; o.wait_timeout_ns = 0;
    DRL_TRY(dev_alloc(h, &o.norm_partials, o.nblk));
    o.step = h->d_step; o.lr_cur = h->d_lr; o.out = h->d_out; o.loss_sums = v.loss_sums;
    o.start_lr = cfg->start_learning_rate; o.end_lr = cfg->end_learning_rate; o.learning_frame = cfg->learning_frame;
    o.clip_norm = cfg->gradient_clip_norm; o.baseline_coef = cfg->baseline_loss_coef; o.entropy_coef = cfg->entropy_coef;
    // staging slots (device), caller's batch-major layout
    const size_t BT = (size_t)h->B * h->T;
    h->slots.resize(h->cfg.num_slots);
    h->graph_fb.assign(h->cfg.num_slots, nullptr);
    h->graph_step.assign(h->cfg.num_slots, nullptr);
    for (Slot& s : h->slots) {
      size_t off = 0;
      const size_t o_frames = off; off = align_up(off + BT * Geo::FRAME, 256);
      const size_t o_rew = off; off = align_up(off + BT * 4, 256);
      const size_t o_act = off; off = align_up(off + BT * 4, 256);
      const size_t o_done = off; off = align_up(off + BT, 256);
      const size_t o_mu = off; off = align_up(off + BT * A * 4, 256);
      const size_t o_pa = off; off = align_up(off + BT * 4, 256);
      const size_t o_h = off; off = align_up(off + BT * Geo::L * 4, 256);
      const size_t o_c = off; off = align_up(off + BT * Geo::L * 4, 256);
      DRL_TRY(dev_alloc(h, &s.base, off));
      s.in.frames = s.base + o_frames;
      s.in.reward = reinterpret_cast<float*>(s.base + o_rew);
      s.in.action = reinterpret_cast<int32_t*>(s.base + o_act);
      s.in.done = s.base + o_done;
      s.in.mu = reinterpret_cast<float*>(s.base + o_mu);
      s.in.pa = reinterpret_cast<int32_t*>(s.base + o_pa);
      s.in.h0 = reinterpret_cast<float*>(s.base + o_h);
      s.in.c0 = reinterpret_cast<float*>(s.base + o_c);
      DRL_CUDA_CHECK(cudaEventCreateWithFlags(&s.staged, cudaEventDisableTiming));
      DRL_CUDA_CHECK(cudaEventCreateWithFlags(&s.consumed, cudaEventDisableTiming));
    }
    DRL_CUDA_CHECK(cudaDeviceSynchronize());
    return DRL_OK;
  }();
  if (rc != DRL_OK) {
    std::string keep = get_error();
    drl_learner_destroy(h);
    set_error("%s", keep.c_str());
    return rc;
  }
  *out = h;
  return DRL_OK;
}

int drl_learner_destroy(drl_learner* h) {
  if (!h) return DRL_OK;
  cudaSetDevice(h->cfg.device);
  cudaDeviceSynchronize();
  for (auto g : h->graph_fb) if (g) cudaGraphExecDestroy(g);
  for (auto g : h->graph_step) if (g) cudaGraphExecDestroy(g);
  if (h->graph_apply) cudaGraphExecDestroy(h->graph_apply);
  for (Slot& s : h->slots) {
    if (s.staged) cudaEventDestroy(s.staged);
    if (s.consumed) cudaEventDestroy(s.consumed);
  }
  for (void* p : h->peer_opened) cudaIpcCloseMemHandle(p);
  if (h->comm) cudaFree(h->comm);
  if (h->h_peer_err) cudaFreeHost(h->h_peer_err);
  for (void* p : h->allocs) cudaFree(p);
  if (h->h_out) cudaFreeHost(h->h_out);
  if (h->h_flat) cudaFreeHost(h->h_flat);
  if (h->ev_start) cudaEventDestroy(h->ev_start);
  if (h->ev_stop) cudaEventDestroy(h->ev_stop);
  if (h->ev_done) cudaEventDestroy(h->ev_done);
  for (auto e : h->ev_done_slot) if (e) cudaEventDestroy(e);
  for (int i = 0; i < 8; ++i) if (h->fj[i]) cudaEventDestroy(h->fj[i]);
  for (int i = 0; i < 4; ++i) if (h->fj2[i]) cudaEventDestroy(h->fj2[i]);
  if (h->side2) cudaStreamDestroy(h->side2);
  if (h->side) cudaStreamDestroy(h->side);
  if (h->xchg) cudaStreamDestroy(h->xchg);
  if (h->ev_lstm_grads) cudaEventDestroy(h->ev_lstm_grads);
  if (h->ev_xchg_done) cudaEventDestroy(h->ev_xchg_done);
  if (h->compute) cudaStreamDestroy(h->compute);
  if (h->copy) cudaStreamDestroy(h->copy);
  cudaGetLastError();
  delete h;
  return DRL_OK;
}

int drl_learner_param_count(const drl_learner* h, int64_t* n) {
  DRL_ENTER(h);
  if (!n) { set_error("null argument"); return DRL_ERR_INVALID; }
  *n = h->pl.packed_total;
  return DRL_OK;
}

int drl_learner_set_params(drl_learner* h, const float* host_flat, int64_t n) {
  DRL_ENTER(h);
  if (!host_flat || n != h->pl.packed_total) { set_error("set_params: expected %lld floats, got %lld", (long long)h->pl.packed_total, (long long)n); return DRL_ERR_INVALID; }
  DRL_TRY(upload_flat(h->pl, h->h_flat, h->compute, h->params, host_flat));
  h->images_stale = true;
  return DRL_OK;
}
int drl_learner_get_params(drl_learner* h, float* host_flat, int64_t n) {
  DRL_ENTER(h);
  DRL_TRY(check_not_failed(h));
  if (!host_flat || n != h->pl.packed_total) { set_error("get_params: expected %lld floats", (long long)h->pl.packed_total); return DRL_ERR_INVALID; }
  return download_flat(h->pl, h->h_flat, h->compute, h->params, host_flat);
}
int drl_learner_set_opt_state(drl_learner* h, const float* host_ms_flat, int64_t n, int64_t step) {
  DRL_ENTER(h);
  if (!host_ms_flat || n != h->pl.packed_total) { set_error("set_opt_state: expected %lld floats", (long long)h->pl.packed_total); return DRL_ERR_INVALID; }
  DRL_TRY(upload_flat(h->pl, h->h_flat, h->compute, h->ms, host_ms_flat, 1.0f));
  long long st = step;
  DRL_CUDA_CHECK(cudaMemcpy(h->d_step, &st, sizeof(st), cudaMemcpyHostToDevice));
  return DRL_OK;
}
int drl_learner_get_opt_state(drl_learner* h, float* host_ms_flat, int64_t n, int64_t* step) {
  DRL_ENTER(h);
  DRL_TRY(check_not_failed(h));
  if (n != h->pl.packed_total) { set_error("get_opt_state: expected %lld floats", (long long)h->pl.packed_total); return DRL_ERR_INVALID; }
  if (host_ms_flat) DRL_TRY(download_flat(h->pl, h->h_flat, h->compute, h->ms, host_ms_flat));
  if (step) {
    long long st = 0;
    DRL_CUDA_CHECK(cudaStreamSynchronize(h->compute));
    DRL_CUDA_CHECK(cudaMemcpy(&st, h->d_step, sizeof(st), cudaMemcpyDeviceToHost));
    *step = st;
  }
  return DRL_OK;
}
int drl_learner_get_grads(drl_learner* h, float* host_flat, int64_t n) {
  DRL_ENTER(h);
  DRL_TRY(check_not_failed(h));
  if (!host_flat || n != h->pl.packed_total) { set_error("get_grads: expected %lld floats", (long long)h->pl.packed_total); return DRL_ERR_INVALID; }
  return download_flat(h->pl, h->h_flat, h->compute, h->peer_on ? reinterpret_cast<float*>(h->comm) : h->bucket, host_flat);
}

int drl_learner_stage(drl_learner* h, int32_t slot, const uint8_t* state, const float* reward, const int32_t* action,
                      const uint8_t* done, const float* behavior_policy, const int32_t* previous_action,
                      const float* initial_h, const float* initial_c) {
  DRL_ENTER(h);
  if (slot < 0 || slot >= (int)h->slots.size()) { set_error("slot %d out of range", slot); return DRL_ERR_INVALID; }
  if (!state || !reward || !action || !done || !behavior_policy || !previous_action || !initial_h || !initial_c) {
    set_error("stage: null input pointer");
    return DRL_ERR_INVALID;
  }
  NvtxRange nvtx_r("drl:stage");
  Slot& s = h->slots[slot];
  const size_t BT = (size_t)h->B * h->T;
  // do not overwrite a slot the compute stream is still reading
  DRL_CUDA_CHECK(cudaStreamWaitEvent(h->copy, s.consumed, 0));
  auto cp = [&](const void* dst, const void* src, size_t bytes) -> cudaError_t {
    return cudaMemcpyAsync(const_cast<void*>(dst), src, bytes, cudaMemcpyHostToDevice, h->copy);
  };
  DRL_CUDA_CHECK(cp(s.in.frames, state, BT * Geo::FRAME));
  DRL_CUDA_CHECK(cp(s.in.reward, reward, BT * 4));
  DRL_CUDA_CHECK(cp(s.in.action, action, BT * 4));
  DRL_CUDA_CHECK(cp(s.in.done, done, BT));
  DRL_CUDA_CHECK(cp(s.in.mu, behavior_policy, BT * h->A * 4));
  DRL_CUDA_CHECK(cp(s.in.pa, previous_action, BT * 4));
  DRL_CUDA_CHECK(cp(s.in.h0, initial_h, BT * Geo::L * 4));
  DRL_CUDA_CHECK(cp(s.in.c0, initial_c, BT * Geo::L * 4));
  DRL_CUDA_CHECK(cudaEventRecord(s.staged, h->copy));
  s.has_data = true;
  return DRL_OK;
}

int drl_learner_forward_backward(drl_learner* h, int32_t slot) {
  DRL_ENTER(h);
  DRL_TRY(check_not_failed(h));
  if (slot < 0 || slot >= (int)h->slots.size()) { set_error("slot %d out of range", slot); return DRL_ERR_INVALID; }
  return run_forward_backward(h, slot);
}

int drl_learner_grad_bucket(drl_learner* h, void** dev_ptr, int64_t* count) {
  DRL_ENTER(h);
  if (dev_ptr) *dev_ptr = h->bucket;
  if (count) *count = h->pl.padded_total + 4;
  return DRL_OK;
}

int drl_learner_reduced_bucket(drl_learner* h, void** dev_ptr, int64_t* count) {
  DRL_ENTER(h);
  if (dev_ptr) *dev_ptr = h->peer_on ? static_cast<void*>(h->comm) : static_cast<void*>(h->bucket);
  if (count) *count = h->pl.padded_total + 4;
  return DRL_OK;
}

int drl_learner_apply(drl_learner* h) {
  DRL_ENTER(h);
  DRL_TRY(check_not_failed(h));
  return run_apply(h);
}

// ---- gradient exchange over NVLink peer memory (peer.cu) -------------------------------------------------------
int drl_learner_peer_export(drl_learner* h, void* handles, int64_t bytes) {
  DRL_ENTER(h);
  if (!handles || bytes != 2 * (int64_t)sizeof(cudaIpcMemHandle_t)) { set_error("peer_export: expected a %d-byte buffer", (int)(2 * sizeof(cudaIpcMemHandle_t))); return DRL_ERR_INVALID; }
  if (!h->comm) {
    const size_t red = align_up((size_t)(h->pl.padded_total + 4) * sizeof(float), 256);
    h->off_partials = red;
    h->off_flags = h->off_partials + align_up((size_t)kPeerParts * kMaxPeers * h->peer_nblk * sizeof(float), 256);
    h->off_epoch = h->off_flags + 2 * kPeerParts * kMaxPeers * sizeof(uint32_t);
    h->off_err = h->off_epoch + 4 * kPeerParts * sizeof(uint32_t);
    h->comm_bytes = h->off_err + 256;
    DRL_CUDA_CHECK(cudaMalloc((void**)&h->comm, h->comm_bytes));
    DRL_CUDA_CHECK(cudaMemset(h->comm, 0, h->comm_bytes));
    DRL_CUDA_CHECK(cudaHostAlloc((void**)&h->h_peer_err, sizeof(uint32_t), cudaHostAllocMapped));   // zero-copy too
    *h->h_peer_err = 0;
  }
  cudaIpcMemHandle_t hd[2];
  DRL_CUDA_CHECK(cudaIpcGetMemHandle(&hd[0], h->bucket));
  DRL_CUDA_CHECK(cudaIpcGetMemHandle(&hd[1], h->comm));
  memcpy(handles, hd, sizeof(hd));
  return DRL_OK;
}

int drl_learner_peer_import(drl_learner* h, int32_t rank, int32_t world, const void* all_handles, int64_t bytes) {
  DRL_ENTER(h);
  if (world < 2 || world > kMaxPeers || rank < 0 || rank >= world) { set_error("peer_import: bad rank %d / world %d (max %d)", rank, world, kMaxPeers); return DRL_ERR_INVALID; }
  if (!all_handles || bytes != (int64_t)world * 2 * (int64_t)sizeof(cudaIpcMemHandle_t)) { set_error("peer_import: expected world x %d bytes", (int)(2 * sizeof(cudaIpcMemHandle_t))); return DRL_ERR_INVALID; }
  if (!h->comm) { set_error("peer_import before peer_export"); return DRL_ERR_STATE; }
  if (h->peer_on) { set_error("peer exchange already set up"); return DRL_ERR_STATE; }
  DRL_CUDA_CHECK(cudaDeviceSynchronize());
  const cudaIpcMemHandle_t* hd = static_cast<const cudaIpcMemHandle_t*>(all_handles);
  for (int p = 0; p < world; ++p) {
    float* bucket = h->bucket;
    uint8_t* comm = h->comm;
    if (p != rank) {
      void *b = nullptr, *c = nullptr;
      DRL_CUDA_CHECK(cudaIpcOpenMemHandle(&b, hd[2 * p], cudaIpcMemLazyEnablePeerAccess));
      h->peer_opened.push_back(b);
      DRL_CUDA_CHECK(cudaIpcOpenMemHandle(&c, hd[2 * p + 1], cudaIpcMemLazyEnablePeerAccess));
      h->peer_opened.push_back(c);
      bucket = static_cast<float*>(b);
      comm = static_cast<uint8_t*>(c);
    }
    h->plan.t.bucket[p] = bucket;
    h->plan.t.reduced[p] = reinterpret_cast<float*>(comm);
    h->plan.t.partials[p] = reinterpret_cast<float*>(comm + h->off_partials);
    h->plan.t.flags[p] = reinterpret_cast<uint32_t*>(comm + h->off_flags);
    h->plan.t.epoch[p] = reinterpret_cast<uint32_t*>(comm + h->off_epoch);
    h->plan.t.err[p] = reinterpret_cast<uint32_t*>(comm + h->off_err);
  }
  DRL_CUDA_CHECK(cudaHostGetDevicePointer((void**)&h->plan.t.err_host, h->h_peer_err, 0));   // host-visible copy
  {
    const char* e = getenv("DRL_B200_PEER_TIMEOUT_S");
    double sec = e ? atof(e) : 600.0;
    if (!(sec > 0.0)) sec = 600.0;
    h->plan.t.timeout_ns = (unsigned long long)(sec * 1e9);
  }
  h->plan.rank = rank;
  h->plan.world = world;
  h->plan.nblk = h->peer_nblk;
  OptState& po = h->plan.o;
  po = h->opt;
  po.grads = reinterpret_cast<float*>(h->comm);
  po.norm_partials = reinterpret_cast<float*>(h->comm + h->off_partials);
  po.npart = kPeerParts * world * h->peer_nblk;
  po.loss_sums = reinterpret_cast<float*>(h->comm) + h->pl.padded_total;
  po.wait_flags = h->plan.t.flags[rank];
  po.wait_epoch = h->plan.t.epoch[rank];
  po.wait_world = world;
  po.wait_err = h->plan.t.err[rank];
  po.wait_err_host = h->plan.t.err_host;
  po.wait_timeout_ns = h->plan.t.timeout_ns;
  po.wait_parts = kPeerParts;
  // graphs captured so far do not contain the exchange
  for (auto& g : h->graph_step) if (g) { cudaGraphExecDestroy(g); g = nullptr; }
  if (h->graph_apply) { cudaGraphExecDestroy(h->graph_apply); h->graph_apply = nullptr; }
  h->peer_on = true;
  return DRL_OK;
}

int drl_learner_peer_disable(drl_learner* h) {
  DRL_ENTER(h);
  DRL_CUDA_CHECK(cudaDeviceSynchronize());
  for (void* p : h->peer_opened) cudaIpcCloseMemHandle(p);
  h->peer_opened.clear();
  cudaGetLastError();
  if (h->peer_on) {
    for (auto& g : h->graph_step) if (g) { cudaGraphExecDestroy(g); g = nullptr; }
    if (h->graph_apply) { cudaGraphExecDestroy(h->graph_apply); h->graph_apply = nullptr; }
  }
  h->peer_on = false;
  return DRL_OK;
}

int drl_learner_stream(drl_learner* h, void** stream) {
  DRL_ENTER(h);
  if (!stream) { set_error("null argument"); return DRL_ERR_INVALID; }
  *stream = h->compute;
  return DRL_OK;
}

int drl_learner_step_async(drl_learner* h, int32_t slot) {
  DRL_ENTER(h);
  DRL_TRY(check_not_failed(h));
  if (slot < 0 || slot >= (int)h->slots.size()) { set_error("slot %d out of range", slot); return DRL_ERR_INVALID; }
  return run_step(h, slot);
}

static int collect(drl_learner* h, int row, drl_step_out* out) {
  DRL_CUDA_CHECK(cudaEventSynchronize(h->ev_done_slot[row]));
  if (h->peer_on && h->h_peer_err && *h->h_peer_err) {
    h->failed = true;
    set_error("peer exchange: rank %d never reached the barrier within %.0f s (DRL_B200_PEER_TIMEOUT_S); this replica "
              "skipped the update and is out of step with its peers: destroy the handle",
              (int)*h->h_peer_err - 1, (double)h->plan.t.timeout_ns * 1e-9);
    return DRL_ERR_STATE;
  }
  if (out) {
    const float* r = h->h_out + 8 * row;
    out->pi_loss = r[0];
    out->baseline_loss = r[1];
    out->entropy = r[2];
    out->learning_rate = r[3];
    out->grad_norm = r[4];
    out->total_loss = r[5];
    out->step = result_row_step(r);
  }
  return DRL_OK;
}

int drl_learner_wait(drl_learner* h, drl_step_out* out) {
  DRL_ENTER(h);
  if (!h->pending) { set_error("wait: no step in flight"); return DRL_ERR_STATE; }
  h->pending = false;
  return collect(h, h->last_out, out);
}

int drl_learner_wait_slot(drl_learner* h, int32_t slot, drl_step_out* out) {
  DRL_ENTER(h);
  if (slot < 0 || slot >= (int)h->slots.size()) { set_error("slot %d out of range", slot); return DRL_ERR_INVALID; }
  if (slot == h->last_out) h->pending = false;
  return collect(h, slot, out);
}

int drl_learner_step(drl_learner* h, int32_t slot, drl_step_out* out) {
  DRL_ENTER(h);
  DRL_TRY(drl_learner_step_async(h, slot));
  return drl_learner_wait(h, out);
}

int drl_learner_forward(drl_learner* h, int32_t slot, float* policy, float* value) {
  DRL_ENTER(h);
  if (slot < 0 || slot >= (int)h->slots.size()) { set_error("slot %d out of range", slot); return DRL_ERR_INVALID; }
  Slot& s = h->slots[slot];
  if (!s.has_data) { set_error("slot %d has not been staged", slot); return DRL_ERR_STATE; }
  DRL_CUDA_CHECK(cudaStreamWaitEvent(h->compute, s.staged, 0));
  DRL_TRY(enqueue_forward(h, s.in, h->B, h->T, h->images_stale));
  h->images_stale = false;
  DRL_CUDA_CHECK(cudaEventRecord(s.consumed, h->compute));
  // time-major device rows -> batch-major host arrays
  const int B = h->B, T = h->T, A = h->A;
  std::vector<float> pol((size_t)B * T * A), val((size_t)B * T);
  DRL_CUDA_CHECK(cudaMemcpyAsync(pol.data(), h->act.policy, pol.size() * 4, cudaMemcpyDeviceToHost, h->compute));
  DRL_CUDA_CHECK(cudaMemcpyAsync(val.data(), h->act.value, val.size() * 4, cudaMemcpyDeviceToHost, h->compute));
  DRL_CUDA_CHECK(cudaStreamSynchronize(h->compute));
  for (int t = 0; t < T; ++t)
    for (int b = 0; b < B; ++b) {
      const size_t m = (size_t)t * B + b, s2 = (size_t)b * T + t;
      if (policy) memcpy(policy + s2 * A, pol.data() + m * A, A * sizeof(float));
      if (value) value[s2] = val[m];
    }
  return DRL_OK;
}

int drl_learner_taps(drl_learner* h, float* vs, float* clipped_rho, float* vs_plus_1, float* pg_advantage) {
  DRL_ENTER(h);
  const size_t n = (size_t)h->B * (h->T - 2) * sizeof(float);
  DRL_CUDA_CHECK(cudaStreamSynchronize(h->compute));
  if (vs) DRL_CUDA_CHECK(cudaMemcpy(vs, h->vt.vs, n, cudaMemcpyDeviceToHost));
  if (clipped_rho) DRL_CUDA_CHECK(cudaMemcpy(clipped_rho, h->vt.clipped_rho, n, cudaMemcpyDeviceToHost));
  if (vs_plus_1) DRL_CUDA_CHECK(cudaMemcpy(vs_plus_1, h->vt.vs_plus_1, n, cudaMemcpyDeviceToHost));
  if (pg_advantage) DRL_CUDA_CHECK(cudaMemcpy(pg_advantage, h->vt.pg_adv, n, cudaMemcpyDeviceToHost));
  return DRL_OK;
}

int drl_learner_read_buffer(drl_learner* h, const char* name, float* host_dst, int64_t n) {
  DRL_ENTER(h);
  if (!name || !host_dst) { set_error("null argument"); return DRL_ERR_INVALID; }
  const size_t M = h->M, Mb = h->Mb, A = h->A;
  const NamedBuffer tab[] = {
      {"a1", h->act.a1, M * 400 * 32}, {"a2", h->act.a2, M * 81 * 64}, {"a3", h->act.a3, M * Geo::FLAT},
      {"emb", h->act.table, A * Geo::EMB}, {"e1", h->act.e1, A * Geo::EMB},
      {"gates", h->act.gates, M * Geo::G4}, {"h1", h->act.h1, M * Geo::L}, {"c1", h->act.c1, M * Geo::L},
      {"hid1", h->act.hid1, 2 * M * Geo::HID}, {"hid2", h->act.hid2, 2 * M * Geo::HID},
      {"logits", h->act.logits, M * A}, {"policy", h->act.policy, M * A}, {"value", h->act.value, M},
      {"dlogits", h->bwd.dlogits, Mb * 32}, {"dv", h->bwd.dv, Mb * 32}, {"dhid2", h->bwd.dhid2, 2 * Mb * Geo::HID},
      {"dhid1", h->bwd.dhid1, 2 * Mb * Geo::HID}, {"dh_part", h->bwd.dh_part, 2 * Mb * Geo::L},
      {"dz", h->bwd.dz, Mb * Geo::G4}, {"da3", h->bwd.da3, Mb * Geo::FLAT}, {"du", h->bwd.du, Mb * Geo::EMB},
      {"da2", h->bwd.da2, Mb * 81 * 64}, {"da1", h->bwd.da1, Mb * 400 * 32}};
  return read_named_buffer(h->compute, tab, sizeof(tab) / sizeof(tab[0]), name, host_dst, n);
}

int drl_learner_act(drl_learner* h, int32_t n, const uint8_t* state, const int32_t* previous_action,
                    const float* h_in, const float* c_in, float* policy, float* h_out, float* c_out) {
  DRL_ENTER(h);
  if (n < 1 || n > h->M) { set_error("act: n must be in [1, %d]", h->M); return DRL_ERR_INVALID; }
  if (!state || !previous_action || !h_in || !c_in) { set_error("act: null input pointer"); return DRL_ERR_INVALID; }
  // reuse staging slot 0 as an [n, 1] batch (B = n, T = 1 makes the time-major/batch-major remap the identity)
  Slot& s = h->slots[0];
  DRL_CUDA_CHECK(cudaStreamSynchronize(h->compute));
  DRL_CUDA_CHECK(cudaStreamSynchronize(h->copy));
  auto cp = [&](const void* dst, const void* src, size_t bytes) -> cudaError_t {
    return cudaMemcpyAsync(const_cast<void*>(dst), src, bytes, cudaMemcpyHostToDevice, h->compute);
  };
  DRL_CUDA_CHECK(cp(s.in.frames, state, (size_t)n * Geo::FRAME));
  DRL_CUDA_CHECK(cp(s.in.pa, previous_action, (size_t)n * 4));
  DRL_CUDA_CHECK(cp(s.in.h0, h_in, (size_t)n * Geo::L * 4));
  DRL_CUDA_CHECK(cp(s.in.c0, c_in, (size_t)n * Geo::L * 4));
  s.has_data = false;   // the slot no longer holds a training batch
  DRL_TRY(enqueue_forward(h, s.in, n, 1, h->images_stale));
  h->images_stale = false;
  if (policy) DRL_CUDA_CHECK(cudaMemcpyAsync(policy, h->act.policy, (size_t)n * h->A * 4, cudaMemcpyDeviceToHost, h->compute));
  if (h_out) DRL_CUDA_CHECK(cudaMemcpyAsync(h_out, h->act.h1, (size_t)n * Geo::L * 4, cudaMemcpyDeviceToHost, h->compute));
  if (c_out) DRL_CUDA_CHECK(cudaMemcpyAsync(c_out, h->act.c1, (size_t)n * Geo::L * 4, cudaMemcpyDeviceToHost, h->compute));
  DRL_CUDA_CHECK(cudaStreamSynchronize(h->compute));
  return DRL_OK;
}

int drl_learner_profile_step(drl_learner* h, int32_t slot, char* names, int64_t names_len, float* ms,
                             int32_t max_kernels, int32_t* count) {
  DRL_ENTER(h);
  if (slot < 0 || slot >= (int)h->slots.size()) { set_error("slot %d out of range", slot); return DRL_ERR_INVALID; }
  if (!names || !ms || !count) { set_error("null argument"); return DRL_ERR_INVALID; }
  Slot& sl = h->slots[slot];
  if (!sl.has_data) { set_error("slot %d has not been staged", slot); return DRL_ERR_STATE; }
  DRL_CUDA_CHECK(cudaStreamWaitEvent(h->compute, sl.staged, 0));
  DRL_CUDA_CHECK(cudaStreamSynchronize(h->compute));
  prof_begin();
  const bool par_saved = h->par;
  h->par = false;                       // serial: the event-to-event times are then per kernel
  int rc = enqueue_forward_backward(h, slot);
  if (rc == DRL_OK) rc = enqueue_apply(h, (int)h->slots.size(), /*local_only=*/true);   // one rank may profile alone
  h->par = par_saved;
  DRL_TRY(prof_end(h->compute, rc, names, names_len, ms, max_kernels, count));
  h->pending = false;
  return DRL_OK;
}

int drl_learner_last_step_ms(drl_learner* h, float* ms) {
  DRL_ENTER(h);
  if (!ms) { set_error("null argument"); return DRL_ERR_INVALID; }
  DRL_CUDA_CHECK(cudaEventSynchronize(h->ev_stop));
  DRL_CUDA_CHECK(cudaEventElapsedTime(ms, h->ev_start, h->ev_stop));
  return DRL_OK;
}

int drl_learner_launches_per_step(const drl_learner* h, int32_t* n) {
  DRL_ENTER(h);
  if (!n) { set_error("null argument"); return DRL_ERR_INVALID; }
  // forward + V-trace/loss kernel + backward + 2 optimizer kernels (valid after the first step)
  *n = forward_launch_count() + 1 + backward_launch_count() + 2;
  return DRL_OK;
}

}  // extern "C"
