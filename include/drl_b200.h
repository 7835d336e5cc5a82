/*
 * drl_b200.h -- C-ABI of the B200-native learner hot paths: IMPALA (the headline path), then the Ape-X DQN, R2D2 and
 * A3C learner steps and the prioritized-replay index (SURVEY.md section 8(f)).
 *
 * The reference (chagmgang/distributed_reinforcement_learning @ 1890ce4) has no FFI: its hot
 * path is a Python call surface over a TF1 graph.  This header is what a replacement of that
 * path binds (ctypes today; see INTEGRATION.md).  Every entry point names the reference
 * interface it replaces (file:line under /root/reference).
 *
 * Conventions: extern "C"; plain pointers and sizes; every function returns int
 * (0 = ok, <0 = error, text via drl_last_error()); no exception crosses the boundary;
 * pointers are caller-owned unless produced by a *_create; a handle is used by one host
 * thread at a time (the ring is the exception: it is multi-producer / single-consumer safe).
 * "host" pointers are CPU memory (pinned or pageable), "dev" pointers are CUDA device memory.
 * There is NO CPU fallback: without a CUDA device every compute entry point fails with
 * DRL_ERR_CUDA.
 */
#ifndef DRL_B200_H_
#define DRL_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DRL_OK 0
#define DRL_ERR_INVALID (-1) /* bad argument / unsupported configuration */
#define DRL_ERR_CUDA (-2)    /* CUDA runtime error (text in drl_last_error) */
#define DRL_ERR_STATE (-3)   /* call out of order (e.g. step before stage) */
#define DRL_ERR_TIMEOUT (-4) /* ring wait timed out */

#define DRL_REWARD_ABS_ONE 0         /* agent/impala.py:45-46 */
#define DRL_REWARD_SOFT_ASYMMETRIC 1 /* agent/impala.py:47-49 */

/* Last error text of the calling thread ("" if none). */
const char* drl_last_error(void);
/* Library version string, e.g. "drl_b200 0.1 sm_100a". */
const char* drl_version(void);
/* Number of CUDA devices visible (0 when there is none / no driver). */
int drl_device_count(void);

/* ------------------------------------------------------------------------------------------
 * Learner: replaces impala.Agent's learner graph + Agent.train (agent/impala.py:11-103,132-148)
 * over model/impala_actor_critic.py:33-118 and optimizer/vtrace.py:29-126.
 * ------------------------------------------------------------------------------------------ */
typedef struct drl_learner drl_learner;

typedef struct drl_learner_config {
  int32_t batch;              /* B trajectories per step on THIS device (config.json:130)      */
  int32_t trajectory;         /* T, 3..32 (config.json:136)                                      */
  int32_t height, width, channels; /* 84,84,4 -- only this geometry is supported (config.json:133) */
  int32_t num_action;         /* A, 2..32 (config.json:134)                                     */
  int32_t lstm_size;          /* 256 -- only this size is supported (config.json:137)           */
  float discount_factor;      /* agent/impala.py:51                                             */
  float start_learning_rate;  /* agent/impala.py:96                                             */
  float end_learning_rate;
  double learning_frame;      /* decay_steps of tf.train.polynomial_decay                       */
  float baseline_loss_coef;   /* agent/impala.py:93                                             */
  float entropy_coef;
  float gradient_clip_norm;   /* agent/impala.py:98                                             */
  int32_t reward_clipping;    /* DRL_REWARD_*                                                   */
  int32_t device;             /* CUDA device ordinal                                            */
  int32_t num_slots;          /* device staging slots for stream-overlapped H2D (>=1, default 2) */
  int32_t use_cuda_graph;     /* 1: capture forward+backward(+apply) into CUDA graphs           */
  int32_t math_mode;          /* 0 = default (5); 1 = FP32 FFMA; 2 = tcgen05 3xTF32; 3 = same, persistent kernels;
                                 4 = as 2 with TMA-fed conv2/conv3 forward (experimental); 5 = tcgen05 kind::f16 on
                                 bf16 hi/lo split operands (three products, fp32-grade) + TMA-fed conv1 kernels +
                                 bulk-fed LSTM weight gradient */
} drl_learner_config;

/* Results of one step: the 4 floats Agent.train returns (agent/impala.py:144-148) + grad norm. */
typedef struct drl_step_out {
  float pi_loss;
  float baseline_loss;
  float entropy;
  float learning_rate;
  float grad_norm;   /* global norm before clipping (tf.clip_by_global_norm's second output) */
  float total_loss;  /* agent/impala.py:93 */
  int64_t step;      /* global_step AFTER this update (agent/impala.py:95,100) */
} drl_step_out;

/* impala.Agent.__init__ (agent/impala.py:11-103): allocates parameters (zeros), RMSProp slots
 * (ones, TF1 semantics), activations, staging slots, streams and events on cfg->device. */
int drl_learner_create(const drl_learner_config* cfg, drl_learner** out);
int drl_learner_destroy(drl_learner* h);

/* Number of learnable floats (4,153,267 for the reference geometry, SURVEY.md App. A.6). */
int drl_learner_param_count(const drl_learner* h, int64_t* n);
/* Flat float32 parameter vector in TF layouts / TF variable-creation order
 * (conv HWIO, dense [in,out], LSTM [in+h, 4*units] gate order i,j,f,o); replaces
 * global_variables_initializer / Saver.restore (agent/impala.py:105-109,114-116). */
int drl_learner_set_params(drl_learner* h, const float* host_flat, int64_t n);
int drl_learner_get_params(drl_learner* h, float* host_flat, int64_t n);      /* parameter_sync / Saver.save */
/* RMSProp "ms" slots (same flat layout) and global_step -- optimizer state of agent/impala.py:95-100. */
int drl_learner_set_opt_state(drl_learner* h, const float* host_ms_flat, int64_t n, int64_t step);
int drl_learner_get_opt_state(drl_learner* h, float* host_ms_flat, int64_t n, int64_t* step);
/* Gradient of total_loss (before clipping; summed over ranks if an all-reduce ran) -- parity tap
 * for optimizer.compute_gradients (agent/impala.py:98). */
int drl_learner_get_grads(drl_learner* h, float* host_flat, int64_t n);

/* Feed of Agent.train (agent/impala.py:134-142): asynchronous H2D of one batch-major batch
 * into device staging slot `slot` on the copy stream.  state u8 [B,T,H,W,C]; reward f32 [B,T];
 * action i32 [B,T]; done u8/bool [B,T]; behavior_policy f32 [B,T,A]; previous_action i32 [B,T];
 * initial_h, initial_c f32 [B,T,L].  The /255 normalisation (agent/impala.py:133) happens on
 * the device.  Host buffers must stay valid until the next drl_learner_wait / _step on the slot. */
int drl_learner_stage(drl_learner* h, int32_t slot,
                      const uint8_t* state, const float* reward, const int32_t* action,
                      const uint8_t* done, const float* behavior_policy,
                      const int32_t* previous_action, const float* initial_h, const float* initial_c);

/* sess.run([pi_loss, baseline_loss, entropy, learning_rate, train_op]) (agent/impala.py:144-146):
 * forward, V-trace, losses, backward, global-norm clip, RMSProp, step += 1 on slot `slot`;
 * blocks until the scalars are on the host. */
int drl_learner_step(drl_learner* h, int32_t slot, drl_step_out* out);
/* Same, asynchronous: enqueue on the compute stream; drl_learner_wait collects the scalars. */
int drl_learner_step_async(drl_learner* h, int32_t slot);
int drl_learner_wait(drl_learner* h, drl_step_out* out);
/* (new) Result of the most recent drl_learner_step_async on `slot` (blocks until that step is done).  Every slot has
 * its own result record, so with two slots the host can keep two steps in flight and read step i-1 while step i runs. */
int drl_learner_wait_slot(drl_learner* h, int32_t slot, drl_step_out* out);

/* Data-parallel split of the step (SURVEY.md 8(e)): forward+backward leaves the local gradient
 * sum in the bucket; the caller all-reduces (SUM) `count` floats at `dev_ptr` across ranks on
 * `stream` (the bucket tail carries the 3 loss sums so one collective covers them); apply does
 * clip + RMSProp on the reduced bucket. */
int drl_learner_forward_backward(drl_learner* h, int32_t slot);
int drl_learner_grad_bucket(drl_learner* h, void** dev_ptr, int64_t* count);
int drl_learner_apply(drl_learner* h);          /* async; follow with drl_learner_wait */
/* (new) Device pointer of the bucket the update reads: the peer exchange's `reduced` buffer when that exchange is
 * on, else the gradient bucket itself (already all-reduced by the caller).  Same shape as drl_learner_grad_bucket.
 * Lets a harness compare the fused exchange with a library all-reduce of the saved local buckets (bench.py,
 * tests/test_gpu_multi.py). */
int drl_learner_reduced_bucket(drl_learner* h, void** dev_ptr, int64_t* count);
/* (new) Gradient exchange over NVLink peer memory, fused with the global-norm partials, INSTEAD of an all-reduce of
 * the bucket (one process per GPU on one node; buffers shared through CUDA IPC).  Every rank calls peer_export (128
 * bytes out: IPC handles of its bucket and of its exchange buffer), the ranks all-gather those blobs by any means
 * (torch.distributed in learner.py), then every rank calls peer_import with the world x 128 bytes in rank order.
 * From then on drl_learner_step / _step_async / _apply perform the exchange themselves inside the step's CUDA graph:
 * device-side barrier, each rank sums its slice of every rank's bucket in rank order and delivers it to every rank
 * (bit-identical replicas), barrier, clip + RMSProp.  Do not all-reduce the bucket as well.  All ranks must step in
 * lockstep; a rank that never arrives is reported by drl_learner_wait after a 20 s device-side time-out. */
int drl_learner_peer_export(drl_learner* h, void* handles, int64_t bytes);
int drl_learner_peer_import(drl_learner* h, int32_t rank, int32_t world, const void* all_handles, int64_t bytes);
/* Back to the local update (the caller all-reduces the bucket again); also the clean-up after a failed import. */
int drl_learner_peer_disable(drl_learner* h);
/* The handle's compute stream (cudaStream_t as void*), for ordering external work (NCCL). */
int drl_learner_stream(drl_learner* h, void** stream);

/* Forward only (no update): the learner-side values of build_network
 * (model/impala_actor_critic.py:71-118): policy [B,T,A] and value [B,T], batch-major, for all T
 * rows (first/middle/last are the slices [:, :-2], [:, 1:-1], [:, 2:]).  Host outputs. */
int drl_learner_forward(drl_learner* h, int32_t slot, float* policy, float* value);

/* Parity taps of the last step (agent/impala.py:68-80): vs, clipped_rho, vs_plus_1, pg_advantage,
 * each host float32 [B, T-2] batch-major.  NULL pointers are skipped. */
int drl_learner_taps(drl_learner* h, float* vs, float* clipped_rho, float* vs_plus_1, float* pg_advantage);

/* Debug/parity read of an internal activation by name into host memory (float32, device layout:
 * rows are TIME-MAJOR m = t*B + b).  Names: "a1" [M,20,20,32], "a2" [M,9,9,64], "a3" [M,3136],
 * "emb" [A,256], "h1","c1" [M,256], "logits","policy" [M,A], "value" [M].  n = element count. */
int drl_learner_read_buffer(drl_learner* h, const char* name, float* host_dst, int64_t n);

/* Actor-side shim of Agent.get_policy_and_action (agent/impala.py:118-130): n independent
 * single-step forwards.  state u8 [n,H,W,C]; previous_action i32 [n]; h,c f32 [n,L] ->
 * policy [n,A], h_out, c_out [n,L] (host).  n <= batch*trajectory. */
int drl_learner_act(drl_learner* h, int32_t n, const uint8_t* state, const int32_t* previous_action,
                    const float* h_in, const float* c_in, float* policy, float* h_out, float* c_out);

/* Measurement aid (bench.py roofline): runs ONE real step on a staged slot with a CUDA event recorded
 * on the compute stream before every kernel launch and returns per-launch device times.  names is a
 * '\n'-joined list (names_len bytes available), ms[i] the time from launch i to launch i+1. */
int drl_learner_profile_step(drl_learner* h, int32_t slot, char* names, int64_t names_len, float* ms,
                             int32_t max_kernels, int32_t* count);
/* Test aid: one plain GEMM C[M,N] = A*B on a chosen contraction core (1 = FP32 FFMA, 2 = tcgen05 3xTF32) and
 * operand-major combination, to validate shared-memory layouts / UMMA descriptors in isolation.
 * a_kmajor: A is [M,K] row-major (1) or [K,M] row-major (0); b_kmajor: B is [N,K] (1) or [K,N] (0).
 * C: `splits` slabs of [(M+1), N] floats (split-K partials; row M = column sums of B for N-major B). */
int drl_debug_gemm(int32_t core, int32_t bn, int32_t a_kmajor, int32_t b_kmajor, int32_t M, int32_t N,
                   int32_t K, int32_t splits, const float* A, const float* B, float* C);
/* Test aid: arm (dev_buf: device buffer of >= 8001 uint64, word 0 = entry count, zeroed by the caller) or disarm
 * (NULL) the kernel start-time trace: CTA 0 of every kernel of the step appends {globaltimer ns, grid size << 32 |
 * block size}.  Gives the true timeline of a CUDA-graph replay across both streams (tools/timeline.py). */
int drl_debug_trace(void* dev_buf);
/* Device-time of the last step's compute (CUDA events on the compute stream), milliseconds. */
int drl_learner_last_step_ms(drl_learner* h, float* ms);
/* Number of kernel launches one step issues (for bench.py's gpu_launches claim). */
int drl_learner_launches_per_step(const drl_learner* h, int32_t* n);

/* ------------------------------------------------------------------------------------------
 * Stand-alone V-trace (optimizer/vtrace.py), host-pointer convenience forms + device forms.
 * ------------------------------------------------------------------------------------------ */
/* vtrace.from_importance_weights (optimizer/vtrace.py:71-103): time-major [T,B] float32 inputs,
 * bootstrap_value [B]; outputs vs, clipped_rhos [T,B].  clip_rho_threshold < 0 means None. */
int drl_vtrace_from_importance_weights(const float* log_rhos, const float* discounts,
                                       const float* rewards, const float* values,
                                       const float* bootstrap_value, int32_t T, int32_t B,
                                       float clip_rho_threshold, float* vs, float* clipped_rhos);
int drl_vtrace_from_importance_weights_dev(const float* log_rhos, const float* discounts,
                                           const float* rewards, const float* values,
                                           const float* bootstrap_value, int32_t T, int32_t B,
                                           float clip_rho_threshold, float* vs, float* clipped_rhos,
                                           void* stream);
/* vtrace.from_softmax (optimizer/vtrace.py:29-69): batch-major behavior/target softmax [B,T,A],
 * actions i32 [B,T], discounts/rewards/values/next_values f32 [B,T] -> vs, clipped_rho [B,T]. */
int drl_vtrace_from_softmax(const float* behavior_policy_softmax, const float* target_policy_softmax,
                            const int32_t* actions, const float* discounts, const float* rewards,
                            const float* values, const float* next_values, int32_t B, int32_t T,
                            int32_t A, float clip_rho_threshold, float* vs, float* clipped_rho);
int drl_vtrace_from_softmax_dev(const float* behavior_policy_softmax, const float* target_policy_softmax,
                                const int32_t* actions, const float* discounts, const float* rewards,
                                const float* values, const float* next_values, int32_t B, int32_t T,
                                int32_t A, float clip_rho_threshold, float* vs, float* clipped_rho,
                                void* stream);

/* The three loss sums of optimizer/vtrace.py:105-126 and log_probs_from_softmax_and_actions (:16-27)
 * in one pass over host arrays: softmax [B,T,A], actions i32 [B,T], advantages/vs/value f32 [B,T] ->
 * sums[3] = { -sum log(pi(a)+1e-8)*adv, 0.5*sum (vs-value)^2, sum pi*log(pi) }, log_probs [B,T]
 * (= log pi(a), no epsilon; may be NULL). */
int drl_vtrace_loss_sums(const float* softmax, const int32_t* actions, const float* advantages,
                         const float* vs, const float* value, int32_t B, int32_t T, int32_t A,
                         float* sums, float* log_probs);

/* ------------------------------------------------------------------------------------------
 * Trajectory ring: replaces buffer_queue.FIFOQueue (distributed_queue/buffer_queue.py:418-512).
 * A FIFO of `capacity` trajectories kept in pinned host memory, organised as batch slots of
 * `batch` trajectories in field-major order so that a popped batch is 8 contiguous [B, ...]
 * arrays ready for one async H2D each.  next_state is accepted by the Python shim and dropped
 * (the learner never reads it, train_impala.py:100-108).
 * ------------------------------------------------------------------------------------------ */
typedef struct drl_ring drl_ring;

typedef struct drl_ring_batch {      /* views into the ring's pinned memory, valid until release */
  uint8_t* state;            /* [B,T,H,W,C] */
  float* reward;             /* [B,T]       */
  uint8_t* done;             /* [B,T]       */
  float* behavior_policy;    /* [B,T,A]     */
  int32_t* action;           /* [B,T]       */
  int32_t* previous_action;  /* [B,T]       */
  float* previous_h;         /* [B,T,L]     */
  float* previous_c;         /* [B,T,L]     */
  int32_t slot;              /* batch-slot index to pass to drl_ring_release */
} drl_ring_batch;

/* FIFOQueue.__init__ (buffer_queue.py:419-466).  capacity is rounded up to a multiple of batch
 * (+ one extra batch slot so producers can fill while the consumer holds one).  pinned=1 uses
 * cudaHostAlloc; if that fails (no device) it falls back to page-aligned malloc and *pinned=0. */
int drl_ring_create(int32_t trajectory, int32_t height, int32_t width, int32_t channels,
                    int32_t num_action, int32_t lstm_size, int32_t capacity, int32_t batch,
                    int32_t want_pinned, drl_ring** out);
int drl_ring_destroy(drl_ring* r);
int drl_ring_is_pinned(const drl_ring* r);
/* FIFOQueue.append_to_queue (buffer_queue.py:468-484): copies one trajectory in; blocks while the
 * ring is full (timeout_ms < 0: forever; DRL_ERR_TIMEOUT otherwise). */
int drl_ring_push(drl_ring* r, const uint8_t* state, const float* reward, const uint8_t* done,
                  const float* behavior_policy, const int32_t* action, const int32_t* previous_action,
                  const float* previous_h, const float* previous_c, int32_t timeout_ms);
/* FIFOQueue.sample_batch (buffer_queue.py:486-505): pops the oldest `batch` trajectories (FIFO
 * order) as one batch slot; blocks until a full batch is available. */
int drl_ring_pop_batch(drl_ring* r, drl_ring_batch* out, int32_t timeout_ms);
/* Hands a popped batch slot back to the producers. */
int drl_ring_release(drl_ring* r, int32_t slot);
/* FIFOQueue.get_size (buffer_queue.py:507-509): trajectories enqueued and not yet popped. */
int drl_ring_size(drl_ring* r);

/* ------------------------------------------------------------------------------------------
 * Ape-X DQN learner (SURVEY.md section 8(f) row 2, BASELINE.json config 4): replaces apex.Agent's learner graph
 * (agent/apex.py:12-76) over model/apex_value.py:4-66 (dueling network: q = value stream - "mean" stream, evaluated
 * as main(s, prev_a), main(s', a), target(s', a)), optimizer/dqn.py:3-7 and TF1 Adam.  The three network
 * evaluations run as ONE main-network forward over 2B rows [s ; s'] plus one target-network forward over B rows;
 * only the first B rows are differentiated.
 * ------------------------------------------------------------------------------------------ */
typedef struct drl_apex drl_apex;

#define DRL_APEX_MAIN 0
#define DRL_APEX_TARGET 1

typedef struct drl_apex_config {
  int32_t batch;              /* B transitions per step (config.json:154)                               */
  int32_t height, width, channels; /* 84,84,4 -- only this geometry is supported (config.json:156)      */
  int32_t num_action;         /* A, 2..32 (config.json:157)                                             */
  float discount_factor;      /* agent/apex.py:43                                                       */
  float start_learning_rate;  /* agent/apex.py:71                                                       */
  float end_learning_rate;
  double learning_frame;      /* decay_steps of tf.train.polynomial_decay                               */
  float gradient_clip_norm;   /* agent/apex.py:74                                                       */
  int32_t reward_clipping;    /* DRL_REWARD_ABS_ONE clips to [-1,1]; anything else passes the reward through
                                 (agent/apex.py:38-41)                                                  */
  int32_t device;             /* CUDA device ordinal                                                    */
  int32_t num_slots;          /* device staging slots for stream-overlapped H2D (>=1, default 2)        */
  int32_t use_cuda_graph;     /* 1: capture the whole step into one CUDA graph per slot                 */
  int32_t math_mode;          /* 0 = default (2); 1 = FP32 FFMA; 2 = tcgen05 3xTF32 convolutions        */
} drl_apex_config;

typedef struct drl_apex_out {
  float loss;           /* value_loss = mean(is_weight * (target_value - state_action_value)^2), agent/apex.py:63-65 */
  float learning_rate;  /* agent/apex.py:71 */
  float grad_norm;      /* global norm before clipping (agent/apex.py:74) */
  int64_t step;         /* global_step AFTER this update (agent/apex.py:70,75) */
} drl_apex_out;

/* apex.Agent.__init__ (agent/apex.py:12-76): parameters of 'main' and 'target' (zeros until set), Adam slots m, v
 * (zeros), beta powers (0.9, 0.999), activations, staging slots, streams on cfg->device. */
int drl_apex_create(const drl_apex_config* cfg, drl_apex** out);
int drl_apex_destroy(drl_apex* h);
/* Learnable floats of ONE network (main and target have the same inventory). */
int drl_apex_param_count(const drl_apex* h, int64_t* n);
/* Flat float32 vector in TF layouts / TF variable-creation order of the scope ({model}/main or {model}/target):
 * conv2d x3 (HWIO), dense x2 (action embedding), dense x3 (value stream), dense x3 ("mean" stream); which =
 * DRL_APEX_MAIN / DRL_APEX_TARGET.  Replaces global_variables_initializer / Saver (agent/apex.py:76,84-86). */
int drl_apex_set_params(drl_apex* h, int32_t which, const float* host_flat, int64_t n);
int drl_apex_get_params(drl_apex* h, int32_t which, float* host_flat, int64_t n);
/* Adam slots of the main network, global_step, beta1_power, beta2_power (agent/apex.py:72). */
int drl_apex_set_opt_state(drl_apex* h, const float* host_m, const float* host_v, int64_t n, int64_t step,
                           float beta1_power, float beta2_power);
int drl_apex_get_opt_state(drl_apex* h, float* host_m, float* host_v, int64_t n, int64_t* step,
                           float* beta1_power, float* beta2_power);
/* Gradient of value_loss w.r.t. the main network, before clipping (parity tap of compute_gradients, agent/apex.py:73). */
int drl_apex_get_grads(drl_apex* h, float* host_flat, int64_t n);
/* Agent.target_to_main (agent/apex.py:78-79 -> utils.main_to_target, utils.py:27-32): despite its name it assigns
 * target <- main. */
int drl_apex_target_to_main(drl_apex* h);

/* Feed of Agent.distributed_train (agent/apex.py:135-149): asynchronous H2D into staging slot `slot`.
 * state, next_state u8 [B,H,W,C] (the /255 of :136-137 happens on the device); previous_action, action i32 [B];
 * reward f32 [B]; done u8/bool [B]; is_weight f32 [B] or NULL (= ones: Agent.train, agent/apex.py:156-168). */
int drl_apex_stage(drl_apex* h, int32_t slot, const uint8_t* state, const uint8_t* next_state,
                   const int32_t* previous_action, const int32_t* action, const float* reward,
                   const uint8_t* done, const float* is_weight);
/* sess.run([value_loss, target_value, state_action_value, train_op]) (agent/apex.py:139-149): forward x3, TD target,
 * weighted squared loss, backward through main(s), global-norm clip, Adam, step += 1.  td_error (host, [B], may be
 * NULL) receives |target_value - state_action_value| from BEFORE the update (agent/apex.py:151): the new priorities. */
int drl_apex_step(drl_apex* h, int32_t slot, drl_apex_out* out, float* td_error);
int drl_apex_step_async(drl_apex* h, int32_t slot);
int drl_apex_wait(drl_apex* h, drl_apex_out* out, float* td_error);
/* (new) Data-parallel step in two halves (one process per GPU, each rank feeds its own B transitions): forward + TD +
 * backward into the gradient bucket [padded grads | loss scalars] -> the CALLER all-reduces (SUM) the bucket on the
 * learner's stream (drl_apex_stream) -> clip + Adam on bucket * grad_scale.  value_loss is a batch MEAN
 * (agent/apex.py:65), so grad_scale = 1 / world_size makes the update that of the undivided global batch. */
int drl_apex_forward_backward(drl_apex* h, int32_t slot);
int drl_apex_grad_bucket(drl_apex* h, void** dev_ptr, int64_t* count);
int drl_apex_apply(drl_apex* h, float grad_scale);   /* async; follow with drl_apex_wait */
/* Agent.get_td_error (agent/apex.py:116-133): forward only, n <= batch transitions -> |target - q(s,a)| [n]. */
int drl_apex_td_error(drl_apex* h, int32_t n, const uint8_t* state, const uint8_t* next_state,
                      const int32_t* previous_action, const int32_t* action, const float* reward,
                      const uint8_t* done, float* td_error);
/* Agent.get_policy_and_action without the epsilon-greedy draw (agent/apex.py:88-102): main_q_value [n, A] for
 * n <= 2*batch (state, previous_action) pairs. */
int drl_apex_act(drl_apex* h, int32_t n, const uint8_t* state, const int32_t* previous_action, float* q_value);
/* Parity taps of the most recent step / td_error call over its n rows (agent/apex.py:45-61): main_q_value,
 * next_main_q_value, target_q_value [n, A]; target_value, state_action_value [n].  Any pointer may be NULL. */
int drl_apex_taps(drl_apex* h, float* main_q, float* next_main_q, float* target_q, float* target_value,
                  float* state_action_value);
/* Debug/parity: copy a named device buffer of the MAIN network's last forward to the host.  Names: a1 a2 a3 e1 emb
 * hid1 hid2 (rows = 2n: [s ; s']), da1 da2 da3 (rows = n). */
int drl_apex_read_buffer(drl_apex* h, const char* name, float* host_dst, int64_t n);
/* Per-launch device times of one real step (CUDA events around every launch, serial). */
int drl_apex_profile_step(drl_apex* h, int32_t slot, char* names, int64_t names_len, float* ms, int32_t max_kernels,
                          int32_t* count);
int drl_apex_last_step_ms(drl_apex* h, float* ms);
/* The learner's compute stream (cudaStream_t), for callers that time or order work against it. */
int drl_apex_stream(drl_apex* h, void** stream);
int drl_apex_launches_per_step(const drl_apex* h, int32_t* n);

/* ------------------------------------------------------------------------------------------
 * Prioritized replay index (host): replaces buffer_queue.SumTree / Memory (distributed_queue/buffer_queue.py:326-416)
 * -- float64 sum tree with the reference's arithmetic order (bit-identical totals), priorities (|td| + 0.001)^0.6,
 * stratified sampling, importance weights (n_entries * p / total)^-beta / max, beta 0.4 -> 1 by +0.001 per sample
 * call.  The transitions themselves stay with the caller (the Python shim keeps them, as the reference does); the
 * uniform draws of random.uniform(a, b) are passed in as u01 in [0,1) so that sampling is reproducible.
 * ------------------------------------------------------------------------------------------ */
typedef struct drl_per drl_per;
int drl_per_create(int64_t capacity, drl_per** out);
int drl_per_destroy(drl_per* p);
/* Memory.add (buffer_queue.py:386-388): stores priority (error + e)^a at the write cursor; returns the data index
 * the caller must store the transition at (SumTree.add, :351-359). */
int drl_per_add(drl_per* p, double error, int64_t* data_index);
/* Memory.sample (buffer_queue.py:390-411): n strata; tree_index[i] (SumTree.get's idx), data_index[i],
 * priority[i], is_weight[i]; also advances beta. */
int drl_per_sample(drl_per* p, int32_t n, const double* u01, int64_t* tree_index, int64_t* data_index,
                   double* priority, double* is_weight);
/* Memory.update (buffer_queue.py:413-415): tree_index as returned by drl_per_sample. */
int drl_per_update(drl_per* p, int64_t tree_index, double error);
int drl_per_total(const drl_per* p, double* total);      /* SumTree.total (:348-349) */
int drl_per_size(const drl_per* p, int64_t* n_entries);  /* SumTree.n_entries */
int drl_per_beta(const drl_per* p, double* beta);

/* ------------------------------------------------------------------------------------------
 * (new) Device-resident prioritized replay of an Ape-X learner: buffer_queue.Memory / SumTree together with the
 * transitions themselves (distributed_queue/buffer_queue.py:326-416), kept in the learner's GPU memory.  Storage is
 * field-major (state / next_state [cap, H*W*C] u8, previous_action / action [cap] i32, reward [cap] f32, done [cap]
 * u8); the sum tree is 2*cap - 1 float64 nodes with the leaves last, updated with the reference's arithmetic order
 * (totals bit-identical to drl_per_* for the same leaf values).  Sampling draws its uniforms on the device: Philox4x32-10
 * with key (seed lo, seed hi) and counter (stratum, draw call lo, draw call hi, 0), u = ((x0 << 32 | x1) >> 11) * 2^-53;
 * the draw call counter advances by one per sample.  Priorities are (|td| + 0.001)^0.6 with CUDA's double pow (within
 * a few ulp of glibc's).  The replay runs on the learner's streams and takes its lock; drl_apex_destroy refuses
 * (DRL_ERR_STATE) while a replay of the learner is alive.  The host drl_per_* path is unchanged.
 * ------------------------------------------------------------------------------------------ */
typedef struct drl_apex_replay drl_apex_replay;
/* Memory.__init__ (buffer_queue.py:378-381) on the learner's device, zero-initialised, beta 0.4.  capacity >= 2;
 * DRL_ERR_INVALID for an A3C handle; DRL_ERR_CUDA (with the byte count) when the storage does not fit. */
int drl_apex_replay_create(drl_apex* h, int64_t capacity, uint64_t seed, drl_apex_replay** out);
int drl_apex_replay_destroy(drl_apex_replay* r);
/* learner.get_td_error + Memory.add for n <= batch transitions (train_apex.py:106-122, buffer_queue.py:386-388): the
 * same forward and |td| as drl_apex_td_error, then the rows are copied at the write cursor (wrapping) and their leaves
 * set in call order.  Synchronous: the host buffers are free on return.  Shapes as drl_apex_stage. */
int drl_apex_replay_add(drl_apex_replay* r, int32_t n, const uint8_t* state, const uint8_t* next_state,
                        const int32_t* previous_action, const int32_t* action, const float* reward,
                        const uint8_t* done);
/* Memory.sample -> distributed_train -> Memory.update (train_apex.py:129-155) as ONE enqueue on the learner's compute
 * stream: sample batch strata, gather them into training slot `slot` (float32 importance weights included), the
 * learner step, then the new priorities of the sampled leaves from the step's |td|.  Collect with drl_apex_wait.  The
 * slot is left unstaged (a plain drl_apex_step on it needs a new drl_apex_stage).  DRL_ERR_STATE on an empty replay. */
int drl_apex_replay_step_async(drl_apex_replay* r, int32_t slot);
int drl_apex_replay_step(drl_apex_replay* r, int32_t slot, drl_apex_out* out, float* td_error);
/* Inspection: the most recent sample's [batch] tree indices, data indices, priorities and float64 weights
 * (Memory.sample's idxs / is_weight); any pointer may be NULL. */
int drl_apex_replay_last_sample(drl_apex_replay* r, int64_t* tree_index, int64_t* data_index, double* priority,
                                double* is_weight);
/* Inspection: the (leaf, priority) list of the most recent add or post-step update, in call order (*count entries,
 * at most max_count copied). */
int drl_apex_replay_last_update(drl_apex_replay* r, int64_t* leaf, double* priority, int32_t max_count,
                                int32_t* count);
/* Inspection: SumTree.n_entries / write, SumTree.total (:348-349), Memory.beta and the draw calls so far. */
int drl_apex_replay_info(drl_apex_replay* r, int64_t* n_entries, int64_t* write, double* total, double* beta,
                         int64_t* draws);
/* Inspection: all 2*capacity - 1 tree nodes (count must equal that). */
int drl_apex_replay_read_tree(drl_apex_replay* r, double* host_nodes, int64_t count);

/* ------------------------------------------------------------------------------------------
 * R2D2 learner (SURVEY.md section 8(f) row 3, BASELINE.json config 5): replaces r2d2.Agent's learner graph
 * (agent/r2d2.py:13-95) over model/r2d2_lstm.py:28-116 (conv stack + action embedding + ONE LSTMCell, unrolled seq_len
 * steps per scope from a stored (h, c) with the carried state multiplied by (1 - done) after every step; dense 128;
 * q = value - "mean"), optimizer/burn_in.py:23-32 (value-function rescaling, eps 1e-3), double-Q targets over the
 * post-burn-in window and TF1 Adam(1e-4) without clipping.  Sequences are batch-major [B, S, ...].
 * ------------------------------------------------------------------------------------------ */
typedef struct drl_r2d2 drl_r2d2;

typedef struct drl_r2d2_config {
  int32_t batch;              /* B sequences per step (config.json:94)                                   */
  int32_t seq_len;            /* S (config.json:95); BASELINE config 5 asks 80                           */
  int32_t burn_in;            /* loss window starts here (config.json:96), 0 <= burn_in <= S - 2         */
  int32_t height, width, channels; /* 84, 84, 1 (config.json:91) or 84, 84, 4                            */
  int32_t num_action;         /* A, 2..32                                                                */
  int32_t lstm_size;          /* 64 -- only this size is supported (config.json:93)                      */
  float discount_factor;      /* agent/r2d2.py:62                                                        */
  float learning_rate;        /* 1e-4 (agent/r2d2.py:91)                                                 */
  int32_t device;
  int32_t num_slots;
  int32_t use_cuda_graph;
  int32_t math_mode;          /* 0 = default (2); 1 = FP32 FFMA; 2 = tcgen05 3xTF32 for the large contractions */
} drl_r2d2_config;

typedef struct drl_r2d2_out {
  float loss;        /* value_loss (agent/r2d2.py:90) */
  float grad_norm;   /* global gradient norm (diagnostic; the reference does not clip) */
  int64_t step;      /* updates applied so far */
} drl_r2d2_out;

int drl_r2d2_create(const drl_r2d2_config* cfg, drl_r2d2** out);
int drl_r2d2_destroy(drl_r2d2* h);
int drl_r2d2_param_count(const drl_r2d2* h, int64_t* n);   /* floats of ONE scope */
/* Flat float32 vector of scope `which` (0 = main, 1 = target) in TF layouts / TF variable-creation order: conv2d x3
 * (HWIO), dense x2 (action embedding), rnn/lstm_cell kernel [3136+256+L, 4L] (gate order i,j,f,o) + bias, dense 128,
 * dense A (value), dense 1 (mean). */
int drl_r2d2_set_params(drl_r2d2* h, int32_t which, const float* host_flat, int64_t n);
int drl_r2d2_get_params(drl_r2d2* h, int32_t which, float* host_flat, int64_t n);
int drl_r2d2_set_opt_state(drl_r2d2* h, const float* host_m, const float* host_v, int64_t n, int64_t step,
                           float beta1_power, float beta2_power);
int drl_r2d2_get_opt_state(drl_r2d2* h, float* host_m, float* host_v, int64_t n, int64_t* step,
                           float* beta1_power, float* beta2_power);
int drl_r2d2_get_grads(drl_r2d2* h, float* host_flat, int64_t n);
/* Agent.main_to_target (agent/r2d2.py:164-165, utils.py:27-32): target <- main. */
int drl_r2d2_main_to_target(drl_r2d2* h);
/* Feed of Agent.train (agent/r2d2.py:132-152): state u8 [B,S,H,W,C]; previous_action, action i32 [B,S]; h0, c0 f32
 * [B,L] (the reference feeds np.stack(h)[:, 0] of the stored [B,S,L] states); reward f32 [B,S]; done u8/bool [B,S];
 * weight f32 [B] or NULL (= ones). */
int drl_r2d2_stage(drl_r2d2* h, int32_t slot, const uint8_t* state, const int32_t* previous_action,
                   const int32_t* action, const float* h0, const float* c0, const float* reward, const uint8_t* done,
                   const float* weight);
/* sess.run([value_loss, target_value, state_action_value, train_op]) (agent/r2d2.py:134-152): both unrolls, TD
 * targets, loss, BPTT through all S steps of the main scope, Adam.  td_error (host [B], may be NULL) receives
 * |mean_t(target_value - state_action_value)| per sequence from BEFORE the update (agent/r2d2.py:154-157). */
int drl_r2d2_step(drl_r2d2* h, int32_t slot, drl_r2d2_out* out, float* td_error);
int drl_r2d2_step_async(drl_r2d2* h, int32_t slot);
int drl_r2d2_wait(drl_r2d2* h, drl_r2d2_out* out, float* td_error);
/* (new) Data-parallel halves, as drl_apex_forward_backward / _grad_bucket / _apply (value_loss is a batch mean,
 * agent/r2d2.py:90: grad_scale = 1 / world_size). */
int drl_r2d2_forward_backward(drl_r2d2* h, int32_t slot);
int drl_r2d2_grad_bucket(drl_r2d2* h, void** dev_ptr, int64_t* count);
int drl_r2d2_apply(drl_r2d2* h, float grad_scale);
/* Agent.get_td_error (agent/r2d2.py:97-130) for n <= batch sequences at once: td_error[i] = |mean(target - q)| of
 * sequence i (the reference calls it with one sequence). */
int drl_r2d2_td_error(drl_r2d2* h, int32_t n, const uint8_t* state, const int32_t* previous_action,
                      const int32_t* action, const float* h0, const float* c0, const float* reward,
                      const uint8_t* done, float* td_error);
/* Agent.get_action without the epsilon-greedy draw (agent/r2d2.py:171-191): one network step for n <= batch*seq_len
 * (state, previous_action, h, c) rows -> q_value [n,A], h' [n,L], c' [n,L]. */
int drl_r2d2_act(drl_r2d2* h, int32_t n, const uint8_t* state, const int32_t* previous_action, const float* h_in,
                 const float* c_in, float* q_value, float* h_out, float* c_out);
/* Parity taps of the most recent step / td_error call over its n sequences: main_q, target_q [n,S,A] (agent/r2d2.py:52),
 * target_value, state_action_value [n, S - burn_in - 1] (:81-88).  Any pointer may be NULL. */
int drl_r2d2_taps(drl_r2d2* h, float* main_q, float* target_q, float* target_value, float* state_action_value);
/* Debug/parity: named device buffer of the main scope (time-major rows m = t*n + b): a1 a2 a3 e1 emb q1 hout hin cin
 * gates dz dhout da3. */
int drl_r2d2_read_buffer(drl_r2d2* h, const char* name, float* host_dst, int64_t n);
int drl_r2d2_profile_step(drl_r2d2* h, int32_t slot, char* names, int64_t names_len, float* ms, int32_t max_kernels,
                          int32_t* count);
int drl_r2d2_last_step_ms(drl_r2d2* h, float* ms);
int drl_r2d2_stream(drl_r2d2* h, void** stream);
int drl_r2d2_launches_per_step(const drl_r2d2* h, int32_t* n);

/* ------------------------------------------------------------------------------------------
 * A3C learner: replaces a3c.Agent's learner graph (agent/a3c.py:11-78) over model/actor_critic.py:3-56 (the same body
 * as the Ape-X network: attention_CNN || action embedding -> concat 3392 -> actor [256,256,A + softmax] and critic
 * [256,256,1]) and optimizer/a2c.py:3-26, with TF1 Adam + polynomial decay + global-norm clipping.  network(s, prev_a)
 * and network(s', a) run as ONE forward over 2B rows; next_value is stop_gradient, so only the first B rows are
 * differentiated.  The handle is the Ape-X handle type in A3C mode.
 * ------------------------------------------------------------------------------------------ */
typedef struct drl_apex drl_a3c;

typedef struct drl_a3c_config {
  int32_t batch;              /* transitions per step: trajectory (config.json:36) -- the learner trains on one unroll */
  int32_t height, width, channels; /* 84,84,4                                                           */
  int32_t num_action;
  float discount_factor;      /* agent/a3c.py:45                                                        */
  float start_learning_rate;  /* agent/a3c.py:76                                                        */
  float end_learning_rate;
  double learning_frame;
  float baseline_loss_coef;   /* agent/a3c.py:73                                                        */
  float entropy_coef;
  float gradient_clip_norm;   /* agent/a3c.py:79                                                        */
  int32_t reward_clipping;    /* DRL_REWARD_ABS_ONE / DRL_REWARD_SOFT_ASYMMETRIC (agent/a3c.py:38-43)    */
  int32_t device;
  int32_t num_slots;
  int32_t use_cuda_graph;
  int32_t math_mode;
} drl_a3c_config;

typedef struct drl_a3c_out {
  float pi_loss;        /* -mean(advantage * pi(a))           (optimizer/a2c.py:17-26) */
  float baseline_loss;  /* mean((r + gamma V(s') - V(s))^2)    (optimizer/a2c.py:9-15)  */
  float entropy;        /* -mean(sum_a -pi log pi)             (optimizer/a2c.py:3-7)   */
  float learning_rate;
  float grad_norm;
  int64_t step;
} drl_a3c_out;

int drl_a3c_create(const drl_a3c_config* cfg, drl_a3c** out);
int drl_a3c_destroy(drl_a3c* h);
int drl_a3c_param_count(const drl_a3c* h, int64_t* n);
/* Flat float32 vector, TF variable order of scope {model}/a3c: conv2d x3, dense x2 (embedding), dense x3 (actor),
 * dense x3 (critic). */
int drl_a3c_set_params(drl_a3c* h, const float* host_flat, int64_t n);
int drl_a3c_get_params(drl_a3c* h, float* host_flat, int64_t n);
int drl_a3c_set_opt_state(drl_a3c* h, const float* host_m, const float* host_v, int64_t n, int64_t step,
                          float beta1_power, float beta2_power);
int drl_a3c_get_opt_state(drl_a3c* h, float* host_m, float* host_v, int64_t n, int64_t* step, float* beta1_power,
                          float* beta2_power);
int drl_a3c_get_grads(drl_a3c* h, float* host_flat, int64_t n);
/* Feed of Agent.train (agent/a3c.py:85-103): state, next_state u8 [B,H,W,C]; previous_action, action i32 [B] (the
 * reference feeds `action` as the next step's previous action, :99); reward f32 [B]; done u8/bool [B]. */
int drl_a3c_stage(drl_a3c* h, int32_t slot, const uint8_t* state, const uint8_t* next_state,
                  const int32_t* previous_action, const int32_t* action, const float* reward, const uint8_t* done);
/* sess.run([pi_loss, baseline_loss, entropy, learning_rate, train_op]) (agent/a3c.py:89-103). */
int drl_a3c_step(drl_a3c* h, int32_t slot, drl_a3c_out* out);
int drl_a3c_step_async(drl_a3c* h, int32_t slot);
int drl_a3c_wait(drl_a3c* h, drl_a3c_out* out);
/* (new) Data-parallel halves (all three A2C losses are batch means: grad_scale = 1 / world_size). */
int drl_a3c_forward_backward(drl_a3c* h, int32_t slot);
int drl_a3c_grad_bucket(drl_a3c* h, void** dev_ptr, int64_t* count);
int drl_a3c_apply(drl_a3c* h, float grad_scale);
/* Agent.get_policy_and_action without the sampling (agent/a3c.py:109-119): policy [n,A] and value [n], n <= 2*batch. */
int drl_a3c_act(drl_a3c* h, int32_t n, const uint8_t* state, const int32_t* previous_action, float* policy,
                float* value);
/* Parity taps of the most recent step: policy [B,A], value [B], next_value [B], advantage [B]. */
int drl_a3c_taps(drl_a3c* h, float* policy, float* value, float* next_value, float* advantage);
int drl_a3c_read_buffer(drl_a3c* h, const char* name, float* host_dst, int64_t n);
int drl_a3c_profile_step(drl_a3c* h, int32_t slot, char* names, int64_t names_len, float* ms, int32_t max_kernels,
                         int32_t* count);
int drl_a3c_stream(drl_a3c* h, void** stream);
int drl_a3c_launches_per_step(const drl_a3c* h, int32_t* n);

#ifdef __cplusplus
}
#endif
#endif /* DRL_B200_H_ */
