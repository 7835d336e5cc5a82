// apex.cu -- the Ape-X DQN learner behind drl_apex_* (include/drl_b200.h): replaces apex.Agent's learner graph
// (agent/apex.py:12-76) over the dueling network of model/apex_value.py:4-66, optimizer/dqn.py:3-7 and TF1 Adam.
//
// The reference builds three network copies -- main(s, prev_a), main(s', a), target(s', a) (model/apex_value.py:43-66).
// Here the two main-network evaluations are ONE forward over 2B rows [s ; s'] (the B rows that receive gradient are
// the contiguous prefix, exactly like the B*(T-2) prefix of the IMPALA learner), the target network is one forward
// over the B rows s'.  The attention_CNN and the action embedding are the same layers as IMPALA's, so they run
// through the same gather-GEMM kernels (layer_defs.cuh); the two streams of the dueling head share their input
// concat = [a3 | emb(prev_a)] (K = 3392), so their first layers are one split-K GEMM with N = 2 x 256.
#include "adam_learner.cuh"
#include "replay.cuh"

namespace drl {

// Offsets (in floats) inside the padded flat vectors of ONE network; same conventions as ParamLayout (kernels.h):
// TF variable order, every bias directly behind its kernel and padded to 4 floats.
struct ApexLayout : FlatLayout<22> {
  int A;
  int64_t conv1_w, conv1_b, conv2_w, conv2_b, conv3_w, conv3_b;
  int64_t emb1_w, emb1_b, emb2_w, emb2_b;
  int64_t value1_w, value1_b, value2_w, value2_b, value3_w, value3_b;
  int64_t mean1_w, mean1_b, mean2_w, mean2_b, mean3_w, mean3_b;
  void init(int num_action) {
    A = num_action;
    const int64_t CAT = Geo::FLAT + Geo::EMB;
    place({8 * 8 * 4 * 32, 32, 4 * 4 * 32 * 64, 64, 3 * 3 * 64 * 64, 64,
           (int64_t)A * 256, 256, 256 * 256, 256,
           CAT * 256, 256, 256 * 256, 256, 256 * (int64_t)A, A,
           CAT * 256, 256, 256 * 256, 256, 256, 1},
          {&conv1_w, &conv1_b, &conv2_w, &conv2_b, &conv3_w, &conv3_b, &emb1_w, &emb1_b, &emb2_w, &emb2_b, &value1_w,
           &value1_b, &value2_w, &value2_b, &value3_w, &value3_b, &mean1_w, &mean1_b, &mean2_w, &mean2_b, &mean3_w,
           &mean3_b});
  }
};

struct ApexActs {          // forward activations of one network over up to `cap` rows (caller row order)
  float* a1;               // [M,20,20,32]
  float* a2;               // [M,9,9,64]
  float* a3;               // [M,3136]
  float* e1;               // [A,256]
  float* table;            // [A,256]
  float* zpart;            // [splits][M,512] split-K partial sums of the two first head layers
  float* hid1;             // [2][M,256]  value / mean stream hidden 1
  float* hid2;             // [2][M,256]
  float* vstream;          // [M,A]  value stream output
  float* scratch_sm;       // [M,A]  (softmax of the value stream: by-product of the shared output kernel, unused)
  float* mstream;          // [M]    "mean" stream output
  int cap;
};

struct ApexBwd {           // backward workspace, Mb = B rows
  float *dq, *dmean;       // [Mb,32] each (columns >= A / >= 1 stay zero)
  float *dhid2, *dhid1;    // [2][Mb,256]
  float *da3, *du, *dpre2, *dpre1, *da2, *da1;
  float *wg_part, *wg_part2, *dcol;
};

constexpr int kHeadN = 2 * Geo::HID;             // 512 columns: [value hidden | mean hidden]
constexpr int kCat = Geo::FLAT + Geo::EMB;       // 3392

static SplitPlan plan_head1(int M) { return plan_split(kCat, cdiv(M, CfgMid::BM) * (kHeadN / CfgMid::BN), 16, 1); }

// hid1[z][m][j] = relu(sum_s zpart[s][m][z*256 + j] + b1[z][j])   (first layers of both streams, model/apex_value.py:17-19)
__global__ void __launch_bounds__(256) apex_hid1_kernel(const float* __restrict__ zpart, int nsplit, size_t slab,
                                                         const float* __restrict__ bv, const float* __restrict__ bm,
                                                         float* __restrict__ hid1, int M) {
  pdl_prologue();
  const int m = blockIdx.x, j = threadIdx.x;
#pragma unroll
  for (int z = 0; z < 2; ++z) {
    float acc = 0.f;
    for (int s = 0; s < nsplit; ++s) acc += zpart[(size_t)s * slab + (size_t)m * kHeadN + z * Geo::HID + j];
    acc += (z == 0 ? bv[j] : bm[j]);
    hid1[((size_t)z * M + m) * Geo::HID + j] = fmaxf(acc, 0.f);
  }
}

// ------------------------------------------------------------------------------------------
// TD target, loss and head gradients (agent/apex.py:43-65, optimizer/dqn.py:3-7), one thread per transition b:
//   q_main(b)      = vstream[b] - mstream[b]                         (model/apex_value.py:40)
//   next_action    = argmax_a q_main(n + b)  (first maximum)          rows n.. hold main(s', a)
//   target_value   = q_target(b)[next_action] * gamma * (1 - done) + clip(r)     (stop_gradient)
//   sav            = q_main(b)[action]
//   loss           = mean_b w_b (target_value - sav)^2
//   d loss / d vstream[b][a] = -2 w_b (target - sav) / n for a == action ; d loss / d mstream[b] = the negative of it
// One block: the loss is a fixed-order block reduction (deterministic).
// ------------------------------------------------------------------------------------------
struct TdArgs {
  const float* vstream; const float* mstream;     // main network, 2n rows
  const float* tvstream; const float* tmstream;   // target network, n rows (s')
  const int32_t* action; const float* reward; const uint8_t* done; const float* weight;   // weight may be null (= 1)
  float discount; int clip; int n; int A;
  float* main_q; float* next_main_q; float* target_q;   // [n, A] taps
  float* target_value; float* sav;                      // [n]
  float* td_dev; float* td_host;                        // [n] |target - sav| (device copy, mapped pinned copy or null)
  float* dq; float* dmean;                              // [n, 32] or null (forward-only call)
  float* loss;                                          // [1] or null
};

__global__ void __launch_bounds__(256) apex_td_kernel(TdArgs a) {
  pdl_prologue();
  __shared__ float red[8];
  float part = 0.f;
  for (int b = threadIdx.x; b < a.n; b += blockDim.x) {
    const float mm = a.mstream[b], mn = a.mstream[a.n + b], mt = a.tmstream[b];
    const int act = a.action[b];
    float best = -INFINITY, sav = 0.f;
    int arg = 0;
    for (int k = 0; k < a.A; ++k) {
      const float qm = a.vstream[(size_t)b * a.A + k] - mm;
      const float qn = a.vstream[(size_t)(a.n + b) * a.A + k] - mn;
      const float qt = a.tvstream[(size_t)b * a.A + k] - mt;
      a.main_q[(size_t)b * a.A + k] = qm;
      a.next_main_q[(size_t)b * a.A + k] = qn;
      a.target_q[(size_t)b * a.A + k] = qt;
      if (k == act) sav = qm;
      if (qn > best) { best = qn; arg = k; }          // tf.argmax: first maximal index
    }
    const float nsav = a.tvstream[(size_t)b * a.A + arg] - mt;
    float r = a.reward[b];
    if (a.clip) r = fminf(fmaxf(r, -1.0f), 1.0f);
    const float disc = a.done[b] ? 0.0f : a.discount;
    const float target = nsav * disc + r;
    const float diff = target - sav;
    const float w = a.weight ? a.weight[b] : 1.0f;
    a.target_value[b] = target;
    a.sav[b] = sav;
    const float td = fabsf(diff);
    a.td_dev[b] = td;
    if (a.td_host) a.td_host[b] = td;
    part += diff * diff * w;
    if (a.dq) {
      const float g = -2.0f * w * diff / (float)a.n;
      for (int k = 0; k < a.A; ++k) a.dq[(size_t)b * 32 + k] = (k == act) ? g : 0.f;
      a.dmean[(size_t)b * 32] = -g;
    }
  }
  if (a.loss) {
    part = warp_sum(part);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = part;
    __syncthreads();
    if (threadIdx.x == 0) {
      float s = 0.f;
#pragma unroll
      for (int i = 0; i < 8; ++i) s += red[i];
      *a.loss = s / (float)a.n;
    }
  }
}

// ------------------------------------------------------------------------------------------
// A3C / A2C losses and head gradients (optimizer/a2c.py:3-26, agent/a3c.py:36-73) on the same network body: the actor
// stream ends in a softmax (model/actor_critic.py:33-34), the critic stream is the scalar value.  Rows [0, n) hold
// network(s, prev_a), rows [n, 2n) network(s', a); next_value is stop_gradient in both losses.
//   adv      = clip(r) + gamma (1 - done) V(s') - V(s)                      (stop_gradient in the policy loss)
//   pi_loss  = -mean(adv * pi(a))        (the probability itself, not its log: optimizer/a2c.py:24)
//   baseline = mean(adv^2) ; entropy = -mean(sum_a -pi log pi)              (no epsilon, like the reference)
//   total    = pi_loss + baseline_coef baseline + entropy_coef entropy
// ------------------------------------------------------------------------------------------
struct A3cArgs {
  const float* policy; const float* value;      // [2n, A], [2n]
  const int32_t* action; const float* reward; const uint8_t* done;
  float discount, baseline_coef, entropy_coef; int clip; int n, A;
  float* adv;                                   // [n] tap
  float* dlogits; float* dv;                    // [n, 32]
  float* loss;                                  // [3] pi, baseline, entropy
};
__global__ void __launch_bounds__(256) a3c_loss_kernel(A3cArgs a) {
  pdl_prologue();
  __shared__ float red[3][8];
  float s_pi = 0.f, s_bl = 0.f, s_en = 0.f;
  const float inv_n = 1.0f / (float)a.n;
  for (int b = threadIdx.x; b < a.n; b += blockDim.x) {
    float r = a.reward[b];
    if (a.clip == DRL_REWARD_ABS_ONE) {
      r = fminf(fmaxf(r, -1.0f), 1.0f);
    } else {                                          // soft_asymmetric (agent/a3c.py:41-43)
      const float sq = tanhf(r / 5.0f);
      r = (r < 0.f ? 0.3f * sq : sq) * 5.0f;
    }
    const float disc = a.done[b] ? 0.0f : a.discount;
    const float adv = r + disc * a.value[a.n + b] - a.value[b];
    a.adv[b] = adv;
    const int act = a.action[b];
    const float* p = a.policy + (size_t)b * a.A;
    float ent = 0.f, sdot = 0.f;
    for (int k = 0; k < a.A; ++k) {
      const float pk = p[k], lp = logf(pk);
      ent += pk * lp;
      const float dpk = ((k == act ? -adv : 0.f) + a.entropy_coef * (lp + 1.0f)) * inv_n;     // d total / d pi_k
      sdot += pk * dpk;
    }
    for (int k = 0; k < a.A; ++k) {                   // through the softmax: dlogit_k = pi_k (dpi_k - sum_j pi_j dpi_j)
      const float pk = p[k];
      const float dpk = ((k == act ? -adv : 0.f) + a.entropy_coef * (logf(pk) + 1.0f)) * inv_n;
      a.dlogits[(size_t)b * 32 + k] = pk * (dpk - sdot);
    }
    a.dv[(size_t)b * 32] = a.baseline_coef * (-2.0f * adv) * inv_n;
    s_pi += (act >= 0 && act < a.A) ? adv * p[act] : 0.f;      // tf.one_hot: an out-of-range action selects nothing
    s_bl += adv * adv;
    s_en += ent;
  }
  s_pi = warp_sum(s_pi); s_bl = warp_sum(s_bl); s_en = warp_sum(s_en);
  if ((threadIdx.x & 31) == 0) { red[0][threadIdx.x >> 5] = s_pi; red[1][threadIdx.x >> 5] = s_bl; red[2][threadIdx.x >> 5] = s_en; }
  __syncthreads();
  if (threadIdx.x == 0) {
    float t0 = 0.f, t1 = 0.f, t2 = 0.f;
#pragma unroll
    for (int i = 0; i < 8; ++i) { t0 += red[0][i]; t1 += red[1][i]; t2 += red[2][i]; }
    a.loss[0] = -t0 * inv_n;
    a.loss[1] = t1 * inv_n;
    a.loss[2] = t2 * inv_n;
  }
}

// ------------------------------------------------------------------------------------------
// Forward of the dueling network (model/apex_value.py:22-41) over M rows.  `tgt` only selects the profile names.
// Weight images (tensor-core modes): img[1]/img[2] conv2/conv3 forward, img[5]/img[6] the dCol operands of backward.
// ------------------------------------------------------------------------------------------

static int apex_forward(const Streams& st, const ApexLayout& pl, const float* P, const WeightImages& wi,
                        const uint8_t* frames, const int32_t* pa, const ApexActs& act, int M, int mode,
                        bool retile_fwd, bool retile_bwd, bool tgt, int* launches) {
  const RowMap map{M, 1};          // rows are already in caller order: src(m) == m
  int n = 0;
  cudaStream_t s = st.main;
  const cudaStream_t side = st.par ? st.side : st.main;
  DRL_TRY(fork_to_side(st, 0));
  s = side;
  if (retile_fwd && mode >= 2) {
    prof_mark(s, tgt ? "target_weight_retile" : "weight_retile");
    DRL_TRY((launch_retile_b<64>(s, PlainB{P + pl.conv2_w, 64, 0}, 64, 512, wi.img[1])));
    DRL_TRY((launch_retile_b<64>(s, PlainB{P + pl.conv3_w, 64, 0}, 64, 576, wi.img[2])));
    n += 2;
  }
  if (st.par) DRL_CUDA_CHECK(cudaEventRecord(st.ev[7], side));
  KERNEL(tgt ? "target_emb_fwd" : "emb_fwd",
         emb_forward(s, P + pl.emb1_w, P + pl.emb1_b, P + pl.emb2_w, P + pl.emb2_b, act.e1, act.table, pl.A), 1);
  if (retile_bwd && mode >= 2) {
    prof_mark(s, "weight_retile_bwd");
    DRL_TRY((launch_retile_b<256>(s, PlainBT{P + pl.conv3_w, 64, 0}, 576, 64, wi.img[5])));
    DRL_TRY((launch_retile_b<256>(s, PlainBT{P + pl.conv2_w, 64, 0}, 512, 64, wi.img[6])));
    n += 2;
  }
  s = st.main;
  {  // conv1: u8 frames -> a1 (model/apex_value.py:5)
    Conv1A al{frames, map};
    PlainB bl{P + pl.conv1_w, 32, 0};
    EpConv1 ep{act.a1, 32, P + pl.conv1_b, nullptr};
    GEMM(tgt ? "target_conv1_fwd" : "conv1_fwd", CfgN32, U32, al, bl, ep, M * 400, 32, 256, 1, 256, 0);
  }
  if (st.par) {
    DRL_CUDA_CHECK(cudaStreamWaitEvent(st.main, st.ev[7], 0));
    pdl_break(st.main);
  }
  {  // conv2 (:6)
    Conv2A al{act.a1, map};
    PlainB bl{P + pl.conv2_w, 64, 0};
    PretiledB<PlainB> blp{wi.img[1], 512 / 32};
    EpBiasAct<true, true> ep{act.a2, 64, 0, P + pl.conv2_b, 0, 1.0f};
    GEMM_W(tgt ? "target_conv2_fwd" : "conv2_fwd", CfgBig, U64L, al, bl, blp, ep, M * 81, 64, 512, 1, 512, 0);
  }
  {  // conv3 -> flatten HWC (:7-9)
    Conv3A al{act.a2, map};
    PlainB bl{P + pl.conv3_w, 64, 0};
    PretiledB<PlainB> blp{wi.img[2], 576 / 32};
    EpBiasAct<true, true> ep{act.a3, 64, 0, P + pl.conv3_b, 0, 1.0f};
    GEMM_W(tgt ? "target_conv3_fwd" : "conv3_fwd", CfgBig, U64L, al, bl, blp, ep, M * 49, 64, 576, 1, 576, 0);
  }
  DRL_TRY(join_from_side(st, 1));
  // first layers of both streams: [M, 3392] x [3392, 256 | 256], split-K partial sums, then bias + ReLU (:17-19,28-37)
  const SplitPlan sp = plan_head1(M);
  {
    CatA al{act.a3, act.table, pa};
    DualB bl{P + pl.value1_w, P + pl.mean1_w, Geo::HID, Geo::HID};
    EpRaw<false> ep{act.zpart, kHeadN, (size_t)M * kHeadN, 1.0f, 0, kHeadN};
    GEMM_FFMA(tgt ? "target_heads_l1_fwd" : "heads_l1_fwd", CfgMid, al, bl, ep, M, kHeadN, kCat, sp.splits, sp.kchunk,
              sp.kchunk);
  }
  prof_mark(s, tgt ? "target_heads_l1_bias_relu" : "heads_l1_bias_relu");
  DRL_CUDA_CHECK((launch_k(apex_hid1_kernel, M, 256, 0, s, act.zpart, sp.splits, (size_t)M * kHeadN, P + pl.value1_b,
                           P + pl.mean1_b, act.hid1, M)));
  ++n;
  const size_t head_stride = (size_t)(pl.mean1_w - pl.value1_w);
  {
    PlainA al{act.hid1, Geo::HID, (size_t)M * Geo::HID};
    PlainB bl{P + pl.value2_w, Geo::HID, head_stride};
    EpBiasAct<true, true> ep{act.hid2, Geo::HID, (size_t)M * Geo::HID, P + pl.value2_b, head_stride, 1.0f};
    GEMM_FFMA(tgt ? "target_heads_l2_fwd" : "heads_l2_fwd", CfgSmall, al, bl, ep, M, Geo::HID, Geo::HID, 2, Geo::HID, 0);
  }
  // output layers: value stream [M, A] (final_activation None) and the "mean" stream [M] (:28-39)
  KERNEL(tgt ? "target_heads_out_fwd" : "heads_out_fwd",
         heads_out_forward(s, act.hid2, act.hid2 + (size_t)M * Geo::HID, P + pl.value3_w, P + pl.value3_b,
                           P + pl.mean3_w, P + pl.mean3_b, act.vstream, act.scratch_sm, act.mstream, M, pl.A), 1);
  if (launches) *launches += n;
  return DRL_OK;
}

// Backward through main(s, prev_a): rows [0, Mb) of a forward over M rows.
static int apex_backward(const Streams& st, const ApexLayout& pl, const float* P, const WeightImages& wi, float* G,
                         const uint8_t* frames, const int32_t* pa, const ApexActs& act, const ApexBwd& bw, int M, int Mb,
                         int mode, int* launches) {
  PdlRegionOff pdl_region;
  cudaStream_t s = st.main;
  const cudaStream_t side = st.par ? st.side : st.main;
  const RowMap map{M, 1};
  const size_t head_stride = (size_t)(pl.mean1_w - pl.value1_w);
  const int A = pl.A;
  int n = 0;
  KERNEL("heads_out_bwd",
         heads_out_backward(s, bw.dq, bw.dmean, P + pl.value3_w, P + pl.mean3_w, act.hid2,
                            act.hid2 + (size_t)M * Geo::HID, bw.dhid2, bw.dhid2 + (size_t)Mb * Geo::HID, Mb, A), 1);
  DRL_TRY(fork_to_side(st, 0));
  s = side;
  {  // d value3 [256(+1), A]
    PlainAT al{act.hid2, Geo::HID, 0};
    PlainB bl{bw.dq, 32, 0};
    EpRaw<true> ep{G + pl.value3_w, A, 0, 1.0f, Geo::HID, A};
    GEMM_FFMA("value3_wgrad", CfgSmall, al, bl, ep, Geo::HID, 32, Mb, 1, Mb, 0);
  }
  {  // d mean3 [256(+1), 1]
    PlainAT al{act.hid2 + (size_t)M * Geo::HID, Geo::HID, 0};
    PlainB bl{bw.dmean, 32, 0};
    EpRaw<true> ep{G + pl.mean3_w, 1, 0, 1.0f, Geo::HID, 1};
    GEMM_FFMA("mean3_wgrad", CfgSmall, al, bl, ep, Geo::HID, 32, Mb, 1, Mb, 0);
  }
  {  // d {value2, mean2} = hid1^T dhid2
    PlainAT al{act.hid1, Geo::HID, (size_t)M * Geo::HID};
    PlainB bl{bw.dhid2, Geo::HID, (size_t)Mb * Geo::HID};
    EpRaw<true> ep{G + pl.value2_w, Geo::HID, head_stride, 1.0f, Geo::HID, Geo::HID};
    GEMM_FFMA("heads_l2_wgrad", CfgSmall, al, bl, ep, Geo::HID, Geo::HID, Mb, 2, Mb, 0);
  }
  s = st.main;
  {  // dhid1 = dhid2 W2^T * relu'(hid1)
    PlainA al{bw.dhid2, Geo::HID, (size_t)Mb * Geo::HID};
    PlainBT bl{P + pl.value2_w, Geo::HID, head_stride};
    EpReluMask ep{bw.dhid1, act.hid1, Geo::HID, (size_t)Mb * Geo::HID, (size_t)M * Geo::HID};
    GEMM_FFMA("heads_l2_dgrad", CfgSmall, al, bl, ep, Mb, Geo::HID, Geo::HID, 2, Geo::HID, 0);
  }
  DRL_TRY(fork_to_side(st, 2));
  s = side;
  {  // d {value1, mean1} [3392(+1), 256] = concat^T dhid1 ; bias gradient = column sums
    CatAT al{act.a3, act.table, pa};
    PlainB bl{bw.dhid1, Geo::HID, (size_t)Mb * Geo::HID};
    EpRaw<true> ep{G + pl.value1_w, Geo::HID, head_stride, 1.0f, kCat, Geo::HID};
    GEMM_FFMA("heads_l1_wgrad", CfgBig, al, bl, ep, kCat, Geo::HID, Mb, 2, Mb, 0);
  }
  s = st.main;
  {  // d concat = dhid1_value W1v^T + dhid1_mean W1m^T  -> d a3 (ReLU mask) | d emb rows
    DualA al{bw.dhid1, bw.dhid1 + (size_t)Mb * Geo::HID, Geo::HID, Geo::HID};
    DualBT bl{P + pl.value1_w, P + pl.mean1_w, Geo::HID, Geo::HID};
    EpLstmDx ep{bw.da3, act.a3, bw.du};
    GEMM_FFMA("heads_l1_dgrad", CfgMid, al, bl, ep, Mb, kCat, kHeadN, 1, kHeadN, 0);
  }
  DRL_TRY(fork_to_side(st, 4));
  s = side;
  KERNEL("emb_bwd",
         emb_backward(s, bw.du, pa, act.e1, act.table, P + pl.emb2_w, bw.dpre2, bw.dpre1, G + pl.emb1_w,
                      G + pl.emb1_b, G + pl.emb2_w, G + pl.emb2_b, bw.wg_part, Mb, M, 1, A), 4);
  {
    const SplitPlan sp = plan_conv3_wgrad(Mb, mode);
    const size_t slab = 577 * 64;
    Conv3WA al{act.a2, map};
    PlainB bl{bw.da3, 64, 0};
    EpRaw<true> ep{bw.wg_part, 64, slab, 1.0f, 576, 64};
    GEMM("conv3_wgrad", CfgBig, U64, al, bl, ep, 576, 64, Mb * 49, sp.splits, sp.kchunk, sp.kchunk);
    KERNEL("conv3_wgrad_reduce", splitk_reduce(s, bw.wg_part, slab, sp.splits, G + pl.conv3_w, slab), 1);
  }
  s = st.main;
  if (mode >= 2) {
    PlainA al{bw.da3, 64, 0};
    EpRaw<false> ep{bw.dcol, 576, 0, 1.0f, 0, 576};
    prof_mark(s, "conv3_dgrad");
    PretiledB<PlainBT> blp{wi.img[5], 2};
    DRL_TRY((launch_gemm_umma_persist<PersistOf<U256>::type>(s, al, blp, ep, Mb * 49, 576, 64, 1, 64, 0)));
    prof_mark(s, "conv3_col2im");
    DRL_TRY(col2im_conv3(s, bw.dcol, act.a2, bw.da2, Mb));
    n += 2;
  } else {
    Conv3DA al{bw.da3};
    Conv3DB bl{P + pl.conv3_w};
    Conv3DE ep{bw.da2, act.a2};
    GEMM_FFMA("conv3_dgrad", CfgBig, al, bl, ep, Mb * 81, 64, 576, 1, 576, 0);
  }
  DRL_TRY(fork_to_side(st, 5));
  s = side;
  {
    const SplitPlan sp = plan_conv2_wgrad(Mb, mode);
    const size_t slab = 513 * 64;
    Conv2WA al{act.a1, map};
    PlainB bl{bw.da2, 64, 0};
    EpRaw<true> ep{bw.wg_part, 64, slab, 1.0f, 512, 64};
    GEMM("conv2_wgrad", CfgBig, U64, al, bl, ep, 512, 64, Mb * 81, sp.splits, sp.kchunk, sp.kchunk);
    KERNEL("conv2_wgrad_reduce", splitk_reduce(s, bw.wg_part, slab, sp.splits, G + pl.conv2_w, slab), 1);
  }
  s = st.main;
  if (mode >= 2) {
    PlainA al{bw.da2, 64, 0};
    EpRaw<false> ep{bw.dcol, 512, 0, 1.0f, 0, 512};
    prof_mark(s, "conv2_dgrad");
    PretiledB<PlainBT> blp{wi.img[6], 2};
    DRL_TRY((launch_gemm_umma_persist<PersistOf<U256>::type>(s, al, blp, ep, Mb * 81, 512, 64, 1, 64, 0)));
    prof_mark(s, "conv2_col2im");
    DRL_TRY(col2im_conv2(s, bw.dcol, act.a1, bw.da1, Mb));
    n += 2;
  } else {
    Conv2DA al{bw.da2};
    Conv2DB bl{P + pl.conv2_w};
    Conv2DE ep{bw.da1, act.a1};
    GEMM_FFMA("conv2_dgrad", CfgN32, al, bl, ep, Mb * 100, 32, 256, 4, 256, 0);
  }
  {
    const SplitPlan sp = plan_conv1_wgrad(Mb, mode);
    const size_t slab = 257 * 32;
    Conv1WA al{frames, map};
    PlainB bl{bw.da1, 32, 0};
    EpRaw<true> ep{bw.wg_part2, 32, slab, 1.0f / 255.0f, 256, 32};
    GEMM("conv1_wgrad", CfgWg1, U32, al, bl, ep, 256, 32, Mb * 400, sp.splits, sp.kchunk, sp.kchunk);
    KERNEL("conv1_wgrad_reduce", splitk_reduce(s, bw.wg_part2, slab, sp.splits, G + pl.conv1_w, slab), 1);
  }
  DRL_TRY(join_from_side(st, 6));
  if (launches) *launches += n;
  return DRL_OK;
}

struct ApexSlot {
  uint8_t* frames = nullptr;   // [2B][84,84,4]: state rows, then next_state rows
  int32_t* pa2 = nullptr;      // [2B]: previous_action, then action (the embedding input of the rows s')
  float* reward = nullptr;     // [B]
  uint8_t* done = nullptr;     // [B]
  float* weight = nullptr;     // [B]
};

}  // namespace drl

using namespace drl;

struct drl_apex : AdamLearner {
  drl_apex_config cfg{};
  int A = 0;
  ApexLayout pl{};
  ApexActs act{}, tact{};
  ApexBwd bwd{};
  float *main_q = nullptr, *next_main_q = nullptr, *target_q = nullptr, *target_value = nullptr, *sav = nullptr,
        *td_dev = nullptr;
  // A3C runs on the same body (drl_a3c_*): no target scope, the loss kernel above, three loss scalars
  int algo = 0;                // 0 = Ape-X DQN, 1 = A3C
  float a3c_baseline_coef = 0.f, a3c_entropy_coef = 0.f;
  int a3c_clip = 0;
  float* adv = nullptr;        // [B] advantage tap
  std::vector<ApexSlot> slots; // payloads of AdamLearner::sync
  int replays = 0;             // device replays attached to this handle (replay.cu)
};

namespace {

int alloc_acts(drl_apex* h, ApexActs& a, int cap) {
  const size_t M = cap, A = h->A;
  a.cap = cap;
  DRL_TRY(dev_alloc(h, &a.a1, M * 400 * 32));
  DRL_TRY(dev_alloc(h, &a.a2, M * 81 * 64));
  DRL_TRY(dev_alloc(h, &a.a3, M * Geo::FLAT));
  DRL_TRY(dev_alloc(h, &a.e1, A * Geo::EMB));
  DRL_TRY(dev_alloc(h, &a.table, A * Geo::EMB));
  size_t zmax = 0;
  for (int m = 1; m <= cap; ++m) zmax = std::max(zmax, (size_t)plan_head1(m).splits * m * kHeadN);
  DRL_TRY(dev_alloc(h, &a.zpart, zmax));
  DRL_TRY(dev_alloc(h, &a.hid1, 2 * M * Geo::HID));
  DRL_TRY(dev_alloc(h, &a.hid2, 2 * M * Geo::HID));
  DRL_TRY(dev_alloc(h, &a.vstream, M * A));
  DRL_TRY(dev_alloc(h, &a.scratch_sm, M * A));
  DRL_TRY(dev_alloc(h, &a.mstream, M));
  return DRL_OK;
}

// forward passes + TD kernel over n transitions held by slot `sl`; train = also head gradients and the loss
int enqueue_forward_td(drl_apex* h, const ApexSlot& sl, int n, bool train, float* td_host, int* launches) {
  pdl_break(h->compute);
  pdl_break(h->side);
  const Streams st = streams_of(h), tst = target_streams_of(h);
  if (h->algo == 1) {      // A3C: one scope; rows [0, n) = network(s, prev_a), rows [n, 2n) = network(s', a)
    DRL_TRY(apex_forward(st, h->pl, h->params, h->wi, sl.frames, sl.pa2, h->act, 2 * n, h->mode, h->main_images_stale,
                         h->main_images_stale, false, launches));
    h->main_images_stale = false;
    A3cArgs a{};
    a.policy = h->act.scratch_sm; a.value = h->act.mstream;
    a.action = sl.pa2 + n; a.reward = sl.reward; a.done = sl.done;
    a.discount = h->cfg.discount_factor; a.baseline_coef = h->a3c_baseline_coef; a.entropy_coef = h->a3c_entropy_coef;
    a.clip = h->a3c_clip; a.n = n; a.A = h->A;
    a.adv = h->adv; a.dlogits = h->bwd.dq; a.dv = h->bwd.dmean; a.loss = h->loss;
    prof_mark(h->compute, "a2c_losses");
    DRL_CUDA_CHECK((launch_k(a3c_loss_kernel, 1, 256, 0, h->compute, a)));
    if (launches) *launches += 1;
    return DRL_OK;
  }
  DRL_TRY(fork_target(h));
  DRL_TRY(apex_forward(tst, h->pl, h->target, h->twi, sl.frames + (size_t)n * Geo::FRAME, sl.pa2 + n, h->tact, n, h->mode,
                       h->target_images_stale, false, true, launches));
  h->target_images_stale = false;
  DRL_TRY(target_done(h));
  // rows [0, n) = s with previous_action, rows [n, 2n) = s' with action: one main-network forward covers both
  DRL_TRY(apex_forward(st, h->pl, h->params, h->wi, sl.frames, sl.pa2, h->act, 2 * n, h->mode, h->main_images_stale,
                       h->main_images_stale, false, launches));
  h->main_images_stale = false;
  DRL_TRY(join_target(h));
  TdArgs a{};
  a.vstream = h->act.vstream; a.mstream = h->act.mstream;
  a.tvstream = h->tact.vstream; a.tmstream = h->tact.mstream;
  a.action = sl.pa2 + n; a.reward = sl.reward; a.done = sl.done; a.weight = sl.weight;
  a.discount = h->cfg.discount_factor; a.clip = (h->cfg.reward_clipping == DRL_REWARD_ABS_ONE) ? 1 : 0;
  a.n = n; a.A = h->A;
  a.main_q = h->main_q; a.next_main_q = h->next_main_q; a.target_q = h->target_q;
  a.target_value = h->target_value; a.sav = h->sav; a.td_dev = h->td_dev; a.td_host = td_host;
  a.dq = train ? h->bwd.dq : nullptr; a.dmean = train ? h->bwd.dmean : nullptr;
  a.loss = train ? h->loss : nullptr;
  prof_mark(h->compute, "td_target_loss");
  DRL_CUDA_CHECK((launch_k(apex_td_kernel, 1, 256, 0, h->compute, a)));
  if (launches) *launches += 1;
  return DRL_OK;
}

// the step's forward passes, loss and backward pass (FwdBwd of the shell, adam_learner.cuh)
int forward_backward(drl_apex* h, int slot, int* launches) {
  const ApexSlot& sl = h->slots[slot];
  DRL_TRY(enqueue_forward_td(h, sl, h->B, true, h->d_td + (size_t)slot * h->B, launches));
  return apex_backward(streams_of(h), h->pl, h->params, h->wi, h->grads, sl.frames, sl.pa2, h->act, h->bwd, 2 * h->B,
                       h->B, h->mode, launches);
}

int stage_into(drl_apex* h, ApexSlot& s, cudaStream_t stream, int n, int row2, const uint8_t* state,
               const uint8_t* next_state, const int32_t* previous_action, const int32_t* action, const float* reward,
               const uint8_t* done, const float* is_weight) {
  auto cp = [&](void* dst, const void* src, size_t bytes) -> cudaError_t {
    return cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, stream);
  };
  DRL_CUDA_CHECK(cp(s.frames, state, (size_t)n * Geo::FRAME));
  if (next_state) DRL_CUDA_CHECK(cp(s.frames + (size_t)row2 * Geo::FRAME, next_state, (size_t)n * Geo::FRAME));
  DRL_CUDA_CHECK(cp(s.pa2, previous_action, (size_t)n * 4));
  if (action) DRL_CUDA_CHECK(cp(s.pa2 + row2, action, (size_t)n * 4));
  if (reward) DRL_CUDA_CHECK(cp(s.reward, reward, (size_t)n * 4));
  if (done) DRL_CUDA_CHECK(cp(s.done, done, (size_t)n));
  // no weights = unit weights (Agent.train, agent/apex.py:167): the slot always holds a weight vector, so a captured
  // graph never depends on which entry point fed it
  if (reward) DRL_CUDA_CHECK(cp(s.weight, is_weight ? is_weight : h->h_ones, (size_t)n * 4));
  return DRL_OK;
}

}  // namespace

// ---- the device replay's view of the handle (replay.cuh) -------------------------------------------------------
namespace drl {

int apex_replay_link(drl_apex* h, ApexReplayLink* out) {
  out->mu = &h->mu;
  out->device = h->cfg.device;
  out->B = h->B;
  out->algo = h->algo;
  out->compute = h->compute;
  out->td_dev = h->td_dev;
  return DRL_OK;
}

void apex_replay_attach(drl_apex* h, int delta) {
  std::lock_guard<std::recursive_mutex> lock(h->mu);
  h->replays += delta;
}

int apex_enqueue_td_error(drl_apex* h, int n, const uint8_t* state, const uint8_t* next_state,
                          const int32_t* previous_action, const int32_t* action, const float* reward,
                          const uint8_t* done, ApexRecordView* scratch) {
  ApexSlot& s = h->slots[h->cfg.num_slots];      // scratch slot
  DRL_CUDA_CHECK(cudaStreamSynchronize(h->compute));
  // rows [0, n) = s, rows [n, 2n) = s' (packed, so that one main-network forward covers both)
  DRL_TRY(stage_into(h, s, h->compute, n, n, state, next_state, previous_action, action, reward, done, nullptr));
  pdl_break(h->compute);
  const Streams st = streams_of(h);
  DRL_TRY(apex_forward(st, h->pl, h->params, h->wi, s.frames, s.pa2, h->act, 2 * n, h->mode, h->main_images_stale,
                       h->main_images_stale, false, nullptr));
  h->main_images_stale = false;
  DRL_TRY(apex_forward(st, h->pl, h->target, h->twi, s.frames + (size_t)n * Geo::FRAME, s.pa2 + n, h->tact, n, h->mode,
                       h->target_images_stale, false, true, nullptr));
  h->target_images_stale = false;
  TdArgs a{};
  a.vstream = h->act.vstream; a.mstream = h->act.mstream;
  a.tvstream = h->tact.vstream; a.tmstream = h->tact.mstream;
  a.action = s.pa2 + n; a.reward = s.reward; a.done = s.done; a.weight = nullptr;
  a.discount = h->cfg.discount_factor; a.clip = (h->cfg.reward_clipping == DRL_REWARD_ABS_ONE) ? 1 : 0;
  a.n = n; a.A = h->A;
  a.main_q = h->main_q; a.next_main_q = h->next_main_q; a.target_q = h->target_q;
  a.target_value = h->target_value; a.sav = h->sav; a.td_dev = h->td_dev; a.td_host = nullptr;
  DRL_CUDA_CHECK((launch_k(apex_td_kernel, 1, 256, 0, h->compute, a)));
  pdl_break(h->compute);
  h->last_rows = n;
  *scratch = ApexRecordView{s.frames, s.pa2, s.reward, s.done, s.weight, n};
  return DRL_OK;
}

int apex_replay_step(drl_apex* h, int slot, std::vector<cudaGraphExec_t>& graphs, const ApexSlotWork& fill,
                     const ApexSlotWork& after) {
  DRL_TRY(check_slot(h, slot));
  const ApexSlot& sl = h->slots[slot];
  const ApexRecordView v{sl.frames, sl.pa2, sl.reward, sl.done, sl.weight, h->B};
  return run_filled_step(h, slot, forward_backward, graphs, [&] { return fill(h->compute, v); },
                         [&] { return after(h->compute, v); });
}

}  // namespace drl

extern "C" {

int drl_apex_create(const drl_apex_config* cfg, drl_apex** out) {
  if (!cfg || !out) { set_error("null argument"); return DRL_ERR_INVALID; }
  *out = nullptr;
  if (cfg->height != Geo::IH || cfg->width != Geo::IW || cfg->channels != Geo::IC) {
    set_error("only the reference input geometry 84x84x4 is supported (got %dx%dx%d)", cfg->height, cfg->width, cfg->channels);
    return DRL_ERR_INVALID;
  }
  if (cfg->num_action < 2 || cfg->num_action > 32) { set_error("num_action must be in [2,32]"); return DRL_ERR_INVALID; }
  if (cfg->batch < 1) { set_error("batch must be >= 1"); return DRL_ERR_INVALID; }
  if (cfg->math_mode < 0 || cfg->math_mode > 2) { set_error("math_mode must be 0 (default), 1 (FP32 FFMA) or 2 (tcgen05 3xTF32)"); return DRL_ERR_INVALID; }
  if (drl_device_count() <= cfg->device) { set_error("CUDA device %d not available (no CPU fallback)", cfg->device); return DRL_ERR_CUDA; }
  drl_apex* h = new drl_apex();
  h->cfg = *cfg;
  h->mode = (cfg->math_mode == 0) ? DRL_DEFAULT_MATH_MODE : cfg->math_mode;
  if (h->cfg.num_slots < 1) h->cfg.num_slots = 2;
  h->B = cfg->batch; h->A = cfg->num_action;
  h->pl.init(h->A);
  int rc = [&]() -> int {
    const size_t B = h->B, A = h->A;
    DRL_TRY(create_shell(h, B, AdamSchedule{cfg->start_learning_rate, cfg->end_learning_rate, cfg->learning_frame,
                                            cfg->gradient_clip_norm}));
    DRL_TRY(alloc_acts(h, h->act, 2 * h->B));
    DRL_TRY(alloc_acts(h, h->tact, h->B));
    ApexBwd& b = h->bwd;
    DRL_TRY(dev_alloc(h, &b.dq, B * 32));
    DRL_TRY(dev_alloc(h, &b.dmean, B * 32));
    DRL_TRY(dev_alloc(h, &b.dhid2, 2 * B * Geo::HID));
    DRL_TRY(dev_alloc(h, &b.dhid1, 2 * B * Geo::HID));
    DRL_TRY(dev_alloc(h, &b.da3, B * Geo::FLAT));
    DRL_TRY(dev_alloc(h, &b.du, B * Geo::EMB));
    DRL_TRY(dev_alloc(h, &b.dpre2, A * Geo::EMB));
    DRL_TRY(dev_alloc(h, &b.dpre1, A * Geo::EMB));
    DRL_TRY(dev_alloc(h, &b.da2, B * 81 * 64));
    DRL_TRY(dev_alloc(h, &b.da1, B * 400 * 32));
    const size_t wg = wgrad_partial_floats(h->B, 3);     // Mb = B * (3 - 2)
    DRL_TRY(dev_alloc(h, &b.wg_part, wg));
    DRL_TRY(dev_alloc(h, &b.wg_part2, wg));
    DRL_TRY(dev_alloc(h, &b.dcol, B * 81 * 512));
    DRL_TRY(dev_alloc(h, &h->main_q, B * A));
    DRL_TRY(dev_alloc(h, &h->next_main_q, B * A));
    DRL_TRY(dev_alloc(h, &h->target_q, B * A));
    DRL_TRY(dev_alloc(h, &h->target_value, B));
    DRL_TRY(dev_alloc(h, &h->sav, B));
    DRL_TRY(dev_alloc(h, &h->td_dev, B));
    DRL_TRY(dev_alloc(h, &h->adv, B));
    h->slots.resize(h->sync.size());
    for (ApexSlot& s : h->slots) {
      size_t off = 0;
      const size_t o_fr = off; off = align_up(off + 2 * B * Geo::FRAME, 256);
      const size_t o_pa = off; off = align_up(off + 2 * B * 4, 256);
      const size_t o_rw = off; off = align_up(off + B * 4, 256);
      const size_t o_dn = off; off = align_up(off + B, 256);
      const size_t o_wt = off; off = align_up(off + B * 4, 256);
      uint8_t* base = nullptr;
      DRL_TRY(dev_alloc(h, &base, off));
      s.frames = base + o_fr;
      s.pa2 = reinterpret_cast<int32_t*>(base + o_pa);
      s.reward = reinterpret_cast<float*>(base + o_rw);
      s.done = base + o_dn;
      s.weight = reinterpret_cast<float*>(base + o_wt);
    }
    DRL_CUDA_CHECK(cudaDeviceSynchronize());
    return DRL_OK;
  }();
  return finish_create(h, rc, out);
}

int drl_apex_destroy(drl_apex* h) {
  if (h && h->replays > 0) {
    set_error("destroy: %d device replay(s) still use this learner; destroy them first", h->replays);
    return DRL_ERR_STATE;
  }
  return destroy_shell(h);
}

int drl_apex_param_count(const drl_apex* h, int64_t* n) {
  DRL_ENTER(h);
  if (!n) { set_error("null argument"); return DRL_ERR_INVALID; }
  *n = h->pl.packed_total;
  return DRL_OK;
}
int drl_apex_set_params(drl_apex* h, int32_t which, const float* host_flat, int64_t n) {
  DRL_ENTER(h);
  return set_params(h, which, host_flat, n);
}
int drl_apex_get_params(drl_apex* h, int32_t which, float* host_flat, int64_t n) {
  DRL_ENTER(h);
  return get_params(h, which, host_flat, n);
}
int drl_apex_set_opt_state(drl_apex* h, const float* host_m, const float* host_v, int64_t n, int64_t step,
                           float beta1_power, float beta2_power) {
  DRL_ENTER(h);
  return set_opt_state(h, host_m, host_v, n, step, beta1_power, beta2_power);
}
int drl_apex_get_opt_state(drl_apex* h, float* host_m, float* host_v, int64_t n, int64_t* step, float* beta1_power,
                           float* beta2_power) {
  DRL_ENTER(h);
  return get_opt_state(h, host_m, host_v, n, step, beta1_power, beta2_power);
}
int drl_apex_get_grads(drl_apex* h, float* host_flat, int64_t n) {
  DRL_ENTER(h);
  return get_grads(h, host_flat, n);
}
int drl_apex_target_to_main(drl_apex* h) {
  DRL_ENTER(h);
  return copy_main_to_target(h);
}

int drl_apex_stage(drl_apex* h, int32_t slot, const uint8_t* state, const uint8_t* next_state,
                   const int32_t* previous_action, const int32_t* action, const float* reward, const uint8_t* done,
                   const float* is_weight) {
  DRL_ENTER(h);
  if (!state || !next_state || !previous_action || !action || !reward || !done) { set_error("stage: null input pointer"); return DRL_ERR_INVALID; }
  return stage_slot(h, slot, [&](cudaStream_t s) {
    return stage_into(h, h->slots[slot], s, h->B, h->B, state, next_state, previous_action, action, reward, done,
                      is_weight);
  });
}

int drl_apex_step_async(drl_apex* h, int32_t slot) {
  DRL_ENTER(h);
  return run_step(h, slot, forward_backward);
}
int drl_apex_forward_backward(drl_apex* h, int32_t slot) {
  DRL_ENTER(h);
  return run_forward_backward(h, slot, forward_backward);
}
int drl_apex_grad_bucket(drl_apex* h, void** dev_ptr, int64_t* count) {
  DRL_ENTER(h);
  return grad_bucket(h, dev_ptr, count);
}
int drl_apex_apply(drl_apex* h, float grad_scale) {
  DRL_ENTER(h);
  return run_apply(h, grad_scale);
}

int drl_apex_wait(drl_apex* h, drl_apex_out* out, float* td_error) {
  DRL_ENTER(h);
  const float* r = nullptr;
  DRL_TRY(wait_step(h, td_error, &r));
  if (out) {
    out->loss = r[0];
    out->learning_rate = r[1];
    out->grad_norm = r[2];
    out->step = result_row_step(r);
  }
  return DRL_OK;
}

int drl_apex_step(drl_apex* h, int32_t slot, drl_apex_out* out, float* td_error) {
  DRL_TRY(drl_apex_step_async(h, slot));
  return drl_apex_wait(h, out, td_error);
}

int drl_apex_td_error(drl_apex* h, int32_t n, const uint8_t* state, const uint8_t* next_state,
                      const int32_t* previous_action, const int32_t* action, const float* reward, const uint8_t* done,
                      float* td_error) {
  DRL_ENTER(h);
  if (n < 1 || n > h->B) { set_error("td_error: n must be in [1, %d]", h->B); return DRL_ERR_INVALID; }
  if (!state || !next_state || !previous_action || !action || !reward || !done || !td_error) { set_error("td_error: null pointer"); return DRL_ERR_INVALID; }
  ApexRecordView scratch{};
  DRL_TRY(apex_enqueue_td_error(h, n, state, next_state, previous_action, action, reward, done, &scratch));
  DRL_CUDA_CHECK(cudaMemcpyAsync(td_error, h->td_dev, (size_t)n * 4, cudaMemcpyDeviceToHost, h->compute));
  DRL_CUDA_CHECK(cudaStreamSynchronize(h->compute));
  return DRL_OK;
}

int drl_apex_act(drl_apex* h, int32_t n, const uint8_t* state, const int32_t* previous_action, float* q_value) {
  DRL_ENTER(h);
  if (n < 1 || n > 2 * h->B) { set_error("act: n must be in [1, %d]", 2 * h->B); return DRL_ERR_INVALID; }
  if (!state || !previous_action || !q_value) { set_error("act: null pointer"); return DRL_ERR_INVALID; }
  ApexSlot& s = h->slots[h->cfg.num_slots];
  DRL_CUDA_CHECK(cudaStreamSynchronize(h->compute));
  DRL_TRY(stage_into(h, s, h->compute, n, n, state, nullptr, previous_action, nullptr, nullptr, nullptr, nullptr));
  pdl_break(h->compute);
  DRL_TRY(apex_forward(streams_of(h), h->pl, h->params, h->wi, s.frames, s.pa2, h->act, n, h->mode, h->main_images_stale,
                       h->main_images_stale, false, nullptr));
  h->main_images_stale = false;
  const int A = h->A;
  std::vector<float> v((size_t)n * A), m((size_t)n);
  DRL_CUDA_CHECK(cudaMemcpyAsync(v.data(), h->act.vstream, v.size() * 4, cudaMemcpyDeviceToHost, h->compute));
  DRL_CUDA_CHECK(cudaMemcpyAsync(m.data(), h->act.mstream, m.size() * 4, cudaMemcpyDeviceToHost, h->compute));
  DRL_CUDA_CHECK(cudaStreamSynchronize(h->compute));
  for (int i = 0; i < n; ++i)
    for (int k = 0; k < A; ++k) q_value[(size_t)i * A + k] = v[(size_t)i * A + k] - m[i];   // model/apex_value.py:40
  h->last_rows = 0;
  return DRL_OK;
}

int drl_apex_taps(drl_apex* h, float* main_q, float* next_main_q, float* target_q, float* target_value,
                  float* state_action_value) {
  DRL_ENTER(h);
  if (h->last_rows < 1) { set_error("taps: no step or td_error call has run"); return DRL_ERR_STATE; }
  DRL_CUDA_CHECK(cudaStreamSynchronize(h->compute));
  const size_t n = h->last_rows, A = h->A;
  if (main_q) DRL_CUDA_CHECK(cudaMemcpy(main_q, h->main_q, n * A * 4, cudaMemcpyDeviceToHost));
  if (next_main_q) DRL_CUDA_CHECK(cudaMemcpy(next_main_q, h->next_main_q, n * A * 4, cudaMemcpyDeviceToHost));
  if (target_q) DRL_CUDA_CHECK(cudaMemcpy(target_q, h->target_q, n * A * 4, cudaMemcpyDeviceToHost));
  if (target_value) DRL_CUDA_CHECK(cudaMemcpy(target_value, h->target_value, n * 4, cudaMemcpyDeviceToHost));
  if (state_action_value) DRL_CUDA_CHECK(cudaMemcpy(state_action_value, h->sav, n * 4, cudaMemcpyDeviceToHost));
  return DRL_OK;
}

int drl_apex_read_buffer(drl_apex* h, const char* name, float* host_dst, int64_t n) {
  DRL_ENTER(h);
  if (!name || !host_dst) { set_error("null argument"); return DRL_ERR_INVALID; }
  if (h->last_rows < 1) { set_error("read_buffer: no step or td_error call has run"); return DRL_ERR_STATE; }
  const size_t Mb = h->last_rows, M = 2 * Mb, A = h->A;
  const NamedBuffer tab[] = {
      {"a1", h->act.a1, M * 400 * 32}, {"a2", h->act.a2, M * 81 * 64}, {"a3", h->act.a3, M * Geo::FLAT},
      {"emb", h->act.table, A * Geo::EMB}, {"e1", h->act.e1, A * Geo::EMB},
      {"hid1", h->act.hid1, 2 * M * Geo::HID}, {"hid2", h->act.hid2, 2 * M * Geo::HID},
      {"da3", h->bwd.da3, Mb * Geo::FLAT}, {"da2", h->bwd.da2, Mb * 81 * 64}, {"da1", h->bwd.da1, Mb * 400 * 32}};
  return read_named_buffer(h->compute, tab, sizeof(tab) / sizeof(tab[0]), name, host_dst, n);
}

int drl_apex_profile_step(drl_apex* h, int32_t slot, char* names, int64_t names_len, float* ms, int32_t max_kernels,
                          int32_t* count) {
  DRL_ENTER(h);
  return profile_step(h, slot, forward_backward, names, names_len, ms, max_kernels, count);
}

int drl_apex_last_step_ms(drl_apex* h, float* ms) {
  DRL_ENTER(h);
  return last_step_ms(h, ms);
}

int drl_apex_stream(drl_apex* h, void** stream) {
  DRL_ENTER(h);
  if (!stream) { set_error("null argument"); return DRL_ERR_INVALID; }
  *stream = h->compute;
  return DRL_OK;
}

int drl_apex_launches_per_step(const drl_apex* h, int32_t* n) {
  DRL_ENTER(h);
  if (!n) { set_error("null argument"); return DRL_ERR_INVALID; }
  *n = h->launches;     // valid after the first step
  return DRL_OK;
}

// ---- A3C learner: the same handle type with algo = 1 (include/drl_b200.h) ---------------------------------------
int drl_a3c_create(const drl_a3c_config* cfg, drl_a3c** out) {
  if (!cfg || !out) { set_error("null argument"); return DRL_ERR_INVALID; }
  *out = nullptr;
  if (cfg->reward_clipping != DRL_REWARD_ABS_ONE && cfg->reward_clipping != DRL_REWARD_SOFT_ASYMMETRIC) {
    set_error("reward_clipping must be DRL_REWARD_ABS_ONE or DRL_REWARD_SOFT_ASYMMETRIC");
    return DRL_ERR_INVALID;
  }
  drl_apex_config c{};
  c.batch = cfg->batch; c.height = cfg->height; c.width = cfg->width; c.channels = cfg->channels;
  c.num_action = cfg->num_action; c.discount_factor = cfg->discount_factor;
  c.start_learning_rate = cfg->start_learning_rate; c.end_learning_rate = cfg->end_learning_rate;
  c.learning_frame = cfg->learning_frame; c.gradient_clip_norm = cfg->gradient_clip_norm;
  c.reward_clipping = cfg->reward_clipping; c.device = cfg->device; c.num_slots = cfg->num_slots;
  c.use_cuda_graph = cfg->use_cuda_graph; c.math_mode = cfg->math_mode;
  drl_apex* h = nullptr;
  DRL_TRY(drl_apex_create(&c, &h));
  h->algo = 1;
  h->a3c_baseline_coef = cfg->baseline_loss_coef;
  h->a3c_entropy_coef = cfg->entropy_coef;
  h->a3c_clip = cfg->reward_clipping;
  *out = h;
  return DRL_OK;
}
int drl_a3c_destroy(drl_a3c* h) { return drl_apex_destroy(h); }
int drl_a3c_param_count(const drl_a3c* h, int64_t* n) { return drl_apex_param_count(h, n); }
int drl_a3c_set_params(drl_a3c* h, const float* host_flat, int64_t n) { return drl_apex_set_params(h, DRL_APEX_MAIN, host_flat, n); }
int drl_a3c_get_params(drl_a3c* h, float* host_flat, int64_t n) { return drl_apex_get_params(h, DRL_APEX_MAIN, host_flat, n); }
int drl_a3c_set_opt_state(drl_a3c* h, const float* m, const float* v, int64_t n, int64_t step, float b1p, float b2p) {
  return drl_apex_set_opt_state(h, m, v, n, step, b1p, b2p);
}
int drl_a3c_get_opt_state(drl_a3c* h, float* m, float* v, int64_t n, int64_t* step, float* b1p, float* b2p) {
  return drl_apex_get_opt_state(h, m, v, n, step, b1p, b2p);
}
int drl_a3c_get_grads(drl_a3c* h, float* host_flat, int64_t n) { return drl_apex_get_grads(h, host_flat, n); }
int drl_a3c_stage(drl_a3c* h, int32_t slot, const uint8_t* state, const uint8_t* next_state, const int32_t* previous_action,
                  const int32_t* action, const float* reward, const uint8_t* done) {
  return drl_apex_stage(h, slot, state, next_state, previous_action, action, reward, done, nullptr);
}
int drl_a3c_step_async(drl_a3c* h, int32_t slot) {
  DRL_ENTER(h);
  if (h->algo != 1) { set_error("not an A3C handle"); return DRL_ERR_INVALID; }
  return run_step(h, slot, forward_backward);
}
int drl_a3c_forward_backward(drl_a3c* h, int32_t slot) { return drl_apex_forward_backward(h, slot); }
int drl_a3c_grad_bucket(drl_a3c* h, void** dev_ptr, int64_t* count) { return drl_apex_grad_bucket(h, dev_ptr, count); }
int drl_a3c_apply(drl_a3c* h, float grad_scale) { return drl_apex_apply(h, grad_scale); }
int drl_a3c_wait(drl_a3c* h, drl_a3c_out* out) {
  DRL_ENTER(h);
  const float* r = nullptr;
  DRL_TRY(wait_step(h, nullptr, &r));
  if (out) {
    out->pi_loss = r[0]; out->baseline_loss = r[3]; out->entropy = r[4];
    out->learning_rate = r[1]; out->grad_norm = r[2]; out->step = result_row_step(r);
  }
  return DRL_OK;
}
int drl_a3c_step(drl_a3c* h, int32_t slot, drl_a3c_out* out) {
  DRL_TRY(drl_a3c_step_async(h, slot));
  return drl_a3c_wait(h, out);
}
int drl_a3c_act(drl_a3c* h, int32_t n, const uint8_t* state, const int32_t* previous_action, float* policy, float* value) {
  DRL_ENTER(h);
  if (n < 1 || n > 2 * h->B) { set_error("act: n must be in [1, %d]", 2 * h->B); return DRL_ERR_INVALID; }
  if (!state || !previous_action) { set_error("act: null pointer"); return DRL_ERR_INVALID; }
  ApexSlot& s = h->slots[h->cfg.num_slots];
  DRL_CUDA_CHECK(cudaStreamSynchronize(h->compute));
  DRL_TRY(stage_into(h, s, h->compute, n, n, state, nullptr, previous_action, nullptr, nullptr, nullptr, nullptr));
  pdl_break(h->compute);
  DRL_TRY(apex_forward(streams_of(h), h->pl, h->params, h->wi, s.frames, s.pa2, h->act, n, h->mode, h->main_images_stale,
                       h->main_images_stale, false, nullptr));
  h->main_images_stale = false;
  if (policy) DRL_CUDA_CHECK(cudaMemcpyAsync(policy, h->act.scratch_sm, (size_t)n * h->A * 4, cudaMemcpyDeviceToHost, h->compute));
  if (value) DRL_CUDA_CHECK(cudaMemcpyAsync(value, h->act.mstream, (size_t)n * 4, cudaMemcpyDeviceToHost, h->compute));
  DRL_CUDA_CHECK(cudaStreamSynchronize(h->compute));
  h->last_rows = 0;
  return DRL_OK;
}
int drl_a3c_taps(drl_a3c* h, float* policy, float* value, float* next_value, float* advantage) {
  DRL_ENTER(h);
  if (h->last_rows < 1) { set_error("taps: no step has run"); return DRL_ERR_STATE; }
  DRL_CUDA_CHECK(cudaStreamSynchronize(h->compute));
  const size_t n = h->last_rows, A = h->A;
  if (policy) DRL_CUDA_CHECK(cudaMemcpy(policy, h->act.scratch_sm, n * A * 4, cudaMemcpyDeviceToHost));
  if (value) DRL_CUDA_CHECK(cudaMemcpy(value, h->act.mstream, n * 4, cudaMemcpyDeviceToHost));
  if (next_value) DRL_CUDA_CHECK(cudaMemcpy(next_value, h->act.mstream + n, n * 4, cudaMemcpyDeviceToHost));
  if (advantage) DRL_CUDA_CHECK(cudaMemcpy(advantage, h->adv, n * 4, cudaMemcpyDeviceToHost));
  return DRL_OK;
}
int drl_a3c_read_buffer(drl_a3c* h, const char* name, float* host_dst, int64_t n) { return drl_apex_read_buffer(h, name, host_dst, n); }
int drl_a3c_profile_step(drl_a3c* h, int32_t slot, char* names, int64_t names_len, float* ms, int32_t max_kernels, int32_t* count) {
  return drl_apex_profile_step(h, slot, names, names_len, ms, max_kernels, count);
}
int drl_a3c_stream(drl_a3c* h, void** stream) { return drl_apex_stream(h, stream); }
int drl_a3c_launches_per_step(const drl_a3c* h, int32_t* n) { return drl_apex_launches_per_step(h, n); }

}  // extern "C"
