// r2d2.cu -- the R2D2 learner behind drl_r2d2_* (include/drl_b200.h): replaces r2d2.Agent's learner graph
// (agent/r2d2.py:13-95) over model/r2d2_lstm.py:28-116 (stored-state LSTM unroll, main and target scope),
// optimizer/burn_in.py:23-32 (value-function rescaling) and TF1 Adam.
//
// The reference unrolls `network` seq_len times per scope with the carried (h, c) multiplied by (1 - done_i) after
// step i (model/r2d2_lstm.py:67-84).  Only the LSTM cell is sequential: the convolutions, the action embedding and
// the input half of the LSTM contraction ([a3 | emb] W_x, 3392 of the 3456 kernel rows) do not depend on the carried
// state, so they run over all M = B*S rows at once through the same gather-GEMM kernels as the IMPALA learner
// (time-major rows m = t*B + b).  What remains per step is h_{t-1} W_h (64 x 256) + the gate nonlinearity: one
// persistent CTA per sequence keeps W_h in shared memory and walks the S steps (r2d2_lstm_fwd_kernel); BPTT is the
// mirror image (r2d2_lstm_bwd_kernel, W_h^T in shared memory), after which every weight / data gradient is again one
// batched GEMM over all M rows (all rows receive gradient: burn-in only slices the loss, agent/r2d2.py:64-68).
#include "adam_learner.cuh"

namespace drl {

constexpr int kR2L = 64;                 // lstm_size (config.json:93): the recurrence kernels keep W_h (L x 4L) on chip
constexpr int kR2G = 4 * kR2L;           // 256 gate columns
constexpr int kR2H = 128;                // dense width between the LSTM and the two output streams (model/r2d2_lstm.py:50)
constexpr int kR2Cat = Geo::FLAT + Geo::EMB;   // 3392 rows of the LSTM kernel that multiply the step input

struct R2Layout : FlatLayout<18> {
  int A, C;
  int64_t conv1_w, conv1_b, conv2_w, conv2_b, conv3_w, conv3_b, emb1_w, emb1_b, emb2_w, emb2_b;
  int64_t lstm_w, lstm_b, q1_w, q1_b, value_w, value_b, mean_w, mean_b;
  void init(int num_action, int channels) {
    A = num_action; C = channels;
    place({8 * 8 * (int64_t)C * 32, 32, 4 * 4 * 32 * 64, 64, 3 * 3 * 64 * 64, 64,
           (int64_t)A * 256, 256, 256 * 256, 256,
           (int64_t)(kR2Cat + kR2L) * kR2G, kR2G,
           (int64_t)kR2L * kR2H, kR2H, (int64_t)kR2H * A, A, kR2H, 1},
          {&conv1_w, &conv1_b, &conv2_w, &conv2_b, &conv3_w, &conv3_b, &emb1_w, &emb1_b, &emb2_w, &emb2_b, &lstm_w,
           &lstm_b, &q1_w, &q1_b, &value_w, &value_b, &mean_w, &mean_b});
  }
};

struct R2Acts {            // activations of one scope, time-major rows m = t*B + b
  float *a1, *a2, *a3, *e1, *table;
  float* zpart;            // [splits][M, 4L]: [a3 | emb] W_x partial sums
  float* zx;               // [M, 4L]: their sum (the recurrence reads one value per gate and step)
  float* gates;            // [M, 4L] sigmoid(i), tanh(j), sigmoid(f + 1), sigmoid(o)
  float *tc, *hout;        // [M, L] tanh(c_t), h_t (the cell output, BEFORE the done mask)
  float *hin, *cin;        // [M, L] the (masked) state that entered step t
  float* q1;               // [M, 128]
  float* q;                // [M, A]
};
struct R2Bwd {
  float *dq, *dmean;       // [M, 32]
  float *dq1, *dhout, *dz; // [M,128], [M,L], [M,4L]
  float *da3, *du, *dpre2, *dpre1, *da2, *da1, *wg_part, *wg_part2, *dcol;
};
struct R2In {              // one staged minibatch, caller's batch-major layout
  const uint8_t* frames;   // [B, S, 84, 84, C]
  const int32_t* pa;       // [B, S]
  const int32_t* action;   // [B, S]
  const float* h0;         // [B, L]
  const float* c0;         // [B, L]
  const float* reward;     // [B, S]
  const uint8_t* done;     // [B, S]
  const float* weight;     // [B]
};

// conv1 over single-channel frames (config.json:91 model_input [84, 84, 1]); the 4-channel instantiations are layer_defs'
using Conv1A1 = ConvFwdA<uint8_t, 84, 84, 1, 20, 20, 8, 4, true>;
using Conv1WA1 = ConvWgradA<uint8_t, 84, 84, 1, 20, 20, 8, 4, true>;

// [x | h_in]^T for the LSTM kernel gradient: feature index i < 3392 -> [a3 | emb] (as LstmAT), else h_in (device, time-major)
struct R2XhAT {
  static constexpr bool kContigK = false;
  const float* e; const float* table; const int* pa; const float* hin; RowMap map;
  struct Row { int i; };
  __device__ __forceinline__ Row row(int, int i) const { Row r; r.i = i; return r; }
  __device__ __forceinline__ float4 load(const Row& r, int m) const {
    if (r.i < 0) return zero4();
    const float* p;
    if (r.i < Geo::FLAT) p = e + (size_t)m * Geo::FLAT + r.i;
    else if (r.i < kR2Cat) p = table + (size_t)__ldg(pa + map.src(m)) * Geo::EMB + (r.i - Geo::FLAT);
    else p = hin + (size_t)m * kR2L + (r.i - kR2Cat);
    return __ldg(reinterpret_cast<const float4*>(p));
  }
};
// step input [a3 | emb[prev_action]] with the (t,b) -> (b,t) remap of prev_action (K = 3392)
struct R2XA {
  static constexpr bool kContigK = true;
  const float* e; const float* table; const int* pa; RowMap map;
  struct Row { const float *pe, *pu; };
  __device__ __forceinline__ Row row(int, int m) const {
    Row r;
    if (m < 0) { r.pe = nullptr; r.pu = nullptr; return r; }
    r.pe = e + (size_t)m * Geo::FLAT;
    r.pu = table + (size_t)__ldg(pa + map.src(m)) * Geo::EMB;
    return r;
  }
  __device__ __forceinline__ float4 load(const Row& r, int k) const {
    if (r.pe == nullptr) return zero4();
    return __ldg(reinterpret_cast<const float4*>((k < Geo::FLAT) ? r.pe + k : r.pu + (k - Geo::FLAT)));
  }
};

static SplitPlan plan_r2_x(int M, int mode) {
  return mode >= 2 ? plan_split(kR2Cat, cdiv(M, 128), 32, 1) : plan_split(kR2Cat, cdiv(M, CfgMid::BM) * (kR2G / CfgMid::BN), 16, 1);
}
// conv1 weight gradient with single-channel frames is a [64 x 32] output with K = M*400: half of a 128-row MMA tile
// would be padding and the producers, not the tensor pipe, set the pace (measured 0.20 ms at M = 1280 on the tcgen05
// core).  A 64 x 32 FFMA tile with the reduction split over ~4 CTAs per SM fits the shape in both math modes.
using CfgWgC1 = TileCfg<64, 32, 16, 4, 4>;
static SplitPlan plan_r2_conv1_wgrad(int M, int) { return plan_split(M * 400, 1, 16, 4); }

// ------------------------------------------------------------------------------------------
// LSTM recurrence, forward (model/r2d2_lstm.py:12-21 inside the unroll :67-84; TF 1.14 LSTMCell):
//   z_t = sum_s zpart[s][m] + b + h_in W_h ; i,j,f,o = split(z_t)
//   c_t = sigmoid(f + 1) c_in + sigmoid(i) tanh(j) ; h_t = sigmoid(o) tanh(c_t)         (h_t feeds the q head)
//   (h_in, c_in) of step t+1 = (h_t, c_t) * (1 - done_t)
// One CTA per sequence, 4L = 256 threads; thread j owns gate column j and keeps W_h[:, j] (L = 64 floats) in REGISTERS for
// all S steps: with W_h in shared memory every step re-read its 64 KB (512 clk of LDS bandwidth per SM, measured
// 1.36 us per step); from registers a step costs 16 broadcast LDS.128 of h plus 64 FMAs per thread.
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kR2G) r2d2_lstm_fwd_kernel(
    const float* __restrict__ zpart, int nsplit, size_t slab, const float* __restrict__ bias,
    const float* __restrict__ Wh, const float* __restrict__ h0, const float* __restrict__ c0,
    const uint8_t* __restrict__ done, float* __restrict__ gates, float* __restrict__ tc, float* __restrict__ hout,
    float* __restrict__ hin, float* __restrict__ cin, float* __restrict__ c_last, int B, int S) {
  pdl_prologue();
  __shared__ __align__(16) float sh[kR2L];
  __shared__ float sz[kR2G];
  const int b = blockIdx.x, j = threadIdx.x;
  float w[kR2L];
#pragma unroll
  for (int k = 0; k < kR2L; ++k) w[k] = Wh[k * kR2G + j];      // coalesced across the CTA, once
  float c_reg = 0.f;
  if (j < kR2L) { sh[j] = h0[(size_t)b * kR2L + j]; c_reg = c0[(size_t)b * kR2L + j]; }
  const float bj = bias[j];
  // the step input z_x[t] and done[t] do not depend on the recurrence: the loads of step t+1 are issued at the top of
  // step t so that their latency (L2 / HBM) is off the serial chain
  auto load_z = [&](int t) {
    const size_t m = (size_t)t * B + b;
    float z = 0.f;
    for (int s = 0; s < nsplit; ++s) z += zpart[(size_t)s * slab + m * kR2G + j];
    return z;
  };
  float z_next = load_z(0);
  float keep_next = (done && done[(size_t)b * S]) ? 0.f : 1.f;
  __syncthreads();
  for (int t = 0; t < S; ++t) {
    const size_t m = (size_t)t * B + b;
    const float z = bj + z_next;
    const float keep = keep_next;
    if (t + 1 < S) {
      z_next = load_z(t + 1);
      keep_next = (done && done[(size_t)b * S + t + 1]) ? 0.f : 1.f;
    }
    float acc0 = 0.f, acc1 = 0.f, acc2 = 0.f, acc3 = 0.f;      // four independent chains: 16 dependent FMAs each
#pragma unroll
    for (int k = 0; k < kR2L; k += 4) {
      const float4 h4 = *reinterpret_cast<const float4*>(sh + k);     // broadcast
      acc0 = fmaf(h4.x, w[k], acc0);
      acc1 = fmaf(h4.y, w[k + 1], acc1);
      acc2 = fmaf(h4.z, w[k + 2], acc2);
      acc3 = fmaf(h4.w, w[k + 3], acc3);
    }
    // every thread applies the nonlinearity of its own gate column (warp-uniform branch: L = 2 warps per gate), so
    // the serial tail below is left with one tanh instead of five transcendentals
    const float pre = z + ((acc0 + acc1) + (acc2 + acc3));
    const int gate = j / kR2L;
    const float actv = (gate == 1) ? tanhf(pre) : sigmoidf_acc(gate == 2 ? pre + 1.0f : pre);
    sz[j] = actv;
    gates[m * kR2G + j] = actv;
    if (j < kR2L) { hin[m * kR2L + j] = sh[j]; cin[m * kR2L + j] = c_reg; }
    __syncthreads();
    if (j < kR2L) {
      const float si = sz[j], tj = sz[kR2L + j], sf = sz[2 * kR2L + j], so = sz[3 * kR2L + j];
      const float c = sf * c_reg + si * tj;
      const float tcv = tanhf(c);
      const float h = so * tcv;
      tc[m * kR2L + j] = tcv;
      hout[m * kR2L + j] = h;
      if (c_last) c_last[m * kR2L + j] = c;
      c_reg = c * keep;
      sh[j] = h * keep;
    }
    __syncthreads();
  }
}

// BPTT through the same recurrence (rows of all S steps receive gradient):
//   dh_t = dhout[m] + (1 - done_t) dh_in[t+1] ; dc_t = (1 - done_t) dc_in[t+1] + dh_t so (1 - tc^2)
//   do = dh_t tc so(1-so) ; di = dc_t tj si(1-si) ; dj = dc_t si (1 - tj^2) ; df = dc_t c_in sf(1-sf)
//   dc_in[t] = dc_t sf ; dh_in[t] = dz_t W_h^T        (the weights again live in registers, 64 per thread)
__global__ void __launch_bounds__(kR2G) r2d2_lstm_bwd_kernel(
    const float* __restrict__ dhout, const float* __restrict__ gates, const float* __restrict__ tc,
    const float* __restrict__ cin, const float* __restrict__ Wh, const uint8_t* __restrict__ done,
    float* __restrict__ dz, int B, int S) {
  pdl_prologue();
  __shared__ __align__(16) float sdz[kR2G];
  __shared__ float sdh[kR2L];
  __shared__ float spart[4 * kR2L];
  const int b = blockIdx.x, tid = threadIdx.x;
  const int kk = tid & (kR2L - 1), q = tid / kR2L;
  // thread (kk, q) accumulates dh_in[kk] over gate columns [q L, (q+1) L): its 64 weights W_h[kk][q L + i] stay in registers
  float w[kR2L];
#pragma unroll
  for (int i = 0; i < kR2L; ++i) w[i] = Wh[(size_t)kk * kR2G + q * kR2L + i];
  float dc_carry = 0.f;
  if (tid < kR2L) sdh[tid] = 0.f;
  __syncthreads();
  // operands of step t-1 are fetched while step t computes (they do not depend on the recurrence)
  struct Ops { float dho, si, tj, sf, so, tcv, cprev, keep; };
  auto fetch = [&](int t) {
    Ops o{};
    if (tid < kR2L) {
      const size_t m = (size_t)t * B + b;
      const float* g = gates + m * kR2G;
      o.dho = dhout[m * kR2L + tid];
      o.si = g[tid]; o.tj = g[kR2L + tid]; o.sf = g[2 * kR2L + tid]; o.so = g[3 * kR2L + tid];
      o.tcv = tc[m * kR2L + tid];
      o.cprev = cin[m * kR2L + tid];
      o.keep = done[(size_t)b * S + t] ? 0.f : 1.f;
    }
    return o;
  };
  Ops nxt = fetch(S - 1);
  for (int t = S - 1; t >= 0; --t) {
    const size_t m = (size_t)t * B + b;
    const Ops cur = nxt;
    if (t > 0) nxt = fetch(t - 1);
    if (tid < kR2L) {
      const float keep = cur.keep;
      const float dh = cur.dho + keep * sdh[tid];
      const float si = cur.si, tj = cur.tj, sf = cur.sf, so = cur.so;
      const float tcv = cur.tcv;
      const float cprev = cur.cprev;
      const float d_o = dh * tcv * so * (1.f - so);
      const float dc = keep * dc_carry + dh * so * (1.f - tcv * tcv);
      const float di = dc * tj * si * (1.f - si);
      const float dj = dc * si * (1.f - tj * tj);
      const float df = dc * cprev * sf * (1.f - sf);
      sdz[tid] = di; sdz[kR2L + tid] = dj; sdz[2 * kR2L + tid] = df; sdz[3 * kR2L + tid] = d_o;
      dc_carry = dc * sf;
    }
    __syncthreads();
    dz[m * kR2G + tid] = sdz[tid];                    // coalesced store of the step's 4L gate gradients
    float acc0 = 0.f, acc1 = 0.f, acc2 = 0.f, acc3 = 0.f;
#pragma unroll
    for (int i = 0; i < kR2L; i += 4) {
      const float4 d4 = *reinterpret_cast<const float4*>(sdz + q * kR2L + i);   // broadcast within the warp
      acc0 = fmaf(d4.x, w[i], acc0);
      acc1 = fmaf(d4.y, w[i + 1], acc1);
      acc2 = fmaf(d4.z, w[i + 2], acc2);
      acc3 = fmaf(d4.w, w[i + 3], acc3);
    }
    spart[q * kR2L + kk] = (acc0 + acc1) + (acc2 + acc3);
    __syncthreads();
    // sdh[tid] is only read by the thread that writes it; spart / sdz are protected by the two barriers above
    if (tid < kR2L) sdh[tid] = (spart[tid] + spart[kR2L + tid]) + (spart[2 * kR2L + tid] + spart[3 * kR2L + tid]);
  }
}

// q[m][a] = (q1[m] Wv[:, a] + bv[a]) - (q1[m] wm + bm)      (model/r2d2_lstm.py:51-53); one warp per row
__global__ void __launch_bounds__(128) r2d2_out_kernel(const float* __restrict__ q1, const float* __restrict__ wv,
                                                        const float* __restrict__ bv, const float* __restrict__ wm,
                                                        const float* __restrict__ bm, float* __restrict__ q, int M, int A) {
  pdl_prologue();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int m = blockIdx.x * 4 + warp;
  if (m >= M) return;
  float x[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) x[i] = q1[(size_t)m * kR2H + lane + 32 * i];
  float mean = 0.f;
#pragma unroll
  for (int i = 0; i < 4; ++i) mean = fmaf(x[i], __ldg(wm + lane + 32 * i), mean);
  mean = warp_sum(mean) + bm[0];
  for (int a = 0; a < A; ++a) {
    float v = 0.f;
#pragma unroll
    for (int i = 0; i < 4; ++i) v = fmaf(x[i], __ldg(wv + (size_t)(lane + 32 * i) * A + a), v);
    v = warp_sum(v);
    if (lane == 0) q[(size_t)m * A + a] = (v + bv[a]) - mean;
  }
}

// dq1[m][k] = relu'(q1) (sum_a dq[m][a] Wv[k][a] + dmean[m] wm[k]);  grid = rows, 128 threads
__global__ void __launch_bounds__(kR2H) r2d2_out_bwd_kernel(const float* __restrict__ dq, const float* __restrict__ dmean,
                                                             const float* __restrict__ wv, const float* __restrict__ wm,
                                                             const float* __restrict__ q1, float* __restrict__ dq1, int A) {
  pdl_prologue();
  __shared__ float sd[32];
  __shared__ float sdm;
  const int m = blockIdx.x, k = threadIdx.x;
  if (k < A) sd[k] = dq[(size_t)m * 32 + k];
  if (k == 0) sdm = dmean[(size_t)m * 32];
  __syncthreads();
  float acc = sdm * __ldg(wm + k);
  for (int a = 0; a < A; ++a) acc = fmaf(sd[a], __ldg(wv + (size_t)k * A + a), acc);
  const size_t o = (size_t)m * kR2H + k;
  dq1[o] = (q1[o] > 0.f) ? acc : 0.f;
}

// ------------------------------------------------------------------------------------------
// TD targets, loss and head gradients (agent/r2d2.py:62-90), window i in [0, Nt), t = burn_in + i, Nt = S - burn_in - 1:
//   sav = main_q[b,t][action[b,t]] ; next_action = argmax main_q[b,t+1] (first maximum) ; nsav = target_q[b,t+1][next_action]
//   target = h(h^-1(nsav) * gamma (1 - done[b,t]) + reward[b,t])        (h = value_function_rescaling, eps 1e-3)
//   loss = mean_b w_b mean_i (target - sav)^2 ; td[b] = |mean_i (target - sav)|
// The two rescalings are evaluated in float64: h^-1 subtracts 1 from sqrt(1 + 4 eps (..)) ~ 1.002, which costs float32
// three digits.  One block; a warp owns sequences b = warp, warp + 8, ...; all reductions in a fixed order.
// ------------------------------------------------------------------------------------------
struct R2TdArgs {
  const float* mq; const float* tq;            // [M, A] time-major
  const int32_t* action; const float* reward; const uint8_t* done; const float* weight;   // batch-major; weight may be null
  float discount; int B, S, burn_in, A;
  float* sav; float* target_value;             // [B, Nt] taps
  float* td_dev; float* td_host;               // [B]
  float* dq; float* dmean;                     // [M, 32] or null
  float* loss;                                 // [1] or null
};
__device__ __forceinline__ double r2_h(double x) {
  const double s = (x > 0.0) - (x < 0.0);
  return s * (sqrt(fabs(x) + 1.0) - 1.0) + 1e-3 * x;
}
__device__ __forceinline__ double r2_hinv(double x) {
  const double s = (x > 0.0) - (x < 0.0);
  const double r = (sqrt(1.0 + 4.0 * 1e-3 * (fabs(x) + 1.0 + 1e-3)) - 1.0) / (2.0 * 1e-3);
  return s * (r * r - 1.0);
}
__global__ void __launch_bounds__(256) r2d2_td_kernel(R2TdArgs a) {
  pdl_prologue();
  __shared__ float red[8];
  const int Nt = a.S - a.burn_in - 1;
  const int M = a.B * a.S;
  if (a.dq) {      // rows outside the loss window carry no gradient; columns >= A / >= 1 are never written (stay zero)
    const int W = a.A + 1;
    for (int i = threadIdx.x; i < M * W; i += blockDim.x) {
      const int m = i / W, k = i - m * W;
      if (k < a.A) a.dq[(size_t)m * 32 + k] = 0.f;
      else a.dmean[(size_t)m * 32] = 0.f;
    }
    __syncthreads();
  }
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  float wloss = 0.f;
  for (int b = warp; b < a.B; b += 8) {
    const float w = a.weight ? a.weight[b] : 1.0f;
    float sdiff = 0.f, ssq = 0.f;
    for (int i = lane; i < Nt; i += 32) {
      const int t = a.burn_in + i;
      const size_t m = (size_t)t * a.B + b, mn = (size_t)(t + 1) * a.B + b;
      const int act = a.action[(size_t)b * a.S + t];
      float best = -INFINITY;
      int arg = 0;
      for (int k = 0; k < a.A; ++k) {
        const float v = a.mq[mn * a.A + k];
        if (v > best) { best = v; arg = k; }
      }
      const bool act_ok = act >= 0 && act < a.A;            // tf.one_hot: an out-of-range action selects nothing
      const float sav = act_ok ? a.mq[m * a.A + act] : 0.f;
      const float nsav = a.tq[mn * a.A + arg];
      const double disc = a.done[(size_t)b * a.S + t] ? 0.0 : (double)a.discount;
      const float target = (float)r2_h(r2_hinv((double)nsav) * disc + (double)a.reward[(size_t)b * a.S + t]);
      const float diff = target - sav;
      a.sav[(size_t)b * Nt + i] = sav;
      a.target_value[(size_t)b * Nt + i] = target;
      sdiff += diff;
      ssq += diff * diff;
      if (a.dq) {
        const float g = -2.0f * w * diff / ((float)Nt * (float)a.B);
        if (act_ok) {
          a.dq[m * 32 + act] = g;
          a.dmean[m * 32] = -g;
        }
      }
    }
    sdiff = warp_sum(sdiff);
    ssq = warp_sum(ssq);
    if (lane == 0) {
      const float td = fabsf(sdiff / (float)Nt);
      a.td_dev[b] = td;
      if (a.td_host) a.td_host[b] = td;
      wloss += w * (ssq / (float)Nt);
    }
  }
  if (a.loss) {
    if (lane == 0) red[warp] = wloss;
    __syncthreads();
    if (threadIdx.x == 0) {
      float s = 0.f;
#pragma unroll
      for (int i = 0; i < 8; ++i) s += red[i];
      *a.loss = s / (float)a.B;
    }
  }
}


constexpr size_t kR2FwdSmem = 0, kR2BwdSmem = 0;     // the recurrence kernels only use small static shared arrays

// Forward of one scope over B sequences of S steps (rows m = t*B + b).  c_last (optional): un-masked c_t (act path).
static int r2_forward(const Streams& st, const R2Layout& pl, const float* P, const WeightImages& wi, const R2In& in,
                      const R2Acts& act, float* c_last, int B, int S, int mode, bool retile_fwd, bool retile_bwd, bool tgt,
                      int* launches) {
  const int M = B * S;
  const RowMap map{B, S};
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
  if (pl.C == 1) {
    Conv1A1 al{in.frames, map};
    PlainB bl{P + pl.conv1_w, 32, 0};
    EpConv1 ep{act.a1, 32, P + pl.conv1_b, nullptr};
    GEMM(tgt ? "target_conv1_fwd" : "conv1_fwd", CfgN32, U32, al, bl, ep, M * 400, 32, 64, 1, 64, 0);
  } else {
    Conv1A al{in.frames, map};
    PlainB bl{P + pl.conv1_w, 32, 0};
    EpConv1 ep{act.a1, 32, P + pl.conv1_b, nullptr};
    GEMM(tgt ? "target_conv1_fwd" : "conv1_fwd", CfgN32, U32, al, bl, ep, M * 400, 32, 256, 1, 256, 0);
  }
  if (st.par) {
    DRL_CUDA_CHECK(cudaStreamWaitEvent(st.main, st.ev[7], 0));
    pdl_break(st.main);
  }
  {
    Conv2A al{act.a1, map};
    PlainB bl{P + pl.conv2_w, 64, 0};
    PretiledB<PlainB> blp{wi.img[1], 512 / 32};
    EpBiasAct<true, true> ep{act.a2, 64, 0, P + pl.conv2_b, 0, 1.0f};
    GEMM_W(tgt ? "target_conv2_fwd" : "conv2_fwd", CfgBig, U64L, al, bl, blp, ep, M * 81, 64, 512, 1, 512, 0);
  }
  {
    Conv3A al{act.a2, map};
    PlainB bl{P + pl.conv3_w, 64, 0};
    PretiledB<PlainB> blp{wi.img[2], 576 / 32};
    EpBiasAct<true, true> ep{act.a3, 64, 0, P + pl.conv3_b, 0, 1.0f};
    GEMM_W(tgt ? "target_conv3_fwd" : "conv3_fwd", CfgBig, U64L, al, bl, blp, ep, M * 49, 64, 576, 1, 576, 0);
  }
  DRL_TRY(join_from_side(st, 1));
  // input half of the LSTM contraction for all S steps at once: [M, 3392] x W[:3392, :4L] (split-K partial sums)
  const SplitPlan sp = plan_r2_x(M, mode);
  {
    R2XA al{act.a3, act.table, in.pa, map};
    PlainB bl{P + pl.lstm_w, kR2G, 0};
    EpRaw<false> ep{act.zpart, kR2G, (size_t)M * kR2G, 1.0f, 0, kR2G};
    GEMM(tgt ? "target_lstm_x_fwd" : "lstm_x_fwd", CfgMid, U256, al, bl, ep, M, kR2G, kR2Cat, sp.splits, sp.kchunk, sp.kchunk);
  }
  KERNEL(tgt ? "target_lstm_x_reduce" : "lstm_x_reduce",
         splitk_reduce(s, act.zpart, (size_t)M * kR2G, sp.splits, act.zx, (size_t)M * kR2G), 1);
  prof_mark(s, tgt ? "target_lstm_unroll_fwd" : "lstm_unroll_fwd");
  DRL_CUDA_CHECK((launch_k(r2d2_lstm_fwd_kernel, B, kR2G, kR2FwdSmem, s, act.zx, 1, (size_t)0,
                           P + pl.lstm_b, P + pl.lstm_w + (size_t)kR2Cat * kR2G, in.h0, in.c0, in.done, act.gates, act.tc,
                           act.hout, act.hin, act.cin, c_last, B, S)));
  ++n;
  {  // dense 128 ReLU (model/r2d2_lstm.py:50)
    PlainA al{act.hout, kR2L, 0};
    PlainB bl{P + pl.q1_w, kR2H, 0};
    EpBiasAct<true, true> ep{act.q1, kR2H, 0, P + pl.q1_b, 0, 1.0f};
    GEMM_FFMA(tgt ? "target_q1_fwd" : "q1_fwd", CfgSmall, al, bl, ep, M, kR2H, kR2L, 1, kR2L, 0);
  }
  prof_mark(s, tgt ? "target_q_out_fwd" : "q_out_fwd");
  DRL_CUDA_CHECK((launch_k(r2d2_out_kernel, cdiv(M, 4), 128, 0, s, act.q1, P + pl.value_w, P + pl.value_b, P + pl.mean_w,
                           P + pl.mean_b, act.q, M, pl.A)));
  ++n;
  if (launches) *launches += n;
  return DRL_OK;
}

static int r2_backward(const Streams& st, const R2Layout& pl, const float* P, const WeightImages& wi, float* G,
                       const R2In& in, const R2Acts& act, const R2Bwd& bw, int B, int S, int mode, int* launches) {
  PdlRegionOff pdl_region;
  const int M = B * S;
  const RowMap map{B, S};
  cudaStream_t s = st.main;
  const cudaStream_t side = st.par ? st.side : st.main;
  const int A = pl.A;
  int n = 0;
  prof_mark(s, "q_out_bwd");
  DRL_CUDA_CHECK((launch_k(r2d2_out_bwd_kernel, M, kR2H, 0, s, bw.dq, bw.dmean, P + pl.value_w, P + pl.mean_w, act.q1,
                           bw.dq1, A)));
  ++n;
  DRL_TRY(fork_to_side(st, 0));
  s = side;
  {  // d value [128(+1), A]
    PlainAT al{act.q1, kR2H, 0};
    PlainB bl{bw.dq, 32, 0};
    EpRaw<true> ep{G + pl.value_w, A, 0, 1.0f, kR2H, A};
    GEMM_FFMA("value_wgrad", CfgSmall, al, bl, ep, kR2H, 32, M, 1, M, 0);
  }
  {  // d mean [128(+1), 1]
    PlainAT al{act.q1, kR2H, 0};
    PlainB bl{bw.dmean, 32, 0};
    EpRaw<true> ep{G + pl.mean_w, 1, 0, 1.0f, kR2H, 1};
    GEMM_FFMA("mean_wgrad", CfgSmall, al, bl, ep, kR2H, 32, M, 1, M, 0);
  }
  {  // d q1 kernel [L(+1), 128] = hout^T dq1
    PlainAT al{act.hout, kR2L, 0};
    PlainB bl{bw.dq1, kR2H, 0};
    EpRaw<true> ep{G + pl.q1_w, kR2H, 0, 1.0f, kR2L, kR2H};
    GEMM_FFMA("q1_wgrad", CfgSmall, al, bl, ep, kR2L, kR2H, M, 1, M, 0);
  }
  s = st.main;
  {  // dhout = dq1 W1^T
    PlainA al{bw.dq1, kR2H, 0};
    PlainBT bl{P + pl.q1_w, kR2H, 0};
    EpRaw<false> ep{bw.dhout, kR2L, 0, 1.0f, 0, kR2L};
    GEMM_FFMA("q1_dgrad", CfgSmall, al, bl, ep, M, kR2L, kR2H, 1, kR2H, 0);
  }
  prof_mark(s, "lstm_unroll_bwd");
  DRL_CUDA_CHECK((launch_k(r2d2_lstm_bwd_kernel, B, kR2G, kR2BwdSmem, s, bw.dhout, act.gates, act.tc, act.cin,
                           P + pl.lstm_w + (size_t)kR2Cat * kR2G, in.done, bw.dz, B, S)));
  ++n;
  DRL_TRY(fork_to_side(st, 3));
  s = side;
  {  // d lstm kernel [3456(+1), 256] = [x | h_in]^T dz ; bias gradient = column sums of dz
    R2XhAT al{act.a3, act.table, in.pa, act.hin, map};
    PlainB bl{bw.dz, kR2G, 0};
    EpRaw<true> ep{G + pl.lstm_w, kR2G, 0, 1.0f, kR2Cat + kR2L, kR2G};
    GEMM("lstm_wgrad", CfgBig, U256, al, bl, ep, kR2Cat + kR2L, kR2G, M, 1, M, 0);
  }
  s = st.main;
  {  // d[a3 | emb] = dz W[:3392]^T
    PlainA al{bw.dz, kR2G, 0};
    PlainBT bl{P + pl.lstm_w, kR2G, 0};
    EpLstmDx ep{bw.da3, act.a3, bw.du};
    GEMM("lstm_dgrad", CfgMid, U128, al, bl, ep, M, kR2Cat, kR2G, 1, kR2G, 0);
  }
  DRL_TRY(fork_to_side(st, 4));
  s = side;
  KERNEL("emb_bwd",
         emb_backward(s, bw.du, in.pa, act.e1, act.table, P + pl.emb2_w, bw.dpre2, bw.dpre1, G + pl.emb1_w,
                      G + pl.emb1_b, G + pl.emb2_w, G + pl.emb2_b, bw.wg_part, M, B, S, A), 4);
  {
    const SplitPlan sp = plan_conv3_wgrad(M, mode);
    const size_t slab = 577 * 64;
    Conv3WA al{act.a2, map};
    PlainB bl{bw.da3, 64, 0};
    EpRaw<true> ep{bw.wg_part, 64, slab, 1.0f, 576, 64};
    GEMM("conv3_wgrad", CfgBig, U64, al, bl, ep, 576, 64, M * 49, sp.splits, sp.kchunk, sp.kchunk);
    KERNEL("conv3_wgrad_reduce", splitk_reduce(s, bw.wg_part, slab, sp.splits, G + pl.conv3_w, slab), 1);
  }
  s = st.main;
  if (mode >= 2) {
    PlainA al{bw.da3, 64, 0};
    EpRaw<false> ep{bw.dcol, 576, 0, 1.0f, 0, 576};
    prof_mark(s, "conv3_dgrad");
    PretiledB<PlainBT> blp{wi.img[5], 2};
    DRL_TRY((launch_gemm_umma_persist<PersistOf<U256>::type>(s, al, blp, ep, M * 49, 576, 64, 1, 64, 0)));
    prof_mark(s, "conv3_col2im");
    DRL_TRY(col2im_conv3(s, bw.dcol, act.a2, bw.da2, M));
    n += 2;
  } else {
    Conv3DA al{bw.da3};
    Conv3DB bl{P + pl.conv3_w};
    Conv3DE ep{bw.da2, act.a2};
    GEMM_FFMA("conv3_dgrad", CfgBig, al, bl, ep, M * 81, 64, 576, 1, 576, 0);
  }
  DRL_TRY(fork_to_side(st, 5));
  s = side;
  {
    const SplitPlan sp = plan_conv2_wgrad(M, mode);
    const size_t slab = 513 * 64;
    Conv2WA al{act.a1, map};
    PlainB bl{bw.da2, 64, 0};
    EpRaw<true> ep{bw.wg_part, 64, slab, 1.0f, 512, 64};
    GEMM("conv2_wgrad", CfgBig, U64, al, bl, ep, 512, 64, M * 81, sp.splits, sp.kchunk, sp.kchunk);
    KERNEL("conv2_wgrad_reduce", splitk_reduce(s, bw.wg_part, slab, sp.splits, G + pl.conv2_w, slab), 1);
  }
  s = st.main;
  if (mode >= 2) {
    PlainA al{bw.da2, 64, 0};
    EpRaw<false> ep{bw.dcol, 512, 0, 1.0f, 0, 512};
    prof_mark(s, "conv2_dgrad");
    PretiledB<PlainBT> blp{wi.img[6], 2};
    DRL_TRY((launch_gemm_umma_persist<PersistOf<U256>::type>(s, al, blp, ep, M * 81, 512, 64, 1, 64, 0)));
    prof_mark(s, "conv2_col2im");
    DRL_TRY(col2im_conv2(s, bw.dcol, act.a1, bw.da1, M));
    n += 2;
  } else {
    Conv2DA al{bw.da2};
    Conv2DB bl{P + pl.conv2_w};
    Conv2DE ep{bw.da1, act.a1};
    GEMM_FFMA("conv2_dgrad", CfgN32, al, bl, ep, M * 100, 32, 256, 4, 256, 0);
  }
  if (pl.C == 1) {
    const SplitPlan sp = plan_r2_conv1_wgrad(M, mode);
    const size_t slab = 65 * 32;
    Conv1WA1 al{in.frames, map};
    PlainB bl{bw.da1, 32, 0};
    EpRaw<true> ep{bw.wg_part2, 32, slab, 1.0f / 255.0f, 64, 32};
    GEMM_FFMA("conv1_wgrad", CfgWgC1, al, bl, ep, 64, 32, M * 400, sp.splits, sp.kchunk, sp.kchunk);
    KERNEL("conv1_wgrad_reduce", splitk_reduce(s, bw.wg_part2, slab, sp.splits, G + pl.conv1_w, slab), 1);
  } else {
    const SplitPlan sp = plan_conv1_wgrad(M, mode);
    const size_t slab = 257 * 32;
    Conv1WA al{in.frames, map};
    PlainB bl{bw.da1, 32, 0};
    EpRaw<true> ep{bw.wg_part2, 32, slab, 1.0f / 255.0f, 256, 32};
    GEMM("conv1_wgrad", CfgWg1, U32, al, bl, ep, 256, 32, M * 400, sp.splits, sp.kchunk, sp.kchunk);
    KERNEL("conv1_wgrad_reduce", splitk_reduce(s, bw.wg_part2, slab, sp.splits, G + pl.conv1_w, slab), 1);
  }
  DRL_TRY(join_from_side(st, 6));
  if (launches) *launches += n;
  return DRL_OK;
}

}  // namespace drl

using namespace drl;

struct drl_r2d2 : AdamLearner {
  drl_r2d2_config cfg{};
  int S = 0, A = 0, C = 1, Nt = 0;
  size_t frame = 0;
  R2Layout pl{};
  R2Acts act{}, tact{};
  R2Bwd bwd{};
  float *sav = nullptr, *target_value = nullptr, *td_dev = nullptr, *c_last = nullptr;
  std::vector<R2In> slots;     // payloads of AdamLearner::sync
};

namespace {

int alloc_acts(drl_r2d2* h, R2Acts& a) {
  const size_t M = (size_t)h->B * h->S, A = h->A;
  DRL_TRY(dev_alloc(h, &a.a1, M * 400 * 32));
  DRL_TRY(dev_alloc(h, &a.a2, M * 81 * 64));
  DRL_TRY(dev_alloc(h, &a.a3, M * Geo::FLAT));
  DRL_TRY(dev_alloc(h, &a.e1, A * Geo::EMB));
  DRL_TRY(dev_alloc(h, &a.table, A * Geo::EMB));
  size_t zmax = 0;
  for (int mode = 1; mode <= 2; ++mode)
    for (int m = 1; m <= (int)M; ++m) zmax = std::max(zmax, (size_t)plan_r2_x(m, mode).splits * m * kR2G);
  DRL_TRY(dev_alloc(h, &a.zpart, zmax));
  DRL_TRY(dev_alloc(h, &a.zx, M * kR2G));
  DRL_TRY(dev_alloc(h, &a.gates, M * kR2G));
  DRL_TRY(dev_alloc(h, &a.tc, M * kR2L));
  DRL_TRY(dev_alloc(h, &a.hout, M * kR2L));
  DRL_TRY(dev_alloc(h, &a.hin, M * kR2L));
  DRL_TRY(dev_alloc(h, &a.cin, M * kR2L));
  DRL_TRY(dev_alloc(h, &a.q1, M * kR2H));
  DRL_TRY(dev_alloc(h, &a.q, M * A));
  return DRL_OK;
}

// both unrolls + TD kernel over nb sequences held by `in`
int enqueue_forward_td(drl_r2d2* h, const R2In& in, int nb, bool train, float* td_host, int* launches) {
  pdl_break(h->compute);
  pdl_break(h->side);
  const Streams st = streams_of(h), tst = target_streams_of(h);
  // the two unrolls are independent (and each recurrence kernel only occupies nb SMs): the target scope runs on its
  // own stream pair beside the main scope and joins before the TD kernel
  DRL_TRY(fork_target(h));
  DRL_TRY(r2_forward(tst, h->pl, h->target, h->twi, in, h->tact, nullptr, nb, h->S, h->mode, h->target_images_stale, false,
                     true, launches));
  h->target_images_stale = false;
  DRL_TRY(target_done(h));
  DRL_TRY(r2_forward(st, h->pl, h->params, h->wi, in, h->act, nullptr, nb, h->S, h->mode, h->main_images_stale,
                     h->main_images_stale, false, launches));
  h->main_images_stale = false;
  DRL_TRY(join_target(h));
  R2TdArgs a{};
  a.mq = h->act.q; a.tq = h->tact.q;
  a.action = in.action; a.reward = in.reward; a.done = in.done; a.weight = train ? in.weight : nullptr;
  a.discount = h->cfg.discount_factor; a.B = nb; a.S = h->S; a.burn_in = h->cfg.burn_in; a.A = h->A;
  a.sav = h->sav; a.target_value = h->target_value; a.td_dev = h->td_dev; a.td_host = td_host;
  a.dq = train ? h->bwd.dq : nullptr; a.dmean = train ? h->bwd.dmean : nullptr;
  a.loss = train ? h->loss : nullptr;
  prof_mark(h->compute, "td_target_loss");
  DRL_CUDA_CHECK((launch_k(r2d2_td_kernel, 1, 256, 0, h->compute, a)));
  if (launches) *launches += 1;
  return DRL_OK;
}

// the step's unrolls, loss and BPTT (FwdBwd of the shell, adam_learner.cuh)
int forward_backward(drl_r2d2* h, int slot, int* launches) {
  const R2In& in = h->slots[slot];
  DRL_TRY(enqueue_forward_td(h, in, h->B, true, h->d_td + (size_t)slot * h->B, launches));
  return r2_backward(streams_of(h), h->pl, h->params, h->wi, h->grads, in, h->act, h->bwd, h->B, h->S, h->mode, launches);
}

// H2D of nb sequences into slot s on `stream` (fields that are null are skipped)
int stage_into(drl_r2d2* h, R2In& s, cudaStream_t stream, int nb, int steps, const uint8_t* state,
               const int32_t* previous_action, const int32_t* action, const float* h0, const float* c0, const float* reward,
               const uint8_t* done, const float* weight) {
  auto cp = [&](const void* dst, const void* src, size_t bytes) -> cudaError_t {
    return cudaMemcpyAsync(const_cast<void*>(dst), src, bytes, cudaMemcpyHostToDevice, stream);
  };
  const size_t n = (size_t)nb * steps;
  DRL_CUDA_CHECK(cp(s.frames, state, n * h->frame));
  DRL_CUDA_CHECK(cp(s.pa, previous_action, n * 4));
  if (action) DRL_CUDA_CHECK(cp(s.action, action, n * 4));
  DRL_CUDA_CHECK(cp(s.h0, h0, (size_t)nb * kR2L * 4));
  DRL_CUDA_CHECK(cp(s.c0, c0, (size_t)nb * kR2L * 4));
  if (reward) DRL_CUDA_CHECK(cp(s.reward, reward, n * 4));
  if (done) DRL_CUDA_CHECK(cp(s.done, done, n));
  if (reward) DRL_CUDA_CHECK(cp(s.weight, weight ? weight : h->h_ones, (size_t)nb * 4));
  return DRL_OK;
}

}  // namespace

extern "C" {

int drl_r2d2_create(const drl_r2d2_config* cfg, drl_r2d2** out) {
  if (!cfg || !out) { set_error("null argument"); return DRL_ERR_INVALID; }
  *out = nullptr;
  if (cfg->height != Geo::IH || cfg->width != Geo::IW || (cfg->channels != 1 && cfg->channels != 4)) {
    set_error("only 84x84x1 (config.json:91) and 84x84x4 frames are supported (got %dx%dx%d)", cfg->height, cfg->width, cfg->channels);
    return DRL_ERR_INVALID;
  }
  if (cfg->lstm_size != kR2L) { set_error("only lstm_size %d (config.json:93) is supported (got %d)", kR2L, cfg->lstm_size); return DRL_ERR_INVALID; }
  if (cfg->num_action < 2 || cfg->num_action > 32) { set_error("num_action must be in [2,32]"); return DRL_ERR_INVALID; }
  if (cfg->batch < 1) { set_error("batch must be >= 1"); return DRL_ERR_INVALID; }
  if (cfg->seq_len < 2 || cfg->burn_in < 0 || cfg->burn_in > cfg->seq_len - 2) {
    set_error("need seq_len >= 2 and 0 <= burn_in <= seq_len - 2 (got seq_len %d, burn_in %d)", cfg->seq_len, cfg->burn_in);
    return DRL_ERR_INVALID;
  }
  if (cfg->math_mode < 0 || cfg->math_mode > 2) { set_error("math_mode must be 0 (default), 1 (FP32 FFMA) or 2 (tcgen05 3xTF32)"); return DRL_ERR_INVALID; }
  if (drl_device_count() <= cfg->device) { set_error("CUDA device %d not available (no CPU fallback)", cfg->device); return DRL_ERR_CUDA; }
  drl_r2d2* h = new drl_r2d2();
  h->cfg = *cfg;
  h->mode = (cfg->math_mode == 0) ? DRL_DEFAULT_MATH_MODE : cfg->math_mode;
  if (h->cfg.num_slots < 1) h->cfg.num_slots = 2;
  h->B = cfg->batch; h->S = cfg->seq_len; h->A = cfg->num_action; h->C = cfg->channels;
  h->Nt = cfg->seq_len - cfg->burn_in - 1;
  h->frame = (size_t)Geo::IH * Geo::IW * h->C;
  h->pl.init(h->A, h->C);
  int rc = [&]() -> int {
    const size_t B = h->B, S = h->S, M = B * S, A = h->A;
    // constant learning rate (agent/r2d2.py:91); minimize(): no clipping
    DRL_TRY(create_shell(h, M, AdamSchedule{cfg->learning_rate, cfg->learning_rate, 1.0, 0.0f}));
    DRL_TRY(alloc_acts(h, h->act));
    DRL_TRY(alloc_acts(h, h->tact));
    R2Bwd& b = h->bwd;
    DRL_TRY(dev_alloc(h, &b.dq, M * 32));
    DRL_TRY(dev_alloc(h, &b.dmean, M * 32));
    DRL_TRY(dev_alloc(h, &b.dq1, M * kR2H));
    DRL_TRY(dev_alloc(h, &b.dhout, M * kR2L));
    DRL_TRY(dev_alloc(h, &b.dz, M * kR2G));
    DRL_TRY(dev_alloc(h, &b.da3, M * Geo::FLAT));
    DRL_TRY(dev_alloc(h, &b.du, M * Geo::EMB));
    DRL_TRY(dev_alloc(h, &b.dpre2, A * Geo::EMB));
    DRL_TRY(dev_alloc(h, &b.dpre1, A * Geo::EMB));
    DRL_TRY(dev_alloc(h, &b.da2, M * 81 * 64));
    DRL_TRY(dev_alloc(h, &b.da1, M * 400 * 32));
    size_t wg = wgrad_partial_floats((int)M, 3);                       // rows with gradient = M * (3 - 2)
    for (int mode = 1; mode <= 2; ++mode) wg = std::max(wg, (size_t)plan_r2_conv1_wgrad((int)M, mode).splits * 65 * 32);
    DRL_TRY(dev_alloc(h, &b.wg_part, wg));
    DRL_TRY(dev_alloc(h, &b.wg_part2, wg));
    DRL_TRY(dev_alloc(h, &b.dcol, M * 81 * 512));
    const size_t Nt = h->Nt;
    DRL_TRY(dev_alloc(h, &h->sav, B * Nt));
    DRL_TRY(dev_alloc(h, &h->target_value, B * Nt));
    DRL_TRY(dev_alloc(h, &h->td_dev, B));
    DRL_TRY(dev_alloc(h, &h->c_last, M * kR2L));
    h->slots.resize(h->sync.size());
    for (R2In& s : h->slots) {
      size_t off = 0;
      const size_t o_fr = off; off = align_up(off + M * h->frame, 256);
      const size_t o_pa = off; off = align_up(off + M * 4, 256);
      const size_t o_ac = off; off = align_up(off + M * 4, 256);
      const size_t o_h = off; off = align_up(off + M * kR2L * 4, 256);    // room for M rows: the act path stages n <= M states
      const size_t o_c = off; off = align_up(off + M * kR2L * 4, 256);
      const size_t o_rw = off; off = align_up(off + M * 4, 256);
      const size_t o_dn = off; off = align_up(off + M, 256);
      const size_t o_wt = off; off = align_up(off + M * 4, 256);
      uint8_t* base = nullptr;
      DRL_TRY(dev_alloc(h, &base, off));
      s.frames = base + o_fr;
      s.pa = reinterpret_cast<int32_t*>(base + o_pa);
      s.action = reinterpret_cast<int32_t*>(base + o_ac);
      s.h0 = reinterpret_cast<float*>(base + o_h);
      s.c0 = reinterpret_cast<float*>(base + o_c);
      s.reward = reinterpret_cast<float*>(base + o_rw);
      s.done = base + o_dn;
      s.weight = reinterpret_cast<float*>(base + o_wt);
    }
    DRL_CUDA_CHECK(cudaDeviceSynchronize());
    return DRL_OK;
  }();
  return finish_create(h, rc, out);
}

int drl_r2d2_destroy(drl_r2d2* h) { return destroy_shell(h); }

int drl_r2d2_param_count(const drl_r2d2* h, int64_t* n) {
  DRL_ENTER(h);
  if (!n) { set_error("null argument"); return DRL_ERR_INVALID; }
  *n = h->pl.packed_total;
  return DRL_OK;
}
int drl_r2d2_set_params(drl_r2d2* h, int32_t which, const float* host_flat, int64_t n) {
  DRL_ENTER(h);
  return set_params(h, which, host_flat, n);
}
int drl_r2d2_get_params(drl_r2d2* h, int32_t which, float* host_flat, int64_t n) {
  DRL_ENTER(h);
  return get_params(h, which, host_flat, n);
}
int drl_r2d2_set_opt_state(drl_r2d2* h, const float* host_m, const float* host_v, int64_t n, int64_t step,
                           float beta1_power, float beta2_power) {
  DRL_ENTER(h);
  return set_opt_state(h, host_m, host_v, n, step, beta1_power, beta2_power);
}
int drl_r2d2_get_opt_state(drl_r2d2* h, float* host_m, float* host_v, int64_t n, int64_t* step, float* beta1_power,
                           float* beta2_power) {
  DRL_ENTER(h);
  return get_opt_state(h, host_m, host_v, n, step, beta1_power, beta2_power);
}
int drl_r2d2_get_grads(drl_r2d2* h, float* host_flat, int64_t n) {
  DRL_ENTER(h);
  return get_grads(h, host_flat, n);
}
int drl_r2d2_main_to_target(drl_r2d2* h) {
  DRL_ENTER(h);
  return copy_main_to_target(h);
}

int drl_r2d2_stage(drl_r2d2* h, int32_t slot, const uint8_t* state, const int32_t* previous_action, const int32_t* action,
                   const float* h0, const float* c0, const float* reward, const uint8_t* done, const float* weight) {
  DRL_ENTER(h);
  if (!state || !previous_action || !action || !h0 || !c0 || !reward || !done) { set_error("stage: null input pointer"); return DRL_ERR_INVALID; }
  return stage_slot(h, slot, [&](cudaStream_t s) {
    return stage_into(h, h->slots[slot], s, h->B, h->S, state, previous_action, action, h0, c0, reward, done, weight);
  });
}

int drl_r2d2_step_async(drl_r2d2* h, int32_t slot) {
  DRL_ENTER(h);
  return run_step(h, slot, forward_backward);
}
int drl_r2d2_forward_backward(drl_r2d2* h, int32_t slot) {
  DRL_ENTER(h);
  return run_forward_backward(h, slot, forward_backward);
}
int drl_r2d2_grad_bucket(drl_r2d2* h, void** dev_ptr, int64_t* count) {
  DRL_ENTER(h);
  return grad_bucket(h, dev_ptr, count);
}
int drl_r2d2_apply(drl_r2d2* h, float grad_scale) {
  DRL_ENTER(h);
  return run_apply(h, grad_scale);
}
int drl_r2d2_wait(drl_r2d2* h, drl_r2d2_out* out, float* td_error) {
  DRL_ENTER(h);
  const float* r = nullptr;
  DRL_TRY(wait_step(h, td_error, &r));
  if (out) {
    out->loss = r[0];
    out->grad_norm = r[2];
    out->step = result_row_step(r);
  }
  return DRL_OK;
}
int drl_r2d2_step(drl_r2d2* h, int32_t slot, drl_r2d2_out* out, float* td_error) {
  DRL_TRY(drl_r2d2_step_async(h, slot));
  return drl_r2d2_wait(h, out, td_error);
}

int drl_r2d2_td_error(drl_r2d2* h, int32_t n, const uint8_t* state, const int32_t* previous_action, const int32_t* action,
                      const float* h0, const float* c0, const float* reward, const uint8_t* done, float* td_error) {
  DRL_ENTER(h);
  if (n < 1 || n > h->B) { set_error("td_error: n must be in [1, %d]", h->B); return DRL_ERR_INVALID; }
  if (!state || !previous_action || !action || !h0 || !c0 || !reward || !done || !td_error) { set_error("td_error: null pointer"); return DRL_ERR_INVALID; }
  R2In& s = h->slots[h->cfg.num_slots];
  DRL_CUDA_CHECK(cudaStreamSynchronize(h->compute));
  DRL_TRY(stage_into(h, s, h->compute, n, h->S, state, previous_action, action, h0, c0, reward, done, nullptr));
  DRL_TRY(enqueue_forward_td(h, s, n, false, nullptr, nullptr));
  DRL_CUDA_CHECK(cudaMemcpyAsync(td_error, h->td_dev, (size_t)n * 4, cudaMemcpyDeviceToHost, h->compute));
  DRL_CUDA_CHECK(cudaStreamSynchronize(h->compute));
  h->last_rows = n;
  return DRL_OK;
}

int drl_r2d2_act(drl_r2d2* h, int32_t n, const uint8_t* state, const int32_t* previous_action, const float* h_in,
                 const float* c_in, float* q_value, float* h_out, float* c_out) {
  DRL_ENTER(h);
  const int M = h->B * h->S;
  if (n < 1 || n > M) { set_error("act: n must be in [1, %d]", M); return DRL_ERR_INVALID; }
  if (!state || !previous_action || !h_in || !c_in) { set_error("act: null pointer"); return DRL_ERR_INVALID; }
  R2In& s = h->slots[h->cfg.num_slots];
  DRL_CUDA_CHECK(cudaStreamSynchronize(h->compute));
  DRL_TRY(stage_into(h, s, h->compute, n, 1, state, previous_action, nullptr, h_in, c_in, nullptr, nullptr, nullptr));
  pdl_break(h->compute);
  pdl_break(h->side);
  R2In in = s;
  in.done = nullptr;                                     // a single step: nothing is carried
  DRL_TRY(r2_forward(streams_of(h), h->pl, h->params, h->wi, in, h->act, h->c_last, n, 1, h->mode, h->main_images_stale,
                     h->main_images_stale, false, nullptr));
  h->main_images_stale = false;
  if (q_value) DRL_CUDA_CHECK(cudaMemcpyAsync(q_value, h->act.q, (size_t)n * h->A * 4, cudaMemcpyDeviceToHost, h->compute));
  if (h_out) DRL_CUDA_CHECK(cudaMemcpyAsync(h_out, h->act.hout, (size_t)n * kR2L * 4, cudaMemcpyDeviceToHost, h->compute));
  if (c_out) DRL_CUDA_CHECK(cudaMemcpyAsync(c_out, h->c_last, (size_t)n * kR2L * 4, cudaMemcpyDeviceToHost, h->compute));
  DRL_CUDA_CHECK(cudaStreamSynchronize(h->compute));
  h->last_rows = 0;
  return DRL_OK;
}

int drl_r2d2_taps(drl_r2d2* h, float* main_q, float* target_q, float* target_value, float* state_action_value) {
  DRL_ENTER(h);
  if (h->last_rows < 1) { set_error("taps: no step or td_error call has run"); return DRL_ERR_STATE; }
  DRL_CUDA_CHECK(cudaStreamSynchronize(h->compute));
  const int nb = h->last_rows, S = h->S, A = h->A;
  // time-major device rows -> batch-major host arrays [nb, S, A]
  for (int which = 0; which < 2; ++which) {
    float* dst = which == 0 ? main_q : target_q;
    if (!dst) continue;
    std::vector<float> tmp((size_t)nb * S * A);
    DRL_CUDA_CHECK(cudaMemcpy(tmp.data(), which == 0 ? h->act.q : h->tact.q, tmp.size() * 4, cudaMemcpyDeviceToHost));
    for (int t = 0; t < S; ++t)
      for (int b = 0; b < nb; ++b)
        memcpy(dst + ((size_t)b * S + t) * A, tmp.data() + ((size_t)t * nb + b) * A, A * sizeof(float));
  }
  const size_t nt = (size_t)nb * h->Nt;
  if (target_value) DRL_CUDA_CHECK(cudaMemcpy(target_value, h->target_value, nt * 4, cudaMemcpyDeviceToHost));
  if (state_action_value) DRL_CUDA_CHECK(cudaMemcpy(state_action_value, h->sav, nt * 4, cudaMemcpyDeviceToHost));
  return DRL_OK;
}

int drl_r2d2_read_buffer(drl_r2d2* h, const char* name, float* host_dst, int64_t n) {
  DRL_ENTER(h);
  if (!name || !host_dst) { set_error("null argument"); return DRL_ERR_INVALID; }
  if (h->last_rows < 1) { set_error("read_buffer: no step or td_error call has run"); return DRL_ERR_STATE; }
  const size_t M = (size_t)h->last_rows * h->S, A = h->A;
  const NamedBuffer tab[] = {
      {"a1", h->act.a1, M * 400 * 32}, {"a2", h->act.a2, M * 81 * 64}, {"a3", h->act.a3, M * Geo::FLAT},
      {"emb", h->act.table, A * Geo::EMB}, {"e1", h->act.e1, A * Geo::EMB}, {"q1", h->act.q1, M * kR2H},
      {"hout", h->act.hout, M * kR2L}, {"hin", h->act.hin, M * kR2L}, {"cin", h->act.cin, M * kR2L},
      {"gates", h->act.gates, M * kR2G}, {"dz", h->bwd.dz, M * kR2G}, {"dhout", h->bwd.dhout, M * kR2L},
      {"da3", h->bwd.da3, M * Geo::FLAT}};
  return read_named_buffer(h->compute, tab, sizeof(tab) / sizeof(tab[0]), name, host_dst, n);
}

int drl_r2d2_profile_step(drl_r2d2* h, int32_t slot, char* names, int64_t names_len, float* ms, int32_t max_kernels,
                          int32_t* count) {
  DRL_ENTER(h);
  return profile_step(h, slot, forward_backward, names, names_len, ms, max_kernels, count);
}
int drl_r2d2_last_step_ms(drl_r2d2* h, float* ms) {
  DRL_ENTER(h);
  return last_step_ms(h, ms);
}
int drl_r2d2_stream(drl_r2d2* h, void** stream) {
  DRL_ENTER(h);
  if (!stream) { set_error("null argument"); return DRL_ERR_INVALID; }
  *stream = h->compute;
  return DRL_OK;
}
int drl_r2d2_launches_per_step(const drl_r2d2* h, int32_t* n) {
  DRL_ENTER(h);
  if (!n) { set_error("null argument"); return DRL_ERR_INVALID; }
  *n = h->launches;
  return DRL_OK;
}

}  // extern "C"
