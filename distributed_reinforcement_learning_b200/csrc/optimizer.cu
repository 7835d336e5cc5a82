// optimizer.cu -- the optimizers of the learners: IMPALA's RMSProp first, TF1 Adam (Ape-X, A3C, R2D2) below.
// RMSProp is the tail of the IMPALA train op (agent/impala.py:95-100) with TF 1.14 semantics:
//   lr    = polynomial_decay(start, global_step, decay_steps, end)  (power 1, evaluated in float32)
//   g    <- g * clip * min(1/||g||_2, 1/clip)                        (tf.clip_by_global_norm over ALL params)
//   ms   <- ms + (1 - 0.99) (g^2 - ms)     (RMSProp slot initialised to ONES)
//   w    <- w - lr * g / sqrt(ms + 0.1)     (epsilon INSIDE the sqrt, momentum 0, not centred; evaluated as
//           lr * g * rsqrt(ms + 0.1) like TF's Eigen kernel -- rsqrt.approx is within 2 ulp and avoids the IEEE-division
//           subroutine, which made this HBM-bound kernel ALU-bound)
//   global_step += 1
// Two launches over the flat padded vectors: (1) partial sums of squares (+ lr, step), (2) every
// block re-reduces the partials in a fixed order (deterministic) and applies the update.
// HBM traffic: read g twice (second time from L2), read+write w and ms: ~5 x 16.6 MB.
#include "kernels.h"
#include "peer_sync.cuh"

namespace drl {

__global__ void __launch_bounds__(256) sqnorm_partial_kernel(OptState o) {
  pdl_prologue();
  __shared__ float red[8];
  const int64_t n4 = o.n / 4;
  const float4* g4 = reinterpret_cast<const float4*>(o.grads);
  float acc = 0.f;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (int64_t)gridDim.x * blockDim.x) {
    const float4 v = g4[i];
    acc = fmaf(v.x, v.x, acc); acc = fmaf(v.y, v.y, acc); acc = fmaf(v.z, v.z, acc); acc = fmaf(v.w, v.w, acc);
  }
  acc = warp_sum(acc);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < 8; ++i) s += red[i];
    o.norm_partials[blockIdx.x] = s;
    if (blockIdx.x == 0) {
      // tf.train.polynomial_decay in float32 (agent/impala.py:96); uses the pre-increment step.
      const long long step = *o.step;
      const float decay = (float)o.learning_frame;
      const float gs = fminf((float)step, decay);
      const float p = gs / decay;
      *o.lr_cur = (o.start_lr - o.end_lr) * (1.0f - p) + o.end_lr;
      *o.step = step + 1;                                                  // agent/impala.py:100
    }
  }
}

__global__ void __launch_bounds__(256) rmsprop_apply_kernel(OptState o) {
  pdl_prologue();
  __shared__ float red[8];
  __shared__ float s_scale;
  // data-parallel: barrier 1 of the peer exchange -- every peer has delivered its slice of the summed gradients and
  // its partial norms into this rank's buffers (peer.cu)
  // A failed barrier (time-out, now or in an earlier step) makes the update a no-op: parameters, slots and the
  // step's scalars keep their values and the host reports the error (peer_sync.cuh).
  if (o.wait_flags) {
    const PeerErr perr{o.wait_err, o.wait_err_host, o.wait_timeout_ns};
    for (int part = 0; part < o.wait_parts; ++part)
      if (!wait_peers(o.wait_flags, 2 * part + 1, o.wait_world, o.wait_epoch[4 * part + 1], perr)) return;
  }
  float acc = 0.f;
  for (int i = threadIdx.x; i < o.npart; i += blockDim.x) acc += o.norm_partials[i];
  acc = warp_sum(acc);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < 8; ++i) s += red[i];
    const float norm = sqrtf(s);
    s_scale = o.clip_norm * fminf(1.0f / norm, 1.0f / o.clip_norm);        // tf.clip_by_global_norm
    if (blockIdx.x == 0) {
      const float pi = o.loss_sums[0], bl = o.loss_sums[1], en = o.loss_sums[2];
      o.out[0] = pi; o.out[1] = bl; o.out[2] = en; o.out[3] = *o.lr_cur; o.out[4] = norm;
      o.out[5] = pi + bl * o.baseline_coef + en * o.entropy_coef;          // agent/impala.py:93
      const long long st = *o.step;
      o.out[6] = __int_as_float((int)(st & 0xffffffffll));
      o.out[7] = __int_as_float((int)(st >> 32));
    }
  }
  __syncthreads();
  const float scale = s_scale;
  const float lr = *o.lr_cur;
  const int64_t n4 = o.n / 4;
  const float4* g4 = reinterpret_cast<const float4*>(o.grads);
  float4* w4 = reinterpret_cast<float4*>(o.params);
  float4* m4 = reinterpret_cast<float4*>(o.ms);
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (int64_t)gridDim.x * blockDim.x) {
    const float4 g = g4[i];
    float4 m = m4[i], w = w4[i];
    float gg;
    gg = g.x * scale; m.x += (gg * gg - m.x) * (1.0f - 0.99f); w.x -= lr * gg * rsqrtf(m.x + 0.1f);
    gg = g.y * scale; m.y += (gg * gg - m.y) * (1.0f - 0.99f); w.y -= lr * gg * rsqrtf(m.y + 0.1f);
    gg = g.z * scale; m.z += (gg * gg - m.z) * (1.0f - 0.99f); w.z -= lr * gg * rsqrtf(m.z + 0.1f);
    gg = g.w * scale; m.w += (gg * gg - m.w) * (1.0f - 0.99f); w.w -= lr * gg * rsqrtf(m.w + 0.1f);
    m4[i] = m; w4[i] = w;
  }
}

int optimizer_update_only(cudaStream_t s, const OptState& o) {
  DRL_CUDA_CHECK((launch_k(rmsprop_apply_kernel, o.nblk, 256, 0, s, o)));
  return DRL_OK;
}

int optimizer_apply(cudaStream_t s, const OptState& o) {
  DRL_CUDA_CHECK((launch_k(sqnorm_partial_kernel, o.nblk, 256, 0, s, o)));
  DRL_CUDA_CHECK((launch_k(rmsprop_apply_kernel, o.nblk, 256, 0, s, o)));
  return DRL_OK;
}

// ------------------------------------------------------------------------------------------
// TF1 Adam: the tail of the Ape-X / A3C train op (agent/apex.py:70-75) and of the R2D2 one, with TF 1.14 semantics:
//   lr    = polynomial_decay(start, global_step, decay_steps, end)      (float32, pre-increment step)
//   g    <- g * clip * min(1/||g||, 1/clip)                              (clip_by_global_norm over the main variables;
//                                                                         the target variables have gradient None)
//   alpha = lr * sqrt(1 - beta2_power) / (1 - beta1_power)               (ApplyAdam, float32)
//   m    += (g - m)(1 - beta1) ; v += (g^2 - v)(1 - beta2) ; w -= m * alpha / (sqrt(v) + eps)
//   beta powers *= beta ; global_step += 1
// Two launches: (1) partial squared norms + the scalars, (2) every block re-reduces the partials in fixed order.
// ------------------------------------------------------------------------------------------
constexpr float kAdamEps = 1e-8f;

__global__ void __launch_bounds__(256) adam_prepare_kernel(AdamState o) {
  pdl_prologue();
  __shared__ float red[8];
  const int64_t n4 = o.n / 4;
  const float4* g4 = reinterpret_cast<const float4*>(o.grads);
  float acc = 0.f;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (int64_t)gridDim.x * blockDim.x) {
    const float4 v = g4[i];
    acc = fmaf(v.x, v.x, acc); acc = fmaf(v.y, v.y, acc); acc = fmaf(v.z, v.z, acc); acc = fmaf(v.w, v.w, acc);
  }
  acc = warp_sum(acc);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < 8; ++i) s += red[i];
    o.norm_partials[blockIdx.x] = s;
    if (blockIdx.x == 0) {
      const long long step = *o.step;
      const float decay = (float)o.learning_frame;
      const float gs = fminf((float)step, decay);
      const float p = gs / decay;
      const float lr = (o.start_lr - o.end_lr) * (1.0f - p) + o.end_lr;
      const float b1 = *o.b1p, b2 = *o.b2p;
      *o.lr_cur = lr;
      *o.alpha = lr * sqrtf(1.0f - b2) / (1.0f - b1);
      *o.b1p = b1 * kAdamBeta1;
      *o.b2p = b2 * kAdamBeta2;
      *o.step = step + 1;
    }
  }
}

__global__ void __launch_bounds__(256) adam_apply_kernel(AdamState o) {
  pdl_prologue();
  __shared__ float red[8];
  __shared__ float s_scale;
  float acc = 0.f;
  for (int i = threadIdx.x; i < o.nblk; i += blockDim.x) acc += o.norm_partials[i];
  acc = warp_sum(acc);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < 8; ++i) s += red[i];
    const float norm = sqrtf(s) * o.grad_scale;
    s_scale = ((o.clip_norm > 0.f) ? o.clip_norm * fminf(1.0f / norm, 1.0f / o.clip_norm) : 1.0f) * o.grad_scale;
    if (blockIdx.x == 0) {
      o.out[0] = o.loss[0] * o.grad_scale; o.out[1] = *o.lr_cur; o.out[2] = norm;
      o.out[3] = o.loss[1] * o.grad_scale; o.out[4] = o.loss[2] * o.grad_scale;          // A3C: baseline loss, entropy (zero for the DQN learners)
      const long long st = *o.step;
      o.out[6] = __int_as_float((int)(st & 0xffffffffll));
      o.out[7] = __int_as_float((int)(st >> 32));
    }
  }
  __syncthreads();
  const float scale = s_scale;
  const float alpha = *o.alpha;
  const int64_t n4 = o.n / 4;
  const float4* g4 = reinterpret_cast<const float4*>(o.grads);
  float4* w4 = reinterpret_cast<float4*>(o.params);
  float4* m4 = reinterpret_cast<float4*>(o.m);
  float4* v4 = reinterpret_cast<float4*>(o.v);
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (int64_t)gridDim.x * blockDim.x) {
    const float4 g = g4[i];
    float4 m = m4[i], v = v4[i], w = w4[i];
    float gg;
    gg = g.x * scale; m.x += (gg - m.x) * (1.0f - kAdamBeta1); v.x += (gg * gg - v.x) * (1.0f - kAdamBeta2); w.x -= (m.x * alpha) / (sqrtf(v.x) + kAdamEps);
    gg = g.y * scale; m.y += (gg - m.y) * (1.0f - kAdamBeta1); v.y += (gg * gg - v.y) * (1.0f - kAdamBeta2); w.y -= (m.y * alpha) / (sqrtf(v.y) + kAdamEps);
    gg = g.z * scale; m.z += (gg - m.z) * (1.0f - kAdamBeta1); v.z += (gg * gg - v.z) * (1.0f - kAdamBeta2); w.z -= (m.z * alpha) / (sqrtf(v.z) + kAdamEps);
    gg = g.w * scale; m.w += (gg - m.w) * (1.0f - kAdamBeta1); v.w += (gg * gg - v.w) * (1.0f - kAdamBeta2); w.w -= (m.w * alpha) / (sqrtf(v.w) + kAdamEps);
    m4[i] = m; v4[i] = v; w4[i] = w;
  }
}

int adam_step(cudaStream_t s, const AdamState& o) {
  DRL_CUDA_CHECK((launch_k(adam_prepare_kernel, o.nblk, 256, 0, s, o)));
  DRL_CUDA_CHECK((launch_k(adam_apply_kernel, o.nblk, 256, 0, s, o)));
  return DRL_OK;
}

}  // namespace drl
