// layers.cu -- forward and backward of the IMPALA actor-critic (model/impala_actor_critic.py:33-42)
// over M = B*T independent rows (the LSTM is a single step from fed state, :18-25 / :73-82, so
// time is embarrassingly parallel; only T distinct forwards exist, SURVEY.md section 0.3).
// Every dense contraction is one launch of a gather-GEMM: the FP32-FFMA core (gemm_simt.cuh, math
// mode 1) or the tcgen05 3xTF32 tensor-core core (gemm_umma.cuh, math mode 2) -- same loaders and
// epilogues.  The small head layers (M x 256 x 256) always use the FFMA core.
#include <stdlib.h>

#include "layer_defs.cuh"

namespace drl {

void ParamLayout::init(int num_action) {
  A = num_action;
  place({8 * 8 * 4 * 32, 32, 4 * 4 * 32 * 64, 64, 3 * 3 * 64 * 64, 64,
         (int64_t)A * 256, 256, 256 * 256, 256,
         (int64_t)Geo::XK * Geo::G4, Geo::G4,
         256 * 256, 256, 256 * 256, 256, 256 * (int64_t)A, A,
         256 * 256, 256, 256 * 256, 256, 256, 1},
        {&conv1_w, &conv1_b, &conv2_w, &conv2_b, &conv3_w, &conv3_b, &emb1_w, &emb1_b, &emb2_w, &emb2_b, &lstm_w,
         &lstm_b, &actor1_w, &actor1_b, &actor2_w, &actor2_b, &actor3_w, &actor3_b, &critic1_w, &critic1_b, &critic2_w,
         &critic2_b, &critic3_w, &critic3_b});
}

static int g_fwd_launches = 0, g_bwd_launches = 0;
int forward_launch_count() { return g_fwd_launches; }
int backward_launch_count() { return g_bwd_launches; }


size_t wgrad_partial_floats(int B, int T) {
  const int Mb = B * (T - 2);
  size_t mx = 0;
  for (int mode : {1, 2, 3, 5}) {
    mx = std::max(mx, (size_t)plan_conv1_wgrad(Mb, mode).splits * 257 * 32);
    mx = std::max(mx, (size_t)plan_conv2_wgrad(Mb, mode).splits * 513 * 64);
    mx = std::max(mx, (size_t)plan_conv3_wgrad(Mb, mode).splits * 577 * 64);
  }
  return std::max(mx, (size_t)16 * 32 * 256);   // also the scratch of emb_backward (kEmbChunks * A * 256)
}

size_t lstm_image_bytes(int which, int M, int Mb) {
  (void)M;
  return which == 1 ? operand_image16_bytes<128>(Geo::XK, Mb)     // x^T  (A of lstm_wgrad)
                    : operand_image16_bytes<256>(Geo::G4, Mb);    // dz^T (B of lstm_wgrad)
}

void weight_image_sizes(size_t (&b)[WeightImages::kCount]) {
  b[0] = weight_image_bytes<32>(32, 256);
  b[1] = weight_image_bytes<64>(64, 512);
  b[2] = weight_image_bytes<64>(64, 576);
  b[3] = weight_image_bytes<256>(Geo::G4, Geo::XK);
  b[4] = weight_image_bytes<128>(Geo::FLAT + Geo::EMB, Geo::G4);
  b[5] = weight_image_bytes<256>(576, 64);
  b[6] = weight_image_bytes<256>(512, 64);
}

// Refresh the weight images (4 launches on the side stream + 1 for the two conv-forward images; ~60 MB written).
// Must run after every parameter change.  Image 0 (conv1) is unused: conv1 is the first kernel of the step and its
// weight tile is 1/5 of a stage.
// math mode 5: the same seven images in the 16-bit K-major form (gemm_umma16.cuh); they fit into the same buffers
int net_retile16(cudaStream_t s_rest, const ParamLayout& pl, const float* P, const WeightImages& wi) {
  prof_mark(s_rest, "weight_retile");
  DRL_TRY((launch_retile_b16<256, Fmt16>(s_rest, PlainB{P + pl.lstm_w, Geo::G4, 0}, Geo::G4, Geo::XK, wi.img[3])));
  DRL_TRY((launch_retile_b16<128, Fmt16>(s_rest, PlainBT{P + pl.lstm_w, Geo::G4, 0}, Geo::FLAT + Geo::EMB, Geo::G4, wi.img[4])));
  DRL_TRY((launch_retile_b16<256, Fmt16>(s_rest, PlainBT{P + pl.conv3_w, 64, 0}, 576, 64, wi.img[5])));
  DRL_TRY((launch_retile_b16<256, Fmt16>(s_rest, PlainBT{P + pl.conv2_w, 64, 0}, 512, 64, wi.img[6])));
  return DRL_OK;
}

int net_retile(cudaStream_t, cudaStream_t s_rest, const ParamLayout& pl, const float* P, const WeightImages& wi) {
  prof_mark(s_rest, "weight_retile");
  DRL_TRY((launch_retile_b<256>(s_rest, PlainB{P + pl.lstm_w, Geo::G4, 0}, Geo::G4, Geo::XK, wi.img[3])));
  DRL_TRY((launch_retile_b<128>(s_rest, PlainBT{P + pl.lstm_w, Geo::G4, 0}, Geo::FLAT + Geo::EMB, Geo::G4, wi.img[4])));
  DRL_TRY((launch_retile_b<256>(s_rest, PlainBT{P + pl.conv3_w, 64, 0}, 576, 64, wi.img[5])));
  DRL_TRY((launch_retile_b<256>(s_rest, PlainBT{P + pl.conv2_w, 64, 0}, 512, 64, wi.img[6])));
  return DRL_OK;
}

int net_forward(const Streams& st, const ParamLayout& pl, const float* P, const WeightImages& wi, const Inputs& in,
                const Acts& act, int B, int T, int mode, bool retile) {
  const int M = B * T;
  const RowMap map{B, T};
  int n = 0, nsplit = 4;
  const bool tma = mode == 4;
  if (mode == 4) mode = 2;
  cudaStream_t s = st.main;
  const cudaStream_t side = st.par ? st.side : st.main;
  // action embedding table (:12-16): only A distinct inputs exist; depends on parameters only -> side stream
  DRL_TRY(fork_to_side(st, 0));
  s = side;
  // weight images of this step's parameters, all on the side stream: the conv2/conv3 forward ones first (main waits
  // for them behind conv1), the LSTM / dgrad ones behind the embedding table (joined before lstm_fwd)
  const bool m16 = mode == 5;
  bool c3_event = false;   // conv3's weight image has its own event (math mode 5)
  static const bool heads_tc = !(getenv("DRL_B200_HEADS_TC") && atoi(getenv("DRL_B200_HEADS_TC")) == 0);   // head layers on tcgen05 (0: FFMA)
  // math mode 5: conv1 is the frame-resident TMA kernel (conv1_tma.cuh), which builds its 32 KB weight image itself;
  // DRL_B200_CONV1_GATHER=1 keeps the generic gather-GEMM, DRL_B200_C1_WIMG=1 the pre-tiled image (one more kernel in
  // front of the step's first kernel)
  static const bool c1_gather = getenv("DRL_B200_CONV1_GATHER") != nullptr;
  static const bool c1_wimg = c1_gather || getenv("DRL_B200_C1_WIMG") != nullptr;
  if (retile && m16) {
    prof_mark(s, "weight_retile");
    if (c1_wimg) {
      DRL_TRY((launch_retile_b16<32, FmtC1>(s, PlainB{P + pl.conv1_w, 32, 0}, 32, 256, wi.img[0])));
      if (st.par) DRL_CUDA_CHECK(cudaEventRecord(st.ev[2], side));        // conv1 waits for its (tiny) image
      ++n;
    }
    DRL_TRY((launch_retile_b16<64, Fmt16>(s, PlainB{P + pl.conv2_w, 64, 0}, 64, 512, wi.img[1])));
    if (st.par) DRL_CUDA_CHECK(cudaEventRecord(st.ev[7], side));          // conv2 image (main waits behind conv1)
    DRL_TRY((launch_retile_b16<64, Fmt16>(s, PlainB{P + pl.conv3_w, 64, 0}, 64, 576, wi.img[2])));
    if (st.par) DRL_CUDA_CHECK(cudaEventRecord(st.ev[4], side));          // conv3 image (main waits behind conv2)
    c3_event = st.par;
    n += 2;
  } else if (retile && mode >= 2) {
    prof_mark(s, "weight_retile");
    DRL_TRY((launch_retile_b<64>(s, PlainB{P + pl.conv2_w, 64, 0}, 64, 512, wi.img[1])));
    DRL_TRY((launch_retile_b<64>(s, PlainB{P + pl.conv3_w, 64, 0}, 64, 576, wi.img[2])));
    n += 2;
    if (st.par) DRL_CUDA_CHECK(cudaEventRecord(st.ev[7], side));
  }
  KERNEL("emb_fwd",
         emb_forward(s, P + pl.emb1_w, P + pl.emb1_b, P + pl.emb2_w, P + pl.emb2_b, act.e1, act.table, pl.A), 1);
  s = st.main;
  bool late_images = false;   // side still carries the images only the backward pass reads when lstm_fwd is enqueued
  if (retile && mode >= 2) {
    if (m16 && st.par) {
      // the LSTM forward image first; lstm_fwd waits for it (and the embedding table) only -- the three images of the
      // backward pass (LSTM dgrad, two dCol) are joined at the end of the forward pass, long after they are done
      prof_mark(side, "weight_retile");
      DRL_TRY((launch_retile_b16<256, Fmt16>(side, PlainB{P + pl.lstm_w, Geo::G4, 0}, Geo::G4, Geo::XK, wi.img[3])));
      DRL_CUDA_CHECK(cudaEventRecord(st.ev[1], side));
      late_images = true;   // LSTM dgrad + two dCol images: behind lstm_gates_fwd, in the shadow of the small head kernels
    } else if (m16) {
      DRL_TRY(net_retile16(side, pl, P, wi));
    } else {
      DRL_TRY(net_retile(st.main, side, pl, P, wi));
    }
    n += 4;
  }
  if (retile && m16 && st.par && c1_wimg) {
    DRL_CUDA_CHECK(cudaStreamWaitEvent(st.main, st.ev[2], 0));
    pdl_break(st.main);
  }
  // conv1: u8 frames -> a1 [M,20,20,32]   (attention_CNN, model/impala_actor_critic.py:6)
  {
    Conv1A al{in.frames, map};
    PlainB bl{P + pl.conv1_w, 32, 0};
    EpConv1 ep{act.a1, 32, P + pl.conv1_b, tma ? act.a1_lo : nullptr};
    if (m16 && !c1_gather) {
      prof_mark(s, "conv1_fwd");
      DRL_TRY(launch_conv1_fwd_tma(s, in.frames, M, map, wi.img[0], c1_wimg ? nullptr : P + pl.conv1_w, ep));
      ++n;
    } else if (m16) {
      PretiledB<PlainB> blp{wi.img[0], 256 / 64};
      GEMM16("conv1_fwd", X32L, al, blp, ep, M * 400, 32, 256, 1, 256, 0);
    } else {
      GEMM("conv1_fwd", CfgN32, U32, al, bl, ep, M * 400, 32, 256, 1, 256, 0);
    }
  }
  if (retile && mode >= 2 && st.par) {
    DRL_CUDA_CHECK(cudaStreamWaitEvent(st.main, st.ev[7], 0));
    pdl_break(st.main);
  }
  // conv2 -> a2 [M,9,9,64]   (:7)
  if (tma) {
    EpBiasAct<true, true> ep{act.a2, 64, 0, P + pl.conv2_b, 0, 1.0f, act.a2_lo};
    KERNEL("conv2_fwd", (launch_conv_fwd_tma<Conv2Tma>(s, act.a1, (size_t)(act.a1_lo - act.a1), M, wi.img[1], ep)), 1);
  } else {
    Conv2A al{act.a1, map};
    PlainB bl{P + pl.conv2_w, 64, 0};
    PretiledB<PlainB> blp{wi.img[1], m16 ? 512 / 64 : 512 / 32};
    EpBiasAct<true, true> ep{act.a2, 64, 0, P + pl.conv2_b, 0, 1.0f};
    static const int c2f = getenv("DRL_B200_C2F") ? atoi(getenv("DRL_B200_C2F")) : 2;
    if (m16 && c2f == 2) GEMM16("conv2_fwd", X64L8x2, al, blp, ep, M * 81, 64, 512, 1, 512, 0);
    else if (m16) GEMM16("conv2_fwd", X64L, al, blp, ep, M * 81, 64, 512, 1, 512, 0);
    else GEMM_W("conv2_fwd", CfgBig, U64L, al, bl, blp, ep, M * 81, 64, 512, 1, 512, 0);
  }
  if (c3_event) {
    DRL_CUDA_CHECK(cudaStreamWaitEvent(st.main, st.ev[4], 0));
    pdl_break(st.main);
  }
  // conv3 -> a3 [M,7,7,64] = flatten HWC [M,3136]   (:8-10)
  if (tma) {
    EpBiasAct<true, true> ep{act.a3, 64, 0, P + pl.conv3_b, 0, 1.0f};
    KERNEL("conv3_fwd", (launch_conv_fwd_tma<Conv3Tma>(s, act.a2, (size_t)(act.a2_lo - act.a2), M, wi.img[2], ep)), 1);
  } else {
    Conv3A al{act.a2, map};
    PlainB bl{P + pl.conv3_w, 64, 0};
    PretiledB<PlainB> blp{wi.img[2], m16 ? 576 / 64 : 576 / 32};
    EpBiasAct<true, true> ep{act.a3, 64, 0, P + pl.conv3_b, 0, 1.0f};
    static const int c3f = getenv("DRL_B200_C2F") ? atoi(getenv("DRL_B200_C2F")) : 2;
    if (m16 && c3f == 2) GEMM16("conv3_fwd", X64L8x2, al, blp, ep, M * 49, 64, 576, 1, 576, 0);
    else if (m16) GEMM16("conv3_fwd", X64L, al, blp, ep, M * 49, 64, 576, 1, 576, 0);
    else GEMM_W("conv3_fwd", CfgBig, U64L, al, bl, blp, ep, M * 49, 64, 576, 1, 576, 0);
  }
  if (late_images) {
    DRL_CUDA_CHECK(cudaStreamWaitEvent(st.main, st.ev[1], 0));
    pdl_break(st.main);
  } else {
    DRL_TRY(join_from_side(st, 1));
  }
  // LSTM pre-activation z = [a3 | emb | h0] W  (split-K partial sums; bias added in the gate kernel) (:18-25)
  {
    LstmA al{act.a3, act.table, in.pa, in.h0, map};
    PlainB bl{P + pl.lstm_w, Geo::G4, 0};
    EpRaw<false> ep{act.zpart, Geo::G4, (size_t)M * Geo::G4, 1.0f, 0, Geo::G4};
    // FFMA: 4 splits of 57 x 16.  tcgen05: 128 x 256 tiles -> 5 x 4 output tiles x 7 splits of 17 x 32 = 140 CTAs (one wave)
    nsplit = (mode >= 2) ? 7 : 4;
    const int kchunk = m16 ? 576 : (mode >= 2) ? 544 : Geo::XK / 4;      // 16-bit: 9 K tiles of 64 per split
    PretiledB<PlainB> blp{wi.img[3], m16 ? Geo::XK / 64 : Geo::XK / 32};
    if (m16) GEMM16("lstm_fwd", X256L, al, blp, ep, M, Geo::G4, Geo::XK, nsplit, kchunk, kchunk);
    else GEMM_W("lstm_fwd", CfgMid, U256L, al, bl, blp, ep, M, Geo::G4, Geo::XK, nsplit, kchunk, kchunk);
  }
  KERNEL("lstm_gates_fwd",
         lstm_gates_forward(s, act.zpart, nsplit, P + pl.lstm_b, in.c0, act.gates, act.c1, act.tc1, act.h1, M, B,
                            T), 1);
  // heads (fully_connected, :27-30,40-41): z = 0 actor, z = 1 critic
  const size_t head_stride = (size_t)(pl.critic1_w - pl.actor1_w);
  if (late_images) {
    // the three images only the backward pass reads (~25 us of memory-bound work) would compete with conv2_fwd / conv3_fwd
    // for the SMs if launched with the others; the head layers that follow leave most of the GPU idle
    DRL_TRY(fork_to_side(st, 3));
    DRL_TRY((launch_retile_b16<128, Fmt16>(side, PlainBT{P + pl.lstm_w, Geo::G4, 0}, Geo::FLAT + Geo::EMB, Geo::G4, wi.img[4])));
    DRL_TRY((launch_retile_b16<256, Fmt16>(side, PlainBT{P + pl.conv3_w, 64, 0}, 576, 64, wi.img[5])));
    DRL_TRY((launch_retile_b16<256, Fmt16>(side, PlainBT{P + pl.conv2_w, 64, 0}, 512, 64, wi.img[6])));
  }
  {
    PlainA al{act.h1, Geo::L, 0};
    PlainB bl{P + pl.actor1_w, Geo::HID, head_stride};
    EpBiasAct<true, true> ep{act.hid1, Geo::HID, (size_t)M * Geo::HID, P + pl.actor1_b, head_stride, 1.0f};
    if (m16 && heads_tc) GEMM16("heads_l1_fwd", XH, al, bl, ep, M, Geo::HID, Geo::L, 2, Geo::L, 0);
    else GEMM_FFMA("heads_l1_fwd", CfgSmall, al, bl, ep, M, Geo::HID, Geo::L, 2, Geo::L, 0);
  }
  {
    PlainA al{act.hid1, Geo::HID, (size_t)M * Geo::HID};
    PlainB bl{P + pl.actor2_w, Geo::HID, head_stride};
    EpBiasAct<true, true> ep{act.hid2, Geo::HID, (size_t)M * Geo::HID, P + pl.actor2_b, head_stride, 1.0f};
    if (m16 && heads_tc) GEMM16("heads_l2_fwd", XH, al, bl, ep, M, Geo::HID, Geo::HID, 2, Geo::HID, 0);
    else GEMM_FFMA("heads_l2_fwd", CfgSmall, al, bl, ep, M, Geo::HID, Geo::HID, 2, Geo::HID, 0);
  }
  KERNEL("heads_out_fwd",
         heads_out_forward(s, act.hid2, act.hid2 + (size_t)M * Geo::HID, P + pl.actor3_w, P + pl.actor3_b,
                           P + pl.critic3_w, P + pl.critic3_b, act.logits, act.policy, act.value, M, pl.A), 1);
  if (late_images) DRL_TRY(join_from_side(st, 1));   // the backward images: done ~70 us ago, keeps net_forward self-contained
  g_fwd_launches = n;
  return DRL_OK;
}

int net_backward(const Streams& st, const ParamLayout& pl, const float* P, const WeightImages& wi, float* G,
                 const Inputs& in, const Acts& act, const Bwd& bw, int B, int T, int mode) {
  PdlRegionOff pdl_region;   // DRL_B200_PDL=2: no early launches while the side stream competes for the same SMs
  if (mode == 4) mode = 2;
  const bool m16 = mode == 5;
  static const bool heads_tc = !(getenv("DRL_B200_HEADS_TC") && atoi(getenv("DRL_B200_HEADS_TC")) == 0);   // head layers on tcgen05 (0: FFMA)
  cudaStream_t s = st.main;
  const cudaStream_t side = st.par ? st.side : st.main;
  const int M = B * T;
  const int Mb = B * (T - 2);   // rows t <= T-3 are the contiguous prefix (time-major)
  const RowMap map{B, T};
  const size_t head_stride = (size_t)(pl.critic1_w - pl.actor1_w);
  const int A = pl.A;
  int n = 0;

  // ---- heads -------------------------------------------------------------------------------
  KERNEL("heads_out_bwd",
         heads_out_backward(s, bw.dlogits, bw.dv, P + pl.actor3_w, P + pl.critic3_w, act.hid2,
                            act.hid2 + (size_t)M * Geo::HID, bw.dhid2, bw.dhid2 + (size_t)Mb * Geo::HID, Mb, A), 1);
  const bool lbulk = m16 && act.img_xt != nullptr && bw.img_dzt != nullptr && M <= act.img_rows;   // bulk-fed lstm_wgrad
  if (lbulk) {
    // x^T as an operand image (A of lstm_wgrad): depends on the forward pass only -> side stream, in the shadow of the
    // small head kernels
    DRL_TRY(fork_to_side(st, 0));
    prof_mark(side, "lstm_xt_image");
    DRL_TRY((launch_retile_t16<128, Fmt16>(side, LstmAT{act.a3, act.table, in.pa, in.h0, map}, Geo::XK, Mb, act.img_xt)));
    ++n;
  }
  // dlogits / dv / dhid2 are ready: three weight gradients can start beside the chain (on the second side lane if any)
  const bool lane2 = st.par && st.side2 != nullptr;
  const cudaStream_t small = lane2 ? st.side2 : side;
  if (lane2) DRL_TRY(fork_to_side2(st, 0));
  else DRL_TRY(fork_to_side(st, 0));
  s = small;
  {  // d actor3 [256(+1), A]
    PlainAT al{act.hid2, Geo::HID, 0};
    PlainB bl{bw.dlogits, 32, 0};
    EpRaw<true> ep{G + pl.actor3_w, A, 0, 1.0f, Geo::HID, A};
    GEMM_FFMA_KS("actor3_wgrad", CfgSmall, 3, al, bl, ep, Geo::HID, 32, Mb, 1, Mb, 0);
  }
  {  // d critic3 [256(+1), 1]
    PlainAT al{act.hid2 + (size_t)M * Geo::HID, Geo::HID, 0};
    PlainB bl{bw.dv, 32, 0};
    EpRaw<true> ep{G + pl.critic3_w, 1, 0, 1.0f, Geo::HID, 1};
    GEMM_FFMA_KS("critic3_wgrad", CfgSmall, 3, al, bl, ep, Geo::HID, 32, Mb, 1, Mb, 0);
  }
  {  // d {actor2, critic2} = hid1^T dhid2
    PlainAT al{act.hid1, Geo::HID, (size_t)M * Geo::HID};
    PlainB bl{bw.dhid2, Geo::HID, (size_t)Mb * Geo::HID};
    EpRaw<true> ep{G + pl.actor2_w, Geo::HID, head_stride, 1.0f, Geo::HID, Geo::HID};
    GEMM_FFMA_KS("heads_l2_wgrad", CfgSmall, 3, al, bl, ep, Geo::HID, Geo::HID, Mb, 2, Mb, 0);
  }
  s = st.main;
  {  // dhid1 = dhid2 W2^T * relu'(hid1)
    PlainA al{bw.dhid2, Geo::HID, (size_t)Mb * Geo::HID};
    PlainBT bl{P + pl.actor2_w, Geo::HID, head_stride};
    EpReluMask ep{bw.dhid1, act.hid1, Geo::HID, (size_t)Mb * Geo::HID, (size_t)M * Geo::HID};
    if (m16 && heads_tc) GEMM16("heads_l2_dgrad", XH, al, bl, ep, Mb, Geo::HID, Geo::HID, 2, Geo::HID, 0);
    else GEMM_FFMA_KS("heads_l2_dgrad", CfgSmall, 4, al, bl, ep, Mb, Geo::HID, Geo::HID, 2, Geo::HID, 0);
  }
  if (lane2) DRL_TRY(fork_to_side2(st, 1));
  else DRL_TRY(fork_to_side(st, 2));
  s = small;
  {  // d {actor1, critic1} = h1^T dhid1
    PlainAT al{act.h1, Geo::L, 0};
    PlainB bl{bw.dhid1, Geo::HID, (size_t)Mb * Geo::HID};
    EpRaw<true> ep{G + pl.actor1_w, Geo::HID, head_stride, 1.0f, Geo::L, Geo::HID};
    GEMM_FFMA_KS("heads_l1_wgrad", CfgSmall, 3, al, bl, ep, Geo::L, Geo::HID, Mb, 2, Mb, 0);
  }
  s = st.main;
  {  // dh1 contributions (actor, critic) = dhid1 W1^T ; summed in the gate kernel
    PlainA al{bw.dhid1, Geo::HID, (size_t)Mb * Geo::HID};
    PlainBT bl{P + pl.actor1_w, Geo::HID, head_stride};
    EpRaw<false> ep{bw.dh_part, Geo::L, (size_t)Mb * Geo::L, 1.0f, 0, Geo::L};
    if (m16 && heads_tc) GEMM16("heads_l1_dgrad", XH, al, bl, ep, Mb, Geo::L, Geo::HID, 2, Geo::HID, 0);
    else GEMM_FFMA_KS("heads_l1_dgrad", CfgSmall, 4, al, bl, ep, Mb, Geo::L, Geo::HID, 2, Geo::HID, 0);
  }
  // ---- LSTM cell ---------------------------------------------------------------------------
  KERNEL("lstm_gates_bwd",
         lstm_gates_backward(s, bw.dh_part, (size_t)Mb * Geo::L, act.gates, act.tc1, in.c0, bw.dz, Mb, B, T), 1);
  DRL_TRY(fork_to_side(st, 3));
  s = side;
  {  // d lstm kernel [3648(+1), 1024] = x^T dz ; bias gradient = column sums of dz
    LstmAT al{act.a3, act.table, in.pa, in.h0, map};
    PlainB bl{bw.dz, Geo::G4, 0};
    EpRaw<true> ep{G + pl.lstm_w, Geo::G4, 0, 1.0f, Geo::XK, Geo::G4};
    if (lbulk) {
      const int ktm = cdiv(Mb, 64);
      prof_mark(s, "lstm_dzt_image");
      DRL_TRY((launch_retile_t16<256, Fmt16>(s, bl, Geo::G4, Mb, bw.img_dzt)));
      // bias gradient = column sums of dz (row XK of [w; b]), fixed order
      DRL_TRY(splitk_reduce(s, bw.dz, Geo::G4, Mb, G + pl.lstm_w + (size_t)Geo::XK * Geo::G4, Geo::G4));
      prof_mark(s, "lstm_wgrad");
      EpRaw<false> epw{G + pl.lstm_w, Geo::G4, 0, 1.0f, Geo::XK, Geo::G4};
      DRL_TRY((launch_gemm_bulk16<BK256>(s, ImageOp{act.img_xt, ktm}, ImageOp{bw.img_dzt, ktm}, epw, Geo::XK, Geo::G4, Mb,
                                         1, Mb, 0)));
      n += 3;
    } else if (m16) GEMM16("lstm_wgrad", X256W, al, bl, ep, Geo::XK, Geo::G4, Mb, 1, Mb, 0);
    else GEMM("lstm_wgrad", CfgBig, U256, al, bl, ep, Geo::XK, Geo::G4, Mb, 1, Mb, 0);   // 29 x 4 = 116 CTAs: one wave
    // the head gradients (earlier on this stream, or on the second lane: joined here) and the LSTM gradient are now
    // in the bucket: [lstm_w .. end)
    if (lane2) DRL_TRY(join_side2_into(st, 2, side));
    if (st.par && st.ev_lstm_grads) DRL_CUDA_CHECK(cudaEventRecord(st.ev_lstm_grads, side));
  }
  s = st.main;
  {  // d[a3 | emb] = dz W[:3392]^T  (h0, c0 are fed data: no gradient, agent/impala.py:38-39)
    PlainA al{bw.dz, Geo::G4, 0};
    PlainBT bl{P + pl.lstm_w, Geo::G4, 0};
    EpLstmDx ep{bw.da3, act.a3, bw.du};
    PretiledB<PlainBT> blp{wi.img[4], m16 ? Geo::G4 / 64 : Geo::G4 / 32};
    if (m16) GEMM16("lstm_dgrad", X128D, al, blp, ep, Mb, Geo::FLAT + Geo::EMB, Geo::G4, 1, Geo::G4, 0);
    else GEMM_W("lstm_dgrad", CfgMid, U128L, al, bl, blp, ep, Mb, Geo::FLAT + Geo::EMB, Geo::G4, 1, Geo::G4, 0);
  }
  // ---- action embedding + conv3 weight gradient (side) -------------------------------------
  // the embedding gradient: four small kernels that the hardware schedules late behind the big GEMMs (32 us alone, ~80 us
  // in the graph).  On one GPU they stay in front of conv3_wgrad on `side` (the second lane measured 0.4 % slower: the
  // backward pass is throughput-bound, earlier weight gradients only take SMs from the main chain).  With the fused peer
  // exchange the side stream IS the tail of the step (the early exchange part competes with it), and moving them to the
  // second lane (own scratch) gains 1 % at 2 GPUs.  DRL_B200_EMB_SIDE2=0/1 forces either.
  static const int emb_lane2_env = getenv("DRL_B200_EMB_SIDE2") ? atoi(getenv("DRL_B200_EMB_SIDE2")) : -1;
  const bool emb2 = lane2 && bw.emb_scratch != nullptr &&
                    (emb_lane2_env == 1 || (emb_lane2_env < 0 && st.ev_lstm_grads != nullptr));
  if (emb2) {
    DRL_TRY(fork_to_side2(st, 3));
    s = st.side2;
    KERNEL("emb_bwd",
           emb_backward(s, bw.du, in.pa, act.e1, act.table, P + pl.emb2_w, bw.dpre2, bw.dpre1, G + pl.emb1_w,
                        G + pl.emb1_b, G + pl.emb2_w, G + pl.emb2_b, bw.emb_scratch, Mb, B, T, A), 4);
  }
  DRL_TRY(fork_to_side(st, 4));
  s = side;
  if (!emb2)
    KERNEL("emb_bwd",
           emb_backward(s, bw.du, in.pa, act.e1, act.table, P + pl.emb2_w, bw.dpre2, bw.dpre1, G + pl.emb1_w,
                        G + pl.emb1_b, G + pl.emb2_w, G + pl.emb2_b, bw.wg_part, Mb, B, T, A), 4);
  // ---- conv3 -------------------------------------------------------------------------------
  {
    const SplitPlan sp = plan_conv3_wgrad(Mb, mode);
    const size_t slab = 577 * 64;
    Conv3WA al{act.a2, map};
    PlainB bl{bw.da3, 64, 0};
    EpRaw<true> ep{bw.wg_part, 64, slab, 1.0f, 576, 64};
    static const int cw8 = getenv("DRL_B200_CW8") ? atoi(getenv("DRL_B200_CW8")) : 1;
    if (m16 && cw8) GEMM16("conv3_wgrad", X64W8x2, al, bl, ep, 576, 64, Mb * 49, sp.splits, sp.kchunk, sp.kchunk);
    else if (m16) GEMM16("conv3_wgrad", X64W, al, bl, ep, 576, 64, Mb * 49, sp.splits, sp.kchunk, sp.kchunk);
    else GEMM("conv3_wgrad", CfgBig, U64, al, bl, ep, 576, 64, Mb * 49, sp.splits, sp.kchunk, sp.kchunk);
    KERNEL("conv3_wgrad_reduce", splitk_reduce(s, bw.wg_part, slab, sp.splits, G + pl.conv3_w, slab), 1);
  }
  s = st.main;
  // DRL_B200_DGRAD_GATHER=1 (math mode 5): the data gradients of conv3 / conv2 as gather-GEMMs over the input pixels
  // (K = taps x 64 output channels, ReLU mask in the epilogue) instead of dCol GEMM + col2im
  static const bool dgrad_gather = getenv("DRL_B200_DGRAD_GATHER") != nullptr;
  if (m16 && dgrad_gather) {
    Conv3DA al{bw.da3};
    Conv3DB bl{P + pl.conv3_w};
    Conv3DE ep{bw.da2, act.a2};
    GEMM16("conv3_dgrad", X64G, al, bl, ep, Mb * 81, 64, 576, 1, 576, 0);
  } else if (mode >= 2) {
    // "dCol" form: one plain GEMM with K = 64 output channels (instead of gathering every dY value 9 times
    // through the producers), then a gather of <= 9 taps per input pixel with the ReLU mask.
    PlainA al{bw.da3, 64, 0};
    PlainBT bl{P + pl.conv3_w, 64, 0};               // B(k = co, n = (ky,kx,ci)) = W[n*64 + co]
    EpRaw<false> ep{bw.dcol, 576, 0, 1.0f, 0, 576};
    // K = 64 (two K tiles) and 128 x 256 outputs per tile: epilogue-dominated, so the persistent kernel with
    // dedicated epilogue warps wins here (measured 0.067 vs 0.073 ms); elsewhere two CTAs per SM win.
    prof_mark(s, "conv3_dgrad");
    PretiledB<PlainBT> blp{wi.img[5], m16 ? 1 : 2};
    if (m16) DRL_TRY((launch_gemm_umma16<X256D>(s, al, blp, ep, Mb * 49, 576, 64, 1, 64, 0)));
    else DRL_TRY((launch_gemm_umma_persist<PersistOf<U256>::type>(s, al, blp, ep, Mb * 49, 576, 64, 1, 64, 0)));
    prof_mark(s, "conv3_col2im");
    DRL_TRY(col2im_conv3(s, bw.dcol, act.a2, bw.da2, Mb));
    n += 2;
  } else {
    Conv3DA al{bw.da3};
    Conv3DB bl{P + pl.conv3_w};
    Conv3DE ep{bw.da2, act.a2};
    GEMM_FFMA("conv3_dgrad", CfgBig, al, bl, ep, Mb * 81, 64, 576, 1, 576, 0);
  }
  // ---- conv2 -------------------------------------------------------------------------------
  DRL_TRY(fork_to_side(st, 5));
  s = side;
  {
    const SplitPlan sp = plan_conv2_wgrad(Mb, mode);
    const size_t slab = 513 * 64;
    Conv2WA al{act.a1, map};
    PlainB bl{bw.da2, 64, 0};
    EpRaw<true> ep{bw.wg_part, 64, slab, 1.0f, 512, 64};
    static const int cw8 = getenv("DRL_B200_CW8") ? atoi(getenv("DRL_B200_CW8")) : 1;
    if (m16 && cw8) GEMM16("conv2_wgrad", X64W8x2, al, bl, ep, 512, 64, Mb * 81, sp.splits, sp.kchunk, sp.kchunk);
    else if (m16) GEMM16("conv2_wgrad", X64W, al, bl, ep, 512, 64, Mb * 81, sp.splits, sp.kchunk, sp.kchunk);
    else GEMM("conv2_wgrad", CfgBig, U64, al, bl, ep, 512, 64, Mb * 81, sp.splits, sp.kchunk, sp.kchunk);
    KERNEL("conv2_wgrad_reduce", splitk_reduce(s, bw.wg_part, slab, sp.splits, G + pl.conv2_w, slab), 1);
  }
  s = st.main;
  if (m16 && dgrad_gather) {
    Conv2DA al{bw.da2};
    Conv2DB bl{P + pl.conv2_w};
    Conv2DE ep{bw.da1, act.a1};
    GEMM16("conv2_dgrad", X32G, al, bl, ep, Mb * 100, 32, 256, 4, 256, 0);
  } else if (mode >= 2) {
    PlainA al{bw.da2, 64, 0};
    PlainBT bl{P + pl.conv2_w, 64, 0};               // B(k = co, n = (ky,kx,ci)) = W[n*64 + co]
    EpRaw<false> ep{bw.dcol, 512, 0, 1.0f, 0, 512};
    prof_mark(s, "conv2_dgrad");                      // persistent kernel: 0.079 vs 0.091 ms
    PretiledB<PlainBT> blp{wi.img[6], m16 ? 1 : 2};
    if (m16) DRL_TRY((launch_gemm_umma16<X256D>(s, al, blp, ep, Mb * 81, 512, 64, 1, 64, 0)));
    else DRL_TRY((launch_gemm_umma_persist<PersistOf<U256>::type>(s, al, blp, ep, Mb * 81, 512, 64, 1, 64, 0)));
    prof_mark(s, "conv2_col2im");
    DRL_TRY(col2im_conv2(s, bw.dcol, act.a1, bw.da1, Mb));
    n += 2;
  } else {
    Conv2DA al{bw.da2};
    Conv2DB bl{P + pl.conv2_w};
    Conv2DE ep{bw.da1, act.a1};
    GEMM_FFMA("conv2_dgrad", CfgN32, al, bl, ep, Mb * 100, 32, 256, 4, 256, 0);
  }
  // ---- conv1 (input is data: weight gradient only) -----------------------------------------
  static const bool c1w_gather = getenv("DRL_B200_CONV1_GATHER") != nullptr;
  if (m16 && !c1w_gather) {
    // frame-resident TMA kernel (conv1_tma.cuh): one partial slab per CTA, then the fixed-order reduce
    const size_t slab = 257 * 32;
    int splits = 0;
    prof_mark(s, "conv1_wgrad");
    DRL_TRY(launch_conv1_wgrad_tma(s, in.frames, M, Mb, map, bw.da1, bw.wg_part2, bw.wg_part_floats, &splits));
    ++n;
    KERNEL("conv1_wgrad_reduce", splitk_reduce(s, bw.wg_part2, slab, splits, G + pl.conv1_w, slab), 1);
  } else {
    const SplitPlan sp = plan_conv1_wgrad(Mb, mode);
    const size_t slab = 257 * 32;
    Conv1WA al{in.frames, map};
    PlainB bl{bw.da1, 32, 0};
    EpRaw<true> ep{bw.wg_part2, 32, slab, 1.0f / 255.0f, 256, 32};   // own partial buffer: runs beside the side stream
    GEMM("conv1_wgrad", CfgWg1, U32, al, bl, ep, 256, 32, Mb * 400, sp.splits, sp.kchunk, sp.kchunk);
    KERNEL("conv1_wgrad_reduce", splitk_reduce(s, bw.wg_part2, slab, sp.splits, G + pl.conv1_w, slab), 1);
  }
  if (lane2) DRL_TRY(join_side2_into(st, 2, st.main));
  DRL_TRY(join_from_side(st, 6));
  g_bwd_launches = n;
  return DRL_OK;
}

}  // namespace drl
