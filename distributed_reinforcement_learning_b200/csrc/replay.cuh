// replay.cuh -- internal interface between the device-resident prioritized replay (replay.cu, drl_apex_replay_*) and
// the Ape-X learner handle (apex.cu).  Not part of the C-ABI.  The replay only sees the learner through these calls:
// it never depends on the handle's layout, and the tree kernels never depend on the Ape-X record layout.
#pragma once
#include <functional>

#include "kernels.h"

struct drl_apex;

namespace drl {

// device pointers of one staging slot of the Ape-X learner, in the layout drl_apex_stage produces: frames = [s rows ;
// s' rows], pa2 = [previous_action ; action], with the second half starting at row `row2`
struct ApexRecordView {
  uint8_t* frames;
  int32_t* pa2;
  float* reward;
  uint8_t* done;
  float* weight;
  int row2;
};

// what a replay needs to know about the learner it is attached to
struct ApexReplayLink {
  std::recursive_mutex* mu;   // the learner's lock (every replay entry point takes it)
  int device, B, algo;        // algo: 0 = Ape-X DQN, 1 = A3C
  cudaStream_t compute;
  const float* td_dev;        // [B] |target - q(s, a)| of the most recent forward (step or td_error)
};
int apex_replay_link(drl_apex* h, ApexReplayLink* out);
// counts the replays attached to h (+1 on create, -1 on destroy); drl_apex_destroy refuses while any is alive
void apex_replay_attach(drl_apex* h, int delta);

// the work of drl_apex_td_error for n <= B transitions, enqueued on the compute stream without the D2H copy: stage
// into the scratch slot, main and target forward, TD kernel.  |td| lands in td_dev; *scratch views the staged rows.
int apex_enqueue_td_error(drl_apex* h, int n, const uint8_t* state, const uint8_t* next_state,
                          const int32_t* previous_action, const int32_t* action, const float* reward,
                          const uint8_t* done, ApexRecordView* scratch);

// a learner step on training slot `slot` whose minibatch is written on the device: fill() is enqueued on the compute
// stream before forward + loss + backward + Adam, after() behind them.  With use_cuda_graph the three are captured
// into graphs[slot] (the caller's cache, separate from the learner's own).  Collect with drl_apex_wait.
using ApexSlotWork = std::function<int(cudaStream_t, const ApexRecordView&)>;
int apex_replay_step(drl_apex* h, int slot, std::vector<cudaGraphExec_t>& graphs, const ApexSlotWork& fill,
                     const ApexSlotWork& after);

}  // namespace drl
