"""Thin object wrapper over the ``drl_learner_*`` C-ABI (include/drl_b200.h).

One ``NativeLearner`` = one process-per-GPU learner replica: it owns the device parameters,
RMSProp slots, gradient bucket, activations and staging slots.  ``step`` is
agent/impala.py:132-148 (``Agent.train``) minus the Python/TF session.  With
``torch.distributed`` initialised (world_size > 1) the step is split into
forward+backward -> one NCCL all-reduce(SUM) of the gradient bucket -> apply
(SURVEY.md section 8(e)); the reduction is a SUM because the reference losses are batch sums
(optimizer/vtrace.py:112,118,126).
"""
import ctypes as C

import numpy as np

from . import _native as N
from ._native import _as_u8

H, W, CH, LSTM = 84, 84, 4, 256


class NativeLearner(N.NativeHandle):
    _prefix = "learner"

    def __init__(self, batch, trajectory=20, num_action=18, lstm_hidden_size=256, input_shape=(84, 84, 4),
                 discount_factor=0.99, start_learning_rate=0.0006, end_learning_rate=0.0,
                 learning_frame=1000000000, baseline_loss_coef=1.0, entropy_coef=0.05,
                 gradient_clip_norm=40.0, reward_clipping="abs_one", device=0, num_slots=2,
                 use_cuda_graph=True, math_mode=0):
        if reward_clipping not in N.REWARD_CLIPPING:
            raise ValueError("reward_clipping must be one of %s" % sorted(N.REWARD_CLIPPING))   # utils.py:45
        h, w, c = input_shape
        self.B, self.T, self.A, self.L = int(batch), int(trajectory), int(num_action), int(lstm_hidden_size)
        self.input_shape = (int(h), int(w), int(c))
        self.device = int(device)
        cfg = N.LearnerConfig(self.B, self.T, h, w, c, self.A, self.L, discount_factor, start_learning_rate,
                              end_learning_rate, float(learning_frame), baseline_loss_coef, entropy_coef,
                              gradient_clip_norm, N.REWARD_CLIPPING[reward_clipping], self.device, int(num_slots),
                              int(bool(use_cuda_graph)), int(math_mode))
        self._open(cfg, num_slots)
        self._bucket = None
        self._ext_stream = None
        self._peer = False
        self._no_collective = False          # diagnostic only (bench.py --collective none)

    # ---- optimizer state ---------------------------------------------------------------
    def set_opt_state(self, ms_flat, step):
        a = N.as_c(ms_flat, np.float32, (self.param_count,), "ms")
        N.check(N.lib.drl_learner_set_opt_state(self._h, N.ptr(a), a.size, int(step)))

    def get_opt_state(self):
        a = np.empty(self.param_count, np.float32)
        st = C.c_int64()
        N.check(N.lib.drl_learner_get_opt_state(self._h, N.ptr(a), a.size, C.byref(st)))
        return a, int(st.value)

    # ---- data path -----------------------------------------------------------------
    def stage(self, slot, state, reward, action, done, behavior_policy, previous_action, initial_h, initial_c):
        """Async H2D of one batch-major batch (feed of agent/impala.py:134-142)."""
        B, T, A, L = self.B, self.T, self.A, self.L
        arrs = (N.as_c(state, np.uint8, (B, T) + self.input_shape, "state"),
                N.as_c(reward, np.float32, (B, T), "reward"),
                N.as_c(action, np.int32, (B, T), "action"),
                N.as_c(_as_u8(done), np.uint8, (B, T), "done"),
                N.as_c(behavior_policy, np.float32, (B, T, A), "behavior_policy"),
                N.as_c(previous_action, np.int32, (B, T), "previous_action"),
                N.as_c(initial_h, np.float32, (B, T, L), "initial_h"),
                N.as_c(initial_c, np.float32, (B, T, L), "initial_c"))
        self._keep[slot] = arrs
        N.check(N.lib.drl_learner_stage(self._h, slot, *[N.ptr(a) for a in arrs]))

    @staticmethod
    def _out(o):
        return dict(pi_loss=o.pi_loss, baseline_loss=o.baseline_loss, entropy=o.entropy,
                    learning_rate=o.learning_rate, grad_norm=o.grad_norm, total_loss=o.total_loss, step=o.step)

    def step(self, slot=0):
        """sess.run([... train_op]) of agent/impala.py:144-146 on a staged slot."""
        if self._distributed() and not self._peer:
            self.step_async(slot)
            return self.wait()
        o = N.StepOut()
        N.check(N.lib.drl_learner_step(self._h, slot, C.byref(o)))
        return self._out(o)

    def step_async(self, slot=0):
        if self._peer or self._no_collective:   # peer: the exchange is part of the step's CUDA graph (csrc/peer.cu)
            N.check(N.lib.drl_learner_step_async(self._h, slot))
        elif self._distributed():
            N.check(N.lib.drl_learner_forward_backward(self._h, slot))
            self._allreduce_bucket()
            N.check(N.lib.drl_learner_apply(self._h))
        else:
            N.check(N.lib.drl_learner_step_async(self._h, slot))

    def wait(self, slot=None):
        """Scalars of the last enqueued step; with `slot`, of the last step_async on that slot (each slot has its own
        result record, so two steps can be in flight: read step i-1 while step i runs)."""
        o = N.StepOut()
        if slot is None:
            N.check(N.lib.drl_learner_wait(self._h, C.byref(o)))
        else:
            N.check(N.lib.drl_learner_wait_slot(self._h, int(slot), C.byref(o)))
        return self._out(o)

    def forward_backward(self, slot=0):
        N.check(N.lib.drl_learner_forward_backward(self._h, slot))

    def apply(self):
        N.check(N.lib.drl_learner_apply(self._h))

    def forward(self, slot=0):
        pol = np.empty((self.B, self.T, self.A), np.float32)
        val = np.empty((self.B, self.T), np.float32)
        N.check(N.lib.drl_learner_forward(self._h, slot, N.ptr(pol), N.ptr(val)))
        return pol, val

    def taps(self):
        shp = (self.B, self.T - 2)
        out = [np.empty(shp, np.float32) for _ in range(4)]
        N.check(N.lib.drl_learner_taps(self._h, *[N.ptr(a) for a in out]))
        return dict(vs=out[0], clipped_rho=out[1], vs_plus_1=out[2], pg_advantage=out[3])

    def act(self, state, previous_action, h, c):
        """n single-step forwards (agent/impala.py:118-130 without the sampling)."""
        st = N.as_c(state, np.uint8)
        n = st.shape[0]
        st = N.as_c(st, np.uint8, (n,) + self.input_shape, "state")
        pa = N.as_c(previous_action, np.int32, (n,), "previous_action")
        hh = N.as_c(h, np.float32, (n, self.L), "h")
        cc = N.as_c(c, np.float32, (n, self.L), "c")
        pol = np.empty((n, self.A), np.float32)
        ho = np.empty((n, self.L), np.float32)
        co = np.empty((n, self.L), np.float32)
        N.check(N.lib.drl_learner_act(self._h, n, N.ptr(st), N.ptr(pa), N.ptr(hh), N.ptr(cc), N.ptr(pol),
                                      N.ptr(ho), N.ptr(co)))
        return pol, ho, co

    # ---- data parallel ---------------------------------------------------------------
    @staticmethod
    def _distributed():
        try:
            import torch.distributed as dist
        except Exception:      # pragma: no cover
            return False
        return dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1

    def enable_peer_exchange(self, group=None):
        """Replace the NCCL all-reduce of the gradient bucket by the fused exchange over NVLink peer memory
        (csrc/peer.cu): the ranks of ONE node swap CUDA-IPC handles here (a 128-byte all_gather), after which
        forward, backward, exchange and update run as one CUDA graph.  Collective: every rank must call it.
        Returns True when every rank could map every peer; otherwise all ranks stay on the NCCL path (False)."""
        import torch
        import torch.distributed as dist
        if not self._distributed():
            raise RuntimeError("enable_peer_exchange needs an initialised process group with world_size > 1")
        rank, world = dist.get_rank(group), dist.get_world_size(group)
        dev = torch.device("cuda", self.device)
        mine = np.zeros(128, np.uint8)
        ok = N.lib.drl_learner_peer_export(self._h, N.ptr(mine), mine.size) == 0
        t = torch.from_numpy(mine).to(dev)
        parts = [torch.empty_like(t) for _ in range(world)]
        dist.all_gather(parts, t, group=group)
        allh = np.ascontiguousarray(torch.stack(parts).cpu().numpy())
        ok = ok and N.lib.drl_learner_peer_import(self._h, rank, world, N.ptr(allh), allh.size) == 0
        flag = torch.tensor([1 if ok else 0], dtype=torch.int32, device=dev)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN, group=group)       # all or nobody
        if int(flag.item()) == 0:
            N.lib.drl_learner_peer_disable(self._h)
            dist.barrier(group=group)
            self._peer = False
            return False
        dist.barrier(group=group)
        self._peer = True
        return True

    def bucket_tensor(self):
        """torch view (no copy) of the device gradient bucket [padded grads | 3 loss sums | pad]."""
        if self._bucket is None:
            import torch
            p, n = C.c_void_p(), C.c_int64()
            N.check(N.lib.drl_learner_grad_bucket(self._h, C.byref(p), C.byref(n)))

            class _View:
                __cuda_array_interface__ = {"shape": (int(n.value),), "typestr": "<f4",
                                            "data": (int(p.value), False), "version": 2}
            self._bucket = torch.as_tensor(_View(), device="cuda:%d" % self.device)
            self._ext_stream = torch.cuda.ExternalStream(self.stream_ptr(), device="cuda:%d" % self.device)
        return self._bucket

    def reduced_tensor(self):
        """torch view (no copy) of the bucket the update reads (the peer exchange's ``reduced`` buffer, else the
        all-reduced gradient bucket) -- for checks against a library all-reduce of the saved local buckets."""
        import torch
        p, n = C.c_void_p(), C.c_int64()
        N.check(N.lib.drl_learner_reduced_bucket(self._h, C.byref(p), C.byref(n)))

        class _View:
            __cuda_array_interface__ = {"shape": (int(n.value),), "typestr": "<f4",
                                        "data": (int(p.value), False), "version": 2}
        return torch.as_tensor(_View(), device="cuda:%d" % self.device)

    def _allreduce_bucket(self):
        import torch
        import torch.distributed as dist
        t = self.bucket_tensor()
        with torch.cuda.stream(self._ext_stream):       # ordered after backward, before apply
            dist.all_reduce(t, op=dist.ReduceOp.SUM)


def shard_range(rank, world_size, batch_total):
    """Rank r takes trajectories [r*B/W, (r+1)*B/W) (SURVEY.md section 8(e))."""
    if batch_total % world_size != 0:
        raise ValueError("global batch %d is not divisible by world size %d" % (batch_total, world_size))
    per = batch_total // world_size
    return rank * per, (rank + 1) * per
