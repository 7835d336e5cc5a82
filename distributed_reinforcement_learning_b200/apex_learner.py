"""Thin object wrapper over the ``drl_apex_*`` C-ABI (include/drl_b200.h): one Ape-X DQN learner replica on one GPU.

``step`` is ``apex.Agent.distributed_train`` (agent/apex.py:135-154) minus the Python/TF session: three dueling-network
evaluations (one main-network forward over [s ; s'], one target-network forward over s'), the double-DQN TD target, the
importance-weighted squared loss, the backward pass through main(s), global-norm clipping and TF1 Adam -- and it
returns the new priorities |target - q(s, a)|.
"""
import ctypes as C

import numpy as np

from . import _native as N
from . import dp
from ._native import _as_u8
from .dp import MAIN, TARGET  # noqa: F401  (the `which` of set_params / get_params)


class NativeApexLearner(dp.AdamLearner):
    _prefix = "apex"
    _Out = N.ApexOut

    def __init__(self, batch, num_action=4, input_shape=(84, 84, 4), discount_factor=0.99, gradient_clip_norm=40.0,
                 reward_clipping="abs_one", start_learning_rate=1e-4, end_learning_rate=0.0,
                 learning_frame=100000000000000, device=0, num_slots=2, use_cuda_graph=False, math_mode=0):
        h, w, c = input_shape
        self.B, self.A = int(batch), int(num_action)
        self.input_shape = (int(h), int(w), int(c))
        self.device = int(device)
        # agent/apex.py:38-41: 'abs_one' clips, anything else feeds the raw reward
        clip = 0 if reward_clipping == "abs_one" else 2
        cfg = N.ApexConfig(self.B, h, w, c, self.A, discount_factor, start_learning_rate, end_learning_rate,
                           float(learning_frame), gradient_clip_norm, clip, self.device, int(num_slots),
                           int(bool(use_cuda_graph)), int(math_mode))
        self._open(cfg, num_slots, self.device)

    def target_to_main(self):
        """agent/apex.py:78-79: assigns target <- main (sic)."""
        N.check(N.lib.drl_apex_target_to_main(self._h))

    # ---- data path ---------------------------------------------------------------------
    def _arrays(self, n, state, next_state, previous_action, action, reward, done):
        return (N.as_c(state, np.uint8, (n,) + self.input_shape, "state"),
                N.as_c(next_state, np.uint8, (n,) + self.input_shape, "next_state"),
                N.as_c(previous_action, np.int32, (n,), "previous_action"),
                N.as_c(action, np.int32, (n,), "action"),
                N.as_c(reward, np.float32, (n,), "reward"),
                N.as_c(_as_u8(done), np.uint8, (n,), "done"))

    def stage(self, slot, state, next_state, previous_action, action, reward, done, is_weight=None):
        arrs = self._arrays(self.B, state, next_state, previous_action, action, reward, done)
        w = None if is_weight is None else N.as_c(is_weight, np.float32, (self.B,), "is_weight")
        self._keep[slot] = arrs + (w,)
        N.check(N.lib.drl_apex_stage(self._h, slot, *[N.ptr(a) for a in arrs], N.ptr(w) if w is not None else None))

    @staticmethod
    def _out(o):
        return dict(loss=o.loss, learning_rate=o.learning_rate, grad_norm=o.grad_norm, step=o.step)

    def td_error(self, state, next_state, previous_action, action, reward, done):
        """agent/apex.py:116-133 for n <= batch transitions."""
        n = int(np.asarray(state).shape[0])
        arrs = self._arrays(n, state, next_state, previous_action, action, reward, done)
        td = np.empty(n, np.float32)
        N.check(N.lib.drl_apex_td_error(self._h, n, *[N.ptr(a) for a in arrs], N.ptr(td)))
        return td

    def act(self, state, previous_action):
        """main_q_value [n, A] (agent/apex.py:88-96)."""
        st = N.as_c(state, np.uint8)
        n = st.shape[0]
        st = N.as_c(st, np.uint8, (n,) + self.input_shape, "state")
        pa = N.as_c(previous_action, np.int32, (n,), "previous_action")
        q = np.empty((n, self.A), np.float32)
        N.check(N.lib.drl_apex_act(self._h, n, N.ptr(st), N.ptr(pa), N.ptr(q)))
        return q

    def taps(self, n=None):
        n = self.B if n is None else int(n)
        out = [np.empty((n, self.A), np.float32) for _ in range(3)] + [np.empty(n, np.float32) for _ in range(2)]
        N.check(N.lib.drl_apex_taps(self._h, *[N.ptr(a) for a in out]))
        return dict(main_q=out[0], next_main_q=out[1], target_q=out[2], target_value=out[3],
                    state_action_value=out[4])


class NativeApexReplay:
    """Prioritized replay of ``learner`` kept in its GPU memory (``drl_apex_replay_*``): ``buffer_queue.Memory`` and the
    transitions it indexes.  ``add`` is ``Agent.get_td_error`` + ``Memory.add`` for any number of transitions;
    ``step(slot)`` is ``Memory.sample`` -> ``distributed_train`` -> ``Memory.update`` as one enqueue on the learner's
    stream, returning what ``learner.step`` returns.  The uniforms of the stratified draw come from a counter-based
    generator seeded with ``seed`` (oracle/replay_np.py restates it).  Close the replay before its learner."""

    def __init__(self, learner, capacity, seed=0):
        self.learner = learner
        self.B = learner.B
        self.capacity = int(capacity)
        self._r = C.c_void_p()
        N.check(N.lib.drl_apex_replay_create(learner._h, self.capacity, C.c_uint64(int(seed)), C.byref(self._r)))

    def close(self):
        if getattr(self, "_r", None) is not None and self._r.value:
            N.lib.drl_apex_replay_destroy(self._r)
            self._r = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def add(self, state, next_state, previous_action, action, reward, done):
        """n transitions, in chunks of the learner's batch (as Agent.get_td_error) -> their |td| are the priorities."""
        n = int(np.asarray(state).shape[0])
        for lo in range(0, n, self.B):
            hi = min(lo + self.B, n)
            arrs = self.learner._arrays(hi - lo, np.asarray(state)[lo:hi], np.asarray(next_state)[lo:hi],
                                        np.asarray(previous_action)[lo:hi], np.asarray(action)[lo:hi],
                                        np.asarray(reward)[lo:hi], np.asarray(done)[lo:hi])
            N.check(N.lib.drl_apex_replay_add(self._r, hi - lo, *[N.ptr(a) for a in arrs]))

    def step_async(self, slot=0):
        N.check(N.lib.drl_apex_replay_step_async(self._r, int(slot)))

    def step(self, slot=0):
        """-> (scalars dict, td_error [B]) like NativeApexLearner.step."""
        self.step_async(slot)
        return self.learner.wait()

    def last_sample(self):
        ti, di = np.empty(self.B, np.int64), np.empty(self.B, np.int64)
        pr, w = np.empty(self.B, np.float64), np.empty(self.B, np.float64)
        N.check(N.lib.drl_apex_replay_last_sample(self._r, N.ptr(ti), N.ptr(di), N.ptr(pr), N.ptr(w)))
        return dict(tree_index=ti, data_index=di, priority=pr, is_weight=w)

    def last_update(self):
        """-> (leaves, priorities) of the most recent add or post-step update, in call order."""
        leaf, p = np.empty(self.B, np.int64), np.empty(self.B, np.float64)
        cnt = C.c_int32()
        N.check(N.lib.drl_apex_replay_last_update(self._r, N.ptr(leaf), N.ptr(p), self.B, C.byref(cnt)))
        return leaf[:cnt.value].copy(), p[:cnt.value].copy()

    def info(self):
        n, w, dr = C.c_int64(), C.c_int64(), C.c_int64()
        t, b = C.c_double(), C.c_double()
        N.check(N.lib.drl_apex_replay_info(self._r, C.byref(n), C.byref(w), C.byref(t), C.byref(b), C.byref(dr)))
        return dict(n_entries=int(n.value), write=int(w.value), total=float(t.value), beta=float(b.value),
                    draws=int(dr.value))

    def tree(self):
        a = np.empty(2 * self.capacity - 1, np.float64)
        N.check(N.lib.drl_apex_replay_read_tree(self._r, N.ptr(a), a.size))
        return a

    def __len__(self):
        return self.info()["n_entries"]
