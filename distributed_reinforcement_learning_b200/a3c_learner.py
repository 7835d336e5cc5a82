"""Thin object wrapper over the ``drl_a3c_*`` C-ABI (include/drl_b200.h): one A3C learner replica on one GPU.
``step`` is ``a3c.Agent.train`` (agent/a3c.py:85-103) minus the Python/TF session."""
import ctypes as C

import numpy as np

from . import _native as N
from . import dp
from ._native import _as_u8


class NativeA3CLearner(dp.AdamLearner):
    _prefix = "a3c"
    set_params = N.NativeHandle.set_params      # one network: no `which`
    get_params = N.NativeHandle.get_params

    def __init__(self, batch, num_action=4, input_shape=(84, 84, 4), discount_factor=0.997, start_learning_rate=1e-4,
                 end_learning_rate=0.0, learning_frame=1000000000, baseline_loss_coef=1.0, entropy_coef=0.05,
                 gradient_clip_norm=40.0, reward_clipping="abs_one", device=0, num_slots=2, use_cuda_graph=False,
                 math_mode=0):
        if reward_clipping not in N.REWARD_CLIPPING:
            raise ValueError("reward_clipping must be one of %s" % sorted(N.REWARD_CLIPPING))     # utils.py:45
        h, w, c = input_shape
        self.B, self.A = int(batch), int(num_action)
        self.input_shape = (int(h), int(w), int(c))
        cfg = N.A3cConfig(self.B, h, w, c, self.A, discount_factor, start_learning_rate, end_learning_rate,
                          float(learning_frame), baseline_loss_coef, entropy_coef, gradient_clip_norm,
                          N.REWARD_CLIPPING[reward_clipping], int(device), int(num_slots), int(bool(use_cuda_graph)),
                          int(math_mode))
        self._open(cfg, num_slots, int(device))

    def stage(self, slot, state, next_state, previous_action, action, reward, done):
        B = self.B
        arrs = (N.as_c(state, np.uint8, (B,) + self.input_shape, "state"),
                N.as_c(next_state, np.uint8, (B,) + self.input_shape, "next_state"),
                N.as_c(previous_action, np.int32, (B,), "previous_action"), N.as_c(action, np.int32, (B,), "action"),
                N.as_c(reward, np.float32, (B,), "reward"), N.as_c(_as_u8(done), np.uint8, (B,), "done"))
        self._keep[slot] = arrs
        N.check(N.lib.drl_a3c_stage(self._h, slot, *[N.ptr(a) for a in arrs]))

    def wait(self):
        o = N.A3cOut()
        N.check(N.lib.drl_a3c_wait(self._h, C.byref(o)))
        return dict(pi_loss=o.pi_loss, baseline_loss=o.baseline_loss, entropy=o.entropy, learning_rate=o.learning_rate,
                    grad_norm=o.grad_norm, step=o.step)

    def act(self, state, previous_action):
        st = N.as_c(state, np.uint8)
        n = st.shape[0]
        st = N.as_c(st, np.uint8, (n,) + self.input_shape, "state")
        pa = N.as_c(previous_action, np.int32, (n,), "previous_action")
        pol = np.empty((n, self.A), np.float32)
        val = np.empty(n, np.float32)
        N.check(N.lib.drl_a3c_act(self._h, n, N.ptr(st), N.ptr(pa), N.ptr(pol), N.ptr(val)))
        return pol, val

    def taps(self):
        B = self.B
        out = [np.empty((B, self.A), np.float32), np.empty(B, np.float32), np.empty(B, np.float32), np.empty(B, np.float32)]
        N.check(N.lib.drl_a3c_taps(self._h, *[N.ptr(a) for a in out]))
        return dict(policy=out[0], value=out[1], next_value=out[2], advantage=out[3])
