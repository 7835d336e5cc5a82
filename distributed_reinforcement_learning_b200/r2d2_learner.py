"""Thin object wrapper over the ``drl_r2d2_*`` C-ABI (include/drl_b200.h): one R2D2 learner replica on one GPU.

``step`` is ``r2d2.Agent.train`` (agent/r2d2.py:132-159) minus the Python/TF session: the stored-state LSTM unroll of
the main and the target scope over seq_len steps, double-Q targets with value-function rescaling over the
post-burn-in window, the weighted loss, BPTT through all steps of the main scope and TF1 Adam; it returns the new
priorities |mean_t(target - q)|.
"""
import ctypes as C

import numpy as np

from . import _native as N
from . import dp
from ._native import _as_u8
from .dp import MAIN, TARGET  # noqa: F401  (the `which` of set_params / get_params)


class NativeR2D2Learner(dp.AdamLearner):
    _prefix = "r2d2"
    _Out = N.R2d2Out

    def __init__(self, batch, seq_len=15, burn_in=7, num_action=4, lstm_size=64, input_shape=(84, 84, 1),
                 discount_factor=0.997, learning_rate=1e-4, device=0, num_slots=2, use_cuda_graph=False, math_mode=0):
        h, w, c = input_shape
        self.B, self.S, self.bi, self.A, self.L = int(batch), int(seq_len), int(burn_in), int(num_action), int(lstm_size)
        self.Nt = self.S - self.bi - 1
        self.input_shape = (int(h), int(w), int(c))
        self.device = int(device)
        cfg = N.R2d2Config(self.B, self.S, self.bi, h, w, c, self.A, self.L, discount_factor, learning_rate,
                           self.device, int(num_slots), int(bool(use_cuda_graph)), int(math_mode))
        self._open(cfg, num_slots, self.device)

    def main_to_target(self):
        N.check(N.lib.drl_r2d2_main_to_target(self._h))

    def _arrays(self, n, state, previous_action, action, h0, c0, reward, done):
        S = self.S
        return (N.as_c(state, np.uint8, (n, S) + self.input_shape, "state"),
                N.as_c(previous_action, np.int32, (n, S), "previous_action"),
                N.as_c(action, np.int32, (n, S), "action"),
                N.as_c(h0, np.float32, (n, self.L), "h0"), N.as_c(c0, np.float32, (n, self.L), "c0"),
                N.as_c(reward, np.float32, (n, S), "reward"), N.as_c(_as_u8(done), np.uint8, (n, S), "done"))

    def stage(self, slot, state, previous_action, action, h0, c0, reward, done, weight=None):
        arrs = self._arrays(self.B, state, previous_action, action, h0, c0, reward, done)
        w = None if weight is None else N.as_c(weight, np.float32, (self.B,), "weight")
        self._keep[slot] = arrs + (w,)
        N.check(N.lib.drl_r2d2_stage(self._h, slot, *[N.ptr(a) for a in arrs], N.ptr(w) if w is not None else None))

    @staticmethod
    def _out(o):
        return dict(loss=o.loss, grad_norm=o.grad_norm, step=o.step)

    def td_error(self, state, previous_action, action, h0, c0, reward, done):
        n = int(np.asarray(state).shape[0])
        arrs = self._arrays(n, state, previous_action, action, h0, c0, reward, done)
        td = np.empty(n, np.float32)
        N.check(N.lib.drl_r2d2_td_error(self._h, n, *[N.ptr(a) for a in arrs], N.ptr(td)))
        return td

    def act(self, state, previous_action, h, c):
        st = N.as_c(state, np.uint8)
        n = st.shape[0]
        st = N.as_c(st, np.uint8, (n,) + self.input_shape, "state")
        pa = N.as_c(previous_action, np.int32, (n,), "previous_action")
        hh = N.as_c(h, np.float32, (n, self.L), "h")
        cc = N.as_c(c, np.float32, (n, self.L), "c")
        q = np.empty((n, self.A), np.float32)
        ho = np.empty((n, self.L), np.float32)
        co = np.empty((n, self.L), np.float32)
        N.check(N.lib.drl_r2d2_act(self._h, n, N.ptr(st), N.ptr(pa), N.ptr(hh), N.ptr(cc), N.ptr(q), N.ptr(ho), N.ptr(co)))
        return q, ho, co

    def taps(self, n=None):
        n = self.B if n is None else int(n)
        mq = np.empty((n, self.S, self.A), np.float32)
        tq = np.empty((n, self.S, self.A), np.float32)
        tv = np.empty((n, self.Nt), np.float32)
        sv = np.empty((n, self.Nt), np.float32)
        N.check(N.lib.drl_r2d2_taps(self._h, N.ptr(mq), N.ptr(tq), N.ptr(tv), N.ptr(sv)))
        return dict(main_q=mq, target_q=tq, target_value=tv, state_action_value=sv)
