"""Data-parallel plumbing shared by the Ape-X, A3C and R2D2 learners: one process per GPU, every rank feeds its own
minibatch, ONE ``all_reduce(SUM)`` of the gradient bucket (loss scalars in its tail) between the two halves of the step
(``drl_<family>_forward_backward`` / ``drl_<family>_apply``).  Their losses are batch MEANS, so the update of the
undivided global batch is the summed bucket times 1 / world_size (``grad_scale``)."""
import ctypes as C

import numpy as np

from . import _native as N


def distributed():
    try:
        import torch.distributed as dist
    except Exception:      # pragma: no cover
        return False
    return dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1


class BucketAllReduce:
    def __init__(self, family, handle, device):
        self.family, self._h, self.device = family, handle, int(device)
        self._bucket = self._stream = None

    def _fn(self, name):
        return getattr(N.lib, "drl_%s_%s" % (self.family, name))

    def _tensor(self):
        if self._bucket is None:
            import torch
            p, n, s = C.c_void_p(), C.c_int64(), C.c_void_p()
            N.check(self._fn("grad_bucket")(self._h, C.byref(p), C.byref(n)))
            N.check(self._fn("stream")(self._h, C.byref(s)))

            class _View:
                __cuda_array_interface__ = {"shape": (int(n.value),), "typestr": "<f4", "data": (int(p.value), False),
                                            "version": 2}
            dev = "cuda:%d" % self.device
            self._bucket = torch.as_tensor(_View(), device=dev)
            self._stream = torch.cuda.ExternalStream(int(s.value or 0), device=dev)
        return self._bucket

    def step_async(self, slot):
        """forward+backward -> all_reduce(SUM) on the learner's stream -> clip + Adam with grad_scale = 1 / world."""
        import torch
        import torch.distributed as dist
        N.check(self._fn("forward_backward")(self._h, slot))
        t = self._tensor()
        with torch.cuda.stream(self._stream):
            dist.all_reduce(t, op=dist.ReduceOp.SUM)
        N.check(self._fn("apply")(self._h, C.c_float(1.0 / dist.get_world_size())))


MAIN, TARGET = 0, 1      # the network a parameter call addresses (Ape-X, R2D2)


class AdamLearner(N.NativeHandle):
    """The Ape-X, A3C and R2D2 wrappers: TF1 Adam state, the main / target parameters and the step, which is data
    parallel through ``BucketAllReduce`` when torch.distributed runs with world > 1.  A family sets ``_prefix`` and,
    for ``wait``, ``_Out`` and ``_out``."""

    def _open(self, cfg, num_slots, device):
        super()._open(cfg, num_slots)
        self._dp = BucketAllReduce(self._prefix, self._h, device)

    def set_params(self, flat, which=MAIN):
        a = N.as_c(flat, np.float32, (self.param_count,), "params")
        N.check(self._fn("set_params")(self._h, int(which), N.ptr(a), a.size))

    def get_params(self, which=MAIN):
        a = np.empty(self.param_count, np.float32)
        N.check(self._fn("get_params")(self._h, int(which), N.ptr(a), a.size))
        return a

    def set_opt_state(self, m, v, step, beta1_power=0.9, beta2_power=0.999):
        am = N.as_c(m, np.float32, (self.param_count,), "m")
        av = N.as_c(v, np.float32, (self.param_count,), "v")
        N.check(self._fn("set_opt_state")(self._h, N.ptr(am), N.ptr(av), am.size, int(step), float(beta1_power),
                                          float(beta2_power)))

    def get_opt_state(self):
        m = np.empty(self.param_count, np.float32)
        v = np.empty(self.param_count, np.float32)
        st, b1, b2 = C.c_int64(), C.c_float(), C.c_float()
        N.check(self._fn("get_opt_state")(self._h, N.ptr(m), N.ptr(v), m.size, C.byref(st), C.byref(b1),
                                          C.byref(b2)))
        return dict(m=m, v=v, step=int(st.value), beta1_power=float(b1.value), beta2_power=float(b2.value))

    def step(self, slot=0):
        self.step_async(slot)
        return self.wait()

    def step_async(self, slot=0):
        if distributed():
            self._dp.step_async(slot)
        else:
            N.check(self._fn("step_async")(self._h, slot))

    def wait(self):
        """-> (scalars dict, td_error [B]) of the step in flight."""
        o = self._Out()
        td = np.empty(self.B, np.float32)
        N.check(self._fn("wait")(self._h, C.byref(o), N.ptr(td)))
        return self._out(o), td
