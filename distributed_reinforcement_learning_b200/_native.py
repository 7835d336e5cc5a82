"""ctypes binding of the C-ABI in ``include/drl_b200.h`` (``csrc/libdrl_b200.so``).

There is no CPU fallback: if the shared library is missing, importing this module raises, and
every compute entry point fails with ``DrlError`` when no CUDA device is visible.
"""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "csrc", "libdrl_b200.so")

DRL_OK, DRL_ERR_INVALID, DRL_ERR_CUDA, DRL_ERR_STATE, DRL_ERR_TIMEOUT = 0, -1, -2, -3, -4
REWARD_CLIPPING = {"abs_one": 0, "soft_asymmetric": 1}   # agent/impala.py:45-49, utils.py:45


class DrlError(RuntimeError):
    def __init__(self, code, text):
        super().__init__("drl_b200 error %d: %s" % (code, text))
        self.code = code


class TimeoutError_(DrlError):
    pass


class LearnerConfig(C.Structure):
    _fields_ = [("batch", C.c_int32), ("trajectory", C.c_int32), ("height", C.c_int32), ("width", C.c_int32),
                ("channels", C.c_int32), ("num_action", C.c_int32), ("lstm_size", C.c_int32),
                ("discount_factor", C.c_float), ("start_learning_rate", C.c_float),
                ("end_learning_rate", C.c_float), ("learning_frame", C.c_double),
                ("baseline_loss_coef", C.c_float), ("entropy_coef", C.c_float),
                ("gradient_clip_norm", C.c_float), ("reward_clipping", C.c_int32), ("device", C.c_int32),
                ("num_slots", C.c_int32), ("use_cuda_graph", C.c_int32), ("math_mode", C.c_int32)]


class StepOut(C.Structure):
    _fields_ = [("pi_loss", C.c_float), ("baseline_loss", C.c_float), ("entropy", C.c_float),
                ("learning_rate", C.c_float), ("grad_norm", C.c_float), ("total_loss", C.c_float),
                ("step", C.c_int64)]


class ApexConfig(C.Structure):
    _fields_ = [("batch", C.c_int32), ("height", C.c_int32), ("width", C.c_int32), ("channels", C.c_int32),
                ("num_action", C.c_int32), ("discount_factor", C.c_float), ("start_learning_rate", C.c_float),
                ("end_learning_rate", C.c_float), ("learning_frame", C.c_double), ("gradient_clip_norm", C.c_float),
                ("reward_clipping", C.c_int32), ("device", C.c_int32), ("num_slots", C.c_int32),
                ("use_cuda_graph", C.c_int32), ("math_mode", C.c_int32)]


class ApexOut(C.Structure):
    _fields_ = [("loss", C.c_float), ("learning_rate", C.c_float), ("grad_norm", C.c_float), ("step", C.c_int64)]


class A3cConfig(C.Structure):
    _fields_ = [("batch", C.c_int32), ("height", C.c_int32), ("width", C.c_int32), ("channels", C.c_int32),
                ("num_action", C.c_int32), ("discount_factor", C.c_float), ("start_learning_rate", C.c_float),
                ("end_learning_rate", C.c_float), ("learning_frame", C.c_double), ("baseline_loss_coef", C.c_float),
                ("entropy_coef", C.c_float), ("gradient_clip_norm", C.c_float), ("reward_clipping", C.c_int32),
                ("device", C.c_int32), ("num_slots", C.c_int32), ("use_cuda_graph", C.c_int32), ("math_mode", C.c_int32)]


class A3cOut(C.Structure):
    _fields_ = [("pi_loss", C.c_float), ("baseline_loss", C.c_float), ("entropy", C.c_float),
                ("learning_rate", C.c_float), ("grad_norm", C.c_float), ("step", C.c_int64)]


class R2d2Config(C.Structure):
    _fields_ = [("batch", C.c_int32), ("seq_len", C.c_int32), ("burn_in", C.c_int32), ("height", C.c_int32),
                ("width", C.c_int32), ("channels", C.c_int32), ("num_action", C.c_int32), ("lstm_size", C.c_int32),
                ("discount_factor", C.c_float), ("learning_rate", C.c_float), ("device", C.c_int32),
                ("num_slots", C.c_int32), ("use_cuda_graph", C.c_int32), ("math_mode", C.c_int32)]


class R2d2Out(C.Structure):
    _fields_ = [("loss", C.c_float), ("grad_norm", C.c_float), ("step", C.c_int64)]


class RingBatch(C.Structure):
    _fields_ = [("state", C.c_void_p), ("reward", C.c_void_p), ("done", C.c_void_p),
                ("behavior_policy", C.c_void_p), ("action", C.c_void_p), ("previous_action", C.c_void_p),
                ("previous_h", C.c_void_p), ("previous_c", C.c_void_p), ("slot", C.c_int32)]


def _load():
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            "%s is missing: build it with `python -m distributed_reinforcement_learning_b200.build` "
            "(there is no CPU fallback)" % LIB_PATH)
    lib = C.CDLL(LIB_PATH)
    vp, i32, i64, f32 = C.c_void_p, C.c_int32, C.c_int64, C.c_float
    sig = {
        "drl_last_error": (C.c_char_p, []),
        "drl_version": (C.c_char_p, []),
        "drl_device_count": (C.c_int, []),
        "drl_learner_create": (C.c_int, [C.POINTER(LearnerConfig), C.POINTER(vp)]),
        "drl_learner_destroy": (C.c_int, [vp]),
        "drl_learner_param_count": (C.c_int, [vp, C.POINTER(i64)]),
        "drl_learner_set_params": (C.c_int, [vp, vp, i64]),
        "drl_learner_get_params": (C.c_int, [vp, vp, i64]),
        "drl_learner_set_opt_state": (C.c_int, [vp, vp, i64, i64]),
        "drl_learner_get_opt_state": (C.c_int, [vp, vp, i64, C.POINTER(i64)]),
        "drl_learner_get_grads": (C.c_int, [vp, vp, i64]),
        "drl_learner_stage": (C.c_int, [vp, i32] + [vp] * 8),
        "drl_learner_step": (C.c_int, [vp, i32, C.POINTER(StepOut)]),
        "drl_learner_step_async": (C.c_int, [vp, i32]),
        "drl_learner_wait": (C.c_int, [vp, C.POINTER(StepOut)]),
        "drl_learner_wait_slot": (C.c_int, [vp, i32, C.POINTER(StepOut)]),
        "drl_learner_forward_backward": (C.c_int, [vp, i32]),
        "drl_learner_grad_bucket": (C.c_int, [vp, C.POINTER(vp), C.POINTER(i64)]),
        "drl_learner_reduced_bucket": (C.c_int, [vp, C.POINTER(vp), C.POINTER(i64)]),
        "drl_learner_apply": (C.c_int, [vp]),
        "drl_learner_stream": (C.c_int, [vp, C.POINTER(vp)]),
        "drl_learner_peer_export": (C.c_int, [vp, vp, i64]),
        "drl_learner_peer_import": (C.c_int, [vp, i32, i32, vp, i64]),
        "drl_learner_peer_disable": (C.c_int, [vp]),
        "drl_learner_forward": (C.c_int, [vp, i32, vp, vp]),
        "drl_learner_taps": (C.c_int, [vp, vp, vp, vp, vp]),
        "drl_learner_read_buffer": (C.c_int, [vp, C.c_char_p, vp, i64]),
        "drl_learner_act": (C.c_int, [vp, i32] + [vp] * 7),
        "drl_learner_profile_step": (C.c_int, [vp, i32, C.c_char_p, i64, vp, i32, C.POINTER(i32)]),
        "drl_debug_gemm": (C.c_int, [i32] * 8 + [vp, vp, vp]),
        "drl_debug_trace": (C.c_int, [vp]),
        "drl_learner_last_step_ms": (C.c_int, [vp, C.POINTER(f32)]),
        "drl_learner_launches_per_step": (C.c_int, [vp, C.POINTER(i32)]),
        "drl_vtrace_from_importance_weights": (C.c_int, [vp] * 5 + [i32, i32, f32, vp, vp]),
        "drl_vtrace_from_importance_weights_dev": (C.c_int, [vp] * 5 + [i32, i32, f32, vp, vp, vp]),
        "drl_vtrace_from_softmax": (C.c_int, [vp] * 7 + [i32, i32, i32, f32, vp, vp]),
        "drl_vtrace_from_softmax_dev": (C.c_int, [vp] * 7 + [i32, i32, i32, f32, vp, vp, vp]),
        "drl_vtrace_loss_sums": (C.c_int, [vp] * 5 + [i32, i32, i32, vp, vp]),
        "drl_ring_create": (C.c_int, [i32] * 9 + [C.POINTER(vp)]),
        "drl_ring_destroy": (C.c_int, [vp]),
        "drl_ring_is_pinned": (C.c_int, [vp]),
        "drl_ring_push": (C.c_int, [vp] + [vp] * 8 + [i32]),
        "drl_ring_pop_batch": (C.c_int, [vp, C.POINTER(RingBatch), i32]),
        "drl_ring_release": (C.c_int, [vp, i32]),
        "drl_ring_size": (C.c_int, [vp]),
        "drl_apex_create": (C.c_int, [C.POINTER(ApexConfig), C.POINTER(vp)]),
        "drl_apex_destroy": (C.c_int, [vp]),
        "drl_apex_param_count": (C.c_int, [vp, C.POINTER(i64)]),
        "drl_apex_set_params": (C.c_int, [vp, i32, vp, i64]),
        "drl_apex_get_params": (C.c_int, [vp, i32, vp, i64]),
        "drl_apex_set_opt_state": (C.c_int, [vp, vp, vp, i64, i64, f32, f32]),
        "drl_apex_get_opt_state": (C.c_int, [vp, vp, vp, i64, C.POINTER(i64), C.POINTER(f32), C.POINTER(f32)]),
        "drl_apex_get_grads": (C.c_int, [vp, vp, i64]),
        "drl_apex_target_to_main": (C.c_int, [vp]),
        "drl_apex_stage": (C.c_int, [vp, i32] + [vp] * 7),
        "drl_apex_step": (C.c_int, [vp, i32, C.POINTER(ApexOut), vp]),
        "drl_apex_step_async": (C.c_int, [vp, i32]),
        "drl_apex_forward_backward": (C.c_int, [vp, i32]),
        "drl_apex_grad_bucket": (C.c_int, [vp, C.POINTER(vp), C.POINTER(i64)]),
        "drl_apex_apply": (C.c_int, [vp, f32]),
        "drl_apex_wait": (C.c_int, [vp, C.POINTER(ApexOut), vp]),
        "drl_apex_td_error": (C.c_int, [vp, i32] + [vp] * 7),
        "drl_apex_act": (C.c_int, [vp, i32, vp, vp, vp]),
        "drl_apex_taps": (C.c_int, [vp] * 6),
        "drl_apex_read_buffer": (C.c_int, [vp, C.c_char_p, vp, i64]),
        "drl_apex_profile_step": (C.c_int, [vp, i32, C.c_char_p, i64, vp, i32, C.POINTER(i32)]),
        "drl_apex_last_step_ms": (C.c_int, [vp, C.POINTER(f32)]),
        "drl_apex_launches_per_step": (C.c_int, [vp, C.POINTER(i32)]),
        "drl_apex_stream": (C.c_int, [vp, C.POINTER(vp)]),
        "drl_a3c_create": (C.c_int, [C.POINTER(A3cConfig), C.POINTER(vp)]),
        "drl_a3c_destroy": (C.c_int, [vp]),
        "drl_a3c_param_count": (C.c_int, [vp, C.POINTER(i64)]),
        "drl_a3c_set_params": (C.c_int, [vp, vp, i64]),
        "drl_a3c_get_params": (C.c_int, [vp, vp, i64]),
        "drl_a3c_set_opt_state": (C.c_int, [vp, vp, vp, i64, i64, f32, f32]),
        "drl_a3c_get_opt_state": (C.c_int, [vp, vp, vp, i64, C.POINTER(i64), C.POINTER(f32), C.POINTER(f32)]),
        "drl_a3c_get_grads": (C.c_int, [vp, vp, i64]),
        "drl_a3c_stage": (C.c_int, [vp, i32] + [vp] * 6),
        "drl_a3c_step": (C.c_int, [vp, i32, C.POINTER(A3cOut)]),
        "drl_a3c_step_async": (C.c_int, [vp, i32]),
        "drl_a3c_forward_backward": (C.c_int, [vp, i32]),
        "drl_a3c_grad_bucket": (C.c_int, [vp, C.POINTER(vp), C.POINTER(i64)]),
        "drl_a3c_apply": (C.c_int, [vp, f32]),
        "drl_a3c_wait": (C.c_int, [vp, C.POINTER(A3cOut)]),
        "drl_a3c_act": (C.c_int, [vp, i32, vp, vp, vp, vp]),
        "drl_a3c_taps": (C.c_int, [vp] * 5),
        "drl_a3c_read_buffer": (C.c_int, [vp, C.c_char_p, vp, i64]),
        "drl_a3c_profile_step": (C.c_int, [vp, i32, C.c_char_p, i64, vp, i32, C.POINTER(i32)]),
        "drl_a3c_stream": (C.c_int, [vp, C.POINTER(vp)]),
        "drl_a3c_launches_per_step": (C.c_int, [vp, C.POINTER(i32)]),
        "drl_r2d2_create": (C.c_int, [C.POINTER(R2d2Config), C.POINTER(vp)]),
        "drl_r2d2_destroy": (C.c_int, [vp]),
        "drl_r2d2_param_count": (C.c_int, [vp, C.POINTER(i64)]),
        "drl_r2d2_set_params": (C.c_int, [vp, i32, vp, i64]),
        "drl_r2d2_get_params": (C.c_int, [vp, i32, vp, i64]),
        "drl_r2d2_set_opt_state": (C.c_int, [vp, vp, vp, i64, i64, f32, f32]),
        "drl_r2d2_get_opt_state": (C.c_int, [vp, vp, vp, i64, C.POINTER(i64), C.POINTER(f32), C.POINTER(f32)]),
        "drl_r2d2_get_grads": (C.c_int, [vp, vp, i64]),
        "drl_r2d2_main_to_target": (C.c_int, [vp]),
        "drl_r2d2_stage": (C.c_int, [vp, i32] + [vp] * 8),
        "drl_r2d2_step": (C.c_int, [vp, i32, C.POINTER(R2d2Out), vp]),
        "drl_r2d2_step_async": (C.c_int, [vp, i32]),
        "drl_r2d2_forward_backward": (C.c_int, [vp, i32]),
        "drl_r2d2_grad_bucket": (C.c_int, [vp, C.POINTER(vp), C.POINTER(i64)]),
        "drl_r2d2_apply": (C.c_int, [vp, f32]),
        "drl_r2d2_wait": (C.c_int, [vp, C.POINTER(R2d2Out), vp]),
        "drl_r2d2_td_error": (C.c_int, [vp, i32] + [vp] * 8),
        "drl_r2d2_act": (C.c_int, [vp, i32] + [vp] * 7),
        "drl_r2d2_taps": (C.c_int, [vp] * 5),
        "drl_r2d2_read_buffer": (C.c_int, [vp, C.c_char_p, vp, i64]),
        "drl_r2d2_profile_step": (C.c_int, [vp, i32, C.c_char_p, i64, vp, i32, C.POINTER(i32)]),
        "drl_r2d2_last_step_ms": (C.c_int, [vp, C.POINTER(f32)]),
        "drl_r2d2_stream": (C.c_int, [vp, C.POINTER(vp)]),
        "drl_r2d2_launches_per_step": (C.c_int, [vp, C.POINTER(i32)]),
        "drl_per_create": (C.c_int, [i64, C.POINTER(vp)]),
        "drl_per_destroy": (C.c_int, [vp]),
        "drl_per_add": (C.c_int, [vp, C.c_double, C.POINTER(i64)]),
        "drl_per_sample": (C.c_int, [vp, i32, vp, vp, vp, vp, vp]),
        "drl_per_update": (C.c_int, [vp, i64, C.c_double]),
        "drl_per_total": (C.c_int, [vp, C.POINTER(C.c_double)]),
        "drl_per_size": (C.c_int, [vp, C.POINTER(i64)]),
        "drl_per_beta": (C.c_int, [vp, C.POINTER(C.c_double)]),
        "drl_apex_replay_create": (C.c_int, [vp, i64, C.c_uint64, C.POINTER(vp)]),
        "drl_apex_replay_destroy": (C.c_int, [vp]),
        "drl_apex_replay_add": (C.c_int, [vp, i32] + [vp] * 6),
        "drl_apex_replay_step_async": (C.c_int, [vp, i32]),
        "drl_apex_replay_step": (C.c_int, [vp, i32, C.POINTER(ApexOut), vp]),
        "drl_apex_replay_last_sample": (C.c_int, [vp] * 5),
        "drl_apex_replay_last_update": (C.c_int, [vp, vp, vp, i32, C.POINTER(i32)]),
        "drl_apex_replay_info": (C.c_int, [vp, C.POINTER(i64), C.POINTER(i64), C.POINTER(C.c_double),
                                           C.POINTER(C.c_double), C.POINTER(i64)]),
        "drl_apex_replay_read_tree": (C.c_int, [vp, vp, i64]),
    }
    for name, (res, args) in sig.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    return lib, sorted(sig)


lib, EXPORTS = _load()


def check(rc):
    if rc != DRL_OK:
        text = lib.drl_last_error().decode("utf-8", "replace")
        if rc == DRL_ERR_TIMEOUT:
            raise TimeoutError_(rc, text)
        raise DrlError(rc, text)


def device_count():
    return int(lib.drl_device_count())


def as_c(arr, dtype, shape=None, name="array"):
    """C-contiguous ndarray of `dtype` (no copy when already so); validates the shape."""
    a = np.ascontiguousarray(arr, dtype=dtype)
    if shape is not None and tuple(a.shape) != tuple(shape):
        raise ValueError("%s: expected shape %s, got %s" % (name, tuple(shape), tuple(a.shape)))
    return a


def ptr(a):
    return C.c_void_p(a.ctypes.data)


def _as_u8(done):
    d = np.asarray(done)
    if d.dtype == np.bool_:
        return np.ascontiguousarray(d).view(np.uint8)      # bool is one byte, 0/1: no copy
    return d.astype(np.uint8, copy=False)


class NativeHandle:
    """What every learner wrapper does the same way through its ``drl_<prefix>_*`` entry points: create and destroy
    the handle, parameters without a scope argument, gradients, named buffers, the per-kernel profile and the step's
    stream, time and launch count."""
    _prefix = None

    def _fn(self, name):
        return getattr(lib, "drl_%s_%s" % (self._prefix, name))

    def _open(self, cfg, num_slots):
        self._h = C.c_void_p()
        check(self._fn("create")(C.byref(cfg), C.byref(self._h)))
        n = C.c_int64()
        check(self._fn("param_count")(self._h, C.byref(n)))
        self.param_count = int(n.value)
        self.num_slots = int(num_slots)
        self._keep = [None] * self.num_slots     # host arrays referenced by in-flight H2D copies

    def close(self):
        if getattr(self, "_h", None) is not None and self._h.value:
            self._fn("destroy")(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_params(self, flat):
        a = as_c(flat, np.float32, (self.param_count,), "params")
        check(self._fn("set_params")(self._h, ptr(a), a.size))

    def get_params(self):
        a = np.empty(self.param_count, np.float32)
        check(self._fn("get_params")(self._h, ptr(a), a.size))
        return a

    def get_grads(self):
        a = np.empty(self.param_count, np.float32)
        check(self._fn("get_grads")(self._h, ptr(a), a.size))
        return a

    def read_buffer(self, name, count):
        a = np.empty(int(count), np.float32)
        check(self._fn("read_buffer")(self._h, name.encode(), ptr(a), a.size))
        return a

    def profile_step(self, slot=0, max_kernels=128):
        """One real step with a CUDA event before every launch -> [(kernel name, device ms)]."""
        names = C.create_string_buffer(8192)
        ms = np.zeros(max_kernels, np.float32)
        cnt = C.c_int32()
        check(self._fn("profile_step")(self._h, slot, names, len(names), ptr(ms), max_kernels, C.byref(cnt)))
        nm = names.value.decode().split("\n") if cnt.value else []
        return list(zip(nm, [float(x) for x in ms[:cnt.value]]))

    def last_step_ms(self):
        ms = C.c_float()
        check(self._fn("last_step_ms")(self._h, C.byref(ms)))
        return float(ms.value)

    def launches_per_step(self):
        n = C.c_int32()
        check(self._fn("launches_per_step")(self._h, C.byref(n)))
        return int(n.value)

    def stream_ptr(self):
        s = C.c_void_p()
        check(self._fn("stream")(self._h, C.byref(s)))
        return int(s.value or 0)
