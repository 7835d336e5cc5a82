"""B200-native stand-in for the reference's ``agent/apex.py``: same constructor kwargs, same methods, same return
values -- so the learner branch of ``train_apex.py:82-155`` runs on it unchanged -- with the TF1 graph +
``tf.Session`` replaced by the CUDA Ape-X learner behind the C-ABI (``drl_apex_*``).

  Agent.__init__              agent/apex.py:12-76
  Agent.target_to_main        agent/apex.py:78-79   (assigns target <- main, as utils.main_to_target does)
  Agent.parameter_sync        agent/apex.py:81-82   (learner -> this agent's variables)
  Agent.set_session           agent/apex.py:84-86   (also initialises every variable, like the reference)
  Agent.get_policy_and_action agent/apex.py:88-102
  Agent.get_td_error          agent/apex.py:116-133
  Agent.distributed_train     agent/apex.py:135-154 -> (loss, td_error)
  Agent.train                 agent/apex.py:156-168
  Agent.make_device_replay    (new) buffer_queue.Memory + the learner calls around it, kept on the GPU
"""
import os
import threading

import numpy as np

from ..apex_learner import MAIN, TARGET, NativeApexLearner, NativeApexReplay
from ..model import apex_value

_AGENTS = {}


class Agent:

    def __init__(self, input_shape, num_action,
                 discount_factor, gradient_clip_norm, reward_clipping,
                 start_learning_rate, end_learning_rate, learning_frame,
                 model_name, learner_name):
        self.input_shape = list(input_shape)
        self.num_action = num_action
        self.discount_factor = discount_factor
        self.gradient_clip_norm = gradient_clip_norm
        self.reward_clipping = reward_clipping
        self.start_learning_rate = start_learning_rate
        self.end_learning_rate = end_learning_rate
        self.learning_frame = learning_frame
        self.model_name = model_name
        self.learner_name = learner_name
        self.device = int(os.environ.get("LOCAL_RANK", "0"))
        self.use_cuda_graph = os.environ.get("DRL_B200_CUDA_GRAPH", "0") == "1"
        self.sess = None
        self._kw = dict(num_action=num_action, input_shape=tuple(input_shape))
        self._main = self._target = None
        self._opt = None
        self._engine = None
        self._slot = 0
        self._last = {}
        self._replay = None
        self._lock = threading.RLock()   # actor threads sync from / act on this agent while the learner thread trains
        _AGENTS[model_name] = self

    # ---- engine management -----------------------------------------------------------
    def _ensure_init(self):
        if self._main is None:
            self._main = apex_value.init_params(**self._kw)
            self._target = apex_value.init_params(**self._kw)        # the two scopes are initialised independently
            z = np.zeros_like(self._main)
            self._opt = dict(m=z, v=z.copy(), step=0, beta1_power=0.9, beta2_power=0.999)

    def _pull_state(self):
        if self._engine is not None:
            self._main = self._engine.get_params(MAIN)
            self._target = self._engine.get_params(TARGET)
            self._opt = self._engine.get_opt_state()

    def _get_engine(self, batch):
        self._ensure_init()
        if self._engine is None or self._engine.B < batch:
            if self._engine is not None:
                self._pull_state()
                self._engine.close()
            self._engine = NativeApexLearner(
                batch=batch, num_action=self.num_action, input_shape=tuple(self.input_shape),
                discount_factor=self.discount_factor, gradient_clip_norm=self.gradient_clip_norm,
                reward_clipping=self.reward_clipping, start_learning_rate=self.start_learning_rate,
                end_learning_rate=self.end_learning_rate, learning_frame=self.learning_frame,
                device=self.device, num_slots=2, use_cuda_graph=self.use_cuda_graph)
            self._push_state()
        return self._engine

    def _push_state(self):
        e = self._engine
        e.set_params(self._main, MAIN)
        e.set_params(self._target, TARGET)
        o = self._opt
        e.set_opt_state(o["m"], o["v"], o["step"], o["beta1_power"], o["beta2_power"])

    # ---- reference API ---------------------------------------------------------------
    def target_to_main(self):
        """agent/apex.py:78-79: runs utils.main_to_target(main, target), i.e. target <- main."""
        self._ensure_init()
        if self._engine is not None:
            self._engine.target_to_main()
        else:
            self._target = self._main.copy()

    def _snapshot_params(self):
        with self._lock:
            self._ensure_init()
            if self._engine is not None:
                return self._engine.get_params(MAIN), self._engine.get_params(TARGET)
            return self._main.copy(), self._target.copy()

    def parameter_sync(self):
        """agent/apex.py:81-82 (utils.copy_src_to_dst(learner_name, model_name)): both scopes are trainable
        variables of the learner, so both are copied."""
        src = _AGENTS.get(self.learner_name)
        if src is None or src is self:
            return
        main, target = src._snapshot_params()            # trainable variables only, into caller-owned buffers
        with self._lock:
            self._ensure_init()
            self._main, self._target = main, target
            if self._engine is not None:
                self._engine.set_params(self._main, MAIN)
                self._engine.set_params(self._target, TARGET)

    def set_session(self, sess):
        self.sess = sess
        self._main = None
        self._ensure_init()
        if self._engine is not None:
            self._push_state()

    def save_weights(self, path):
        self._ensure_init()
        self._pull_state()
        if not path.endswith(".npz"):
            path = path + ".npz"
        o = self._opt
        np.savez(path, main=self._main, target=self._target, m=o["m"], v=o["v"], step=np.int64(o["step"]),
                 beta1_power=np.float32(o["beta1_power"]), beta2_power=np.float32(o["beta2_power"]))

    def load_weights(self, path):
        if not path.endswith(".npz"):
            path = path + ".npz"
        z = np.load(path)
        n = apex_value.param_count(**self._kw)
        if z["main"].size != n:
            raise ValueError("checkpoint has %d parameters per scope, this agent has %d" % (z["main"].size, n))
        self._main, self._target = z["main"].astype(np.float32), z["target"].astype(np.float32)
        self._opt = dict(m=z["m"].astype(np.float32), v=z["v"].astype(np.float32), step=int(z["step"]),
                         beta1_power=float(z["beta1_power"]), beta2_power=float(z["beta2_power"]))
        if self._engine is not None:
            self._push_state()

    @staticmethod
    def _u8(state):
        st = np.asarray(state)
        if st.dtype != np.uint8:
            raise TypeError("states must be uint8 frames (the /255 normalisation runs on the GPU)")
        return st

    def get_policy_and_action(self, state, previous_action, epsilon):
        """agent/apex.py:88-102 -> (action, main_q_value, main_q_value[action])."""
        eng = self._engine if self._engine is not None else self._get_engine(1)
        q = eng.act(self._u8(state)[None], np.asarray([previous_action], np.int32))[0]
        if np.random.rand() > epsilon:
            action = np.argmax(q, axis=0)
        else:
            action = np.random.choice(self.num_action)
        return action, q, q[action]

    def get_td_error(self, state, next_state, previous_action, action, reward, done):
        """agent/apex.py:116-133 -> |target_value - state_action_value| [n]."""
        st = self._u8(np.stack(state))
        # evaluation only: reuse the training engine and go through it in chunks of its batch size; never rebuild it
        # for a larger n (train_apex.py calls this with `trajectory` transitions, which may exceed batch_size)
        eng = self._engine if self._engine is not None else self._get_engine(st.shape[0])
        out = np.empty(st.shape[0], np.float32)
        B = eng.B
        ns = self._u8(np.stack(next_state))
        for lo in range(0, st.shape[0], B):
            hi = min(lo + B, st.shape[0])
            out[lo:hi] = eng.td_error(st[lo:hi], ns[lo:hi], np.asarray(previous_action)[lo:hi],
                                      np.asarray(action)[lo:hi], np.asarray(reward)[lo:hi], np.asarray(done)[lo:hi])
        return out

    def _train(self, state, next_state, previous_action, action, reward, done, is_weight):
        st = self._u8(np.stack(state))
        if self._replay is not None and self._engine.B != st.shape[0]:
            raise ValueError("a device replay of batch %d is attached: training on %d transitions would rebuild the "
                             "learner under it" % (self._engine.B, st.shape[0]))
        if self._engine is not None and self._engine.B != st.shape[0]:
            self._pull_state()
            self._engine.close()
            self._engine = None
        eng = self._get_engine(st.shape[0])
        slot = self._slot
        self._slot = (self._slot + 1) % eng.num_slots
        eng.stage(slot, st, self._u8(np.stack(next_state)), previous_action, action, reward, done, is_weight)
        out, td = eng.step(slot)
        self._last = out
        return out["loss"], td

    def distributed_train(self, state, next_state, previous_action, action, reward, done, is_weight):
        """agent/apex.py:135-154 -> (loss, td_error)."""
        return self._train(state, next_state, previous_action, action, reward, done, is_weight)

    def train(self, state, next_state, previous_action, action, reward, done):
        """agent/apex.py:156-168 (unit importance weights; returns None like the reference)."""
        self._train(state, next_state, previous_action, action, reward, done, None)

    def make_device_replay(self, capacity, batch_size, seed=0):
        """(new) A prioritized replay of `capacity` transitions in this learner's GPU memory, trained on in minibatches
        of `batch_size`.  Its ``add`` replaces get_td_error + the Memory.add loop, its ``train`` replaces Memory.sample +
        distributed_train + the Memory.update loop (train_apex.py:106-155)."""
        with self._lock:
            if self._replay is not None:
                raise RuntimeError("this agent already has a device replay; close it first")
            if self._engine is not None and self._engine.B != int(batch_size):
                self._pull_state()
                self._engine.close()
                self._engine = None
            eng = self._get_engine(int(batch_size))
            self._replay = DeviceReplay(self, NativeApexReplay(eng, capacity, seed))
            return self._replay

    learning_rate = property(lambda self: self._last.get("learning_rate"))
    grad_norm = property(lambda self: self._last.get("grad_norm"))
    value_loss = property(lambda self: self._last.get("loss"))
    num_env_frames = property(lambda self: self._last.get("step", (self._opt or {}).get("step", 0)))


class DeviceReplay:
    """What Agent.make_device_replay returns: the learner loop of train_apex.py:106-155 over a replay in GPU memory.

        replay.add(state, next_state, previous_action, action, reward, done)   # get_td_error + Memory.add, per record
        loss, td_error = replay.train()     # Memory.sample -> distributed_train -> Memory.update
    """

    def __init__(self, agent, native):
        self._agent, self.native = agent, native

    def add(self, state, next_state, previous_action, action, reward, done):
        with self._agent._lock:
            self.native.add(self._agent._u8(np.stack(state)), self._agent._u8(np.stack(next_state)),
                            np.asarray(previous_action), np.asarray(action), np.asarray(reward), np.asarray(done))

    def train(self):
        """-> (loss, td_error [batch]) of one step on a prioritized minibatch; the sampled priorities are updated."""
        a = self._agent
        with a._lock:
            slot = a._slot
            a._slot = (a._slot + 1) % self.native.learner.num_slots
            out, td = self.native.step(slot)
            a._last = out
            return out["loss"], td

    def __len__(self):
        return len(self.native)

    def total(self):
        """SumTree.total (buffer_queue.py:348-349)."""
        return self.native.info()["total"]

    @property
    def beta(self):
        return self.native.info()["beta"]

    def close(self):
        with self._agent._lock:
            self.native.close()
            if self._agent._replay is self:
                self._agent._replay = None


def _locked(fn):
    def wrapper(self, *a, **k):
        with self._lock:
            return fn(self, *a, **k)
    wrapper.__name__, wrapper.__doc__ = fn.__name__, fn.__doc__
    return wrapper


# actor threads call these on a shared agent while the learner thread trains (in-process launch mode)
for _n in ('save_weights', 'load_weights', 'set_session', 'target_to_main', 'get_policy_and_action', 'get_td_error', '_train'):
    if hasattr(Agent, _n):
        setattr(Agent, _n, _locked(getattr(Agent, _n)))
