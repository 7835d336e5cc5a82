"""Runs the UNMODIFIED reference files over the TF1 API stand-in -- TEST INFRASTRUCTURE ONLY.

``load()`` puts ``oracle/tf1_shim`` (a ``tensorflow`` 1.14 API stand-in over torch-CPU, see its docstring for what
is restated) and the reference checkout on ``sys.path`` and imports the reference's own modules
(``agent/impala.py``, ``optimizer/vtrace.py``, ``model/impala_actor_critic.py``, ``agent/apex.py``, ``agent/r2d2.py``,
``distributed_queue/buffer_queue.py`` ...) exactly as they lie under ``/root/reference``: nothing is copied or edited.
This is what pins ``oracle/impala_torch.py`` & co. to the reference itself: ``tests/golden/make_golden.py`` writes
the committed golden vectors from the executed reference, and ``tests/test_oracle_refexec.py`` asserts that the
restatements equal them (losses, V-trace taps, every gradient, the optimizer step).

``DRL_REFERENCE_DIR`` names the reference checkout; the tests do not need one.
"""
import importlib
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
SHIM_DIR = os.path.join(HERE, "tf1_shim")
REFERENCE_DIR = os.environ.get("DRL_REFERENCE_DIR", "/root/reference")

# top-level module names of the reference checkout (they must not leak into / collide with the caller's modules)
_REF_TOP = ("agent", "model", "optimizer", "distributed_queue", "utils", "wrappers")
_SHIM_TOP = ("tensorflow", "gym", "tensorboardX")


def available():
    return os.path.isfile(os.path.join(REFERENCE_DIR, "agent", "impala.py"))


class Reference:
    """Handle on the imported reference modules + the shim (``.tf``)."""

    def __init__(self, modules, tf):
        self.modules = modules
        self.tf = tf

    def __getitem__(self, name):
        return self.modules[name]


def load(names=("agent.impala", "optimizer.vtrace", "model.impala_actor_critic", "utils",
                "distributed_queue.buffer_queue"), float_dtype=None, fresh_graph=True):
    """Imports the named reference modules over the shim and returns a ``Reference``.  The imported modules are
    removed from ``sys.modules`` again (the objects stay alive through the returned handle), so the caller's own
    ``utils``/``agent`` ... are never shadowed."""
    if not available():
        raise FileNotFoundError("reference checkout not found at %s" % REFERENCE_DIR)
    saved_path = list(sys.path)
    saved_mods = {k: sys.modules.pop(k) for k in list(sys.modules)
                  if k.split(".")[0] in _REF_TOP + _SHIM_TOP}
    sys.path[:0] = [SHIM_DIR, REFERENCE_DIR]
    try:
        tf = importlib.import_module("tensorflow")
        assert tf.__version__.endswith("-shim"), "a real tensorflow is importable: use it instead of the shim"
        if float_dtype is not None:
            tf._shim.FLOAT = float_dtype
        if fresh_graph:
            tf.reset_default_graph()
        mods = {n: importlib.import_module(n) for n in names}
        for m in mods.values():
            assert os.path.abspath(m.__file__).startswith(os.path.abspath(REFERENCE_DIR)), m.__file__
    finally:
        sys.path[:] = saved_path
        for k in list(sys.modules):
            if k.split(".")[0] in _REF_TOP + _SHIM_TOP:
                del sys.modules[k]
        sys.modules.update(saved_mods)
    return Reference(mods, tf)


# ----------------------------------------------------------------------------------------------------------------
# IMPALA learner through the reference's own Agent (agent/impala.py:11-148)
# ----------------------------------------------------------------------------------------------------------------
IMPALA_VAR_ORDER = (  # TF1 creation order under <model_name>/impala/ (SURVEY.md App. A.2) -> oracle parameter names
    ("conv2d", "conv1"), ("conv2d_1", "conv2"), ("conv2d_2", "conv3"), ("dense", "emb1"), ("dense_1", "emb2"),
    ("rnn/lstm_cell", "lstm"), ("dense_2", "actor1"), ("dense_3", "actor2"), ("dense_4", "actor3"),
    ("dense_5", "critic1"), ("dense_6", "critic2"), ("dense_7", "critic3"))


class ReferenceImpala:
    """The reference ``impala.Agent`` built with model_name == learner_name == 'learner' (train_impala.py:48-62),
    its variables loaded from an oracle-style parameter dict, and helpers to read back what ``sess.run`` produced."""

    def __init__(self, params, float_dtype=None, **cfg):
        import torch
        from oracle import impala_torch as it
        self.ref = load(float_dtype=float_dtype or torch.float64)
        tf = self.ref.tf
        c = dict(it.DEFAULT_CFG)
        c.update(cfg)
        self.cfg = c
        self.agent = self.ref["agent.impala"].Agent(
            trajectory=c["trajectory"], input_shape=list(c["input_shape"]), num_action=c["num_action"],
            lstm_hidden_size=c["lstm_hidden_size"], discount_factor=c["discount_factor"],
            start_learning_rate=c["start_learning_rate"], end_learning_rate=c["end_learning_rate"],
            learning_frame=c["learning_frame"], baseline_loss_coef=c["baseline_loss_coef"],
            entropy_coef=c["entropy_coef"], gradient_clip_norm=c["gradient_clip_norm"],
            reward_clipping=c["reward_clipping"], model_name="learner", learner_name="learner")
        self.sess = tf.Session()
        self.agent.set_session(self.sess)                       # runs global_variables_initializer
        self.var = {}
        names = [v.op_name for v in tf.trainable_variables()]
        expect = []
        for tf_name, our in IMPALA_VAR_ORDER:
            expect += ["learner/impala/%s/kernel" % tf_name, "learner/impala/%s/bias" % tf_name]
            self.var[our + ".w"] = tf.get_default_graph().var_by_name["learner/impala/%s/kernel" % tf_name]
            self.var[our + ".b"] = tf.get_default_graph().var_by_name["learner/impala/%s/bias" % tf_name]
        assert names == expect, "variable creation order differs from SURVEY App. A.2: %r" % (names,)
        for n, v in params.items():
            assert tuple(self.var[n]._shape) == tuple(v.shape), (n, self.var[n]._shape, tuple(v.shape))
            self.var[n].set(v.detach().to(torch.float32).numpy())

    def feed(self, state, reward, action, done, behavior_policy, previous_action, initial_h, initial_c):
        """The feed_dict of Agent.train (agent/impala.py:133-142), for fetching graph attributes without training."""
        import numpy as np
        a = self.agent
        return {a.t_s_ph: np.stack(state) / 255, a.t_pa_ph: previous_action, a.t_initial_h_ph: initial_h,
                a.t_initial_c_ph: initial_c, a.a_ph: action, a.d_ph: done, a.r_ph: reward, a.b_ph: behavior_policy}

    def fetch(self, batch_args, names):
        a = self.agent
        return dict(zip(names, self.sess.run([getattr(a, n) for n in names], feed_dict=self.feed(*batch_args))))

    def gradients(self, batch_args):
        """d total_loss / d variable for all 24 variables (tf.gradients on the agent's own total_loss)."""
        tf = self.ref.tf
        if not hasattr(self, "_grad_nodes"):
            self._grad_nodes = tf.gradients(self.agent.total_loss, [self.var[n] for n in self.var])
        vals = self.sess.run(self._grad_nodes, feed_dict=self.feed(*batch_args))
        return dict(zip(self.var, vals))

    def train(self, *batch_args):
        return self.agent.train(*batch_args)

    def params(self):
        return {n: v.numpy() for n, v in self.var.items()}

    def rms(self):
        return {n: self.agent.optimizer.get_slot(v, "rms").numpy() for n, v in self.var.items()}

    def global_step(self):
        return int(self.agent.num_env_frames.numpy())


# ----------------------------------------------------------------------------------------------------------------
# Ape-X and R2D2 learners through the reference's own Agents (agent/apex.py:11-168, agent/r2d2.py:12-159)
# ----------------------------------------------------------------------------------------------------------------
APEX_VAR_ORDER = (("conv2d", "conv1"), ("conv2d_1", "conv2"), ("conv2d_2", "conv3"), ("dense", "emb1"),
                  ("dense_1", "emb2"), ("dense_2", "value1"), ("dense_3", "value2"), ("dense_4", "value3"),
                  ("dense_5", "mean1"), ("dense_6", "mean2"), ("dense_7", "mean3"))
R2D2_VAR_ORDER = (("conv2d", "conv1"), ("conv2d_1", "conv2"), ("conv2d_2", "conv3"), ("dense", "emb1"),
                  ("dense_1", "emb2"), ("rnn/lstm_cell", "lstm"), ("dense_2", "q1"), ("dense_3", "value"),
                  ("dense_4", "mean"))


class _TwoScopeAgent:
    """Shared plumbing of the two double-network agents: variables under learner/main and learner/target."""
    ORDER = ()

    def _bind(self, params, target_params):
        import torch
        tf = self.ref.tf
        g = tf.get_default_graph()
        self.var, self.tvar = {}, {}
        expect = []
        for scope, dst in (("main", self.var), ("target", self.tvar)):
            for tf_name, our in self.ORDER:
                for kind, suffix in (("kernel", ".w"), ("bias", ".b")):
                    full = "learner/%s/%s/%s" % (scope, tf_name, kind)
                    expect.append(full)
                    dst[our + suffix] = g.var_by_name[full]
        names = [v.op_name for v in tf.trainable_variables()]
        assert names == expect, "variable creation order differs from the oracle's parameter order: %r" % (names,)
        for dst, src in ((self.var, params), (self.tvar, target_params)):
            for n, v in src.items():
                assert tuple(dst[n]._shape) == tuple(v.shape), (n, dst[n]._shape, tuple(v.shape))
                dst[n].set(v.detach().to(torch.float32).numpy())

    def params(self):
        return {n: v.numpy() for n, v in self.var.items()}

    def target_params(self):
        return {n: v.numpy() for n, v in self.tvar.items()}

    def adam_slots(self):
        opt = self.agent.optimizer
        return ({n: opt.get_slot(v, "m").numpy() for n, v in self.var.items()},
                {n: opt.get_slot(v, "v").numpy() for n, v in self.var.items()})

    def gradients(self, feed):
        tf = self.ref.tf
        if not hasattr(self, "_grad_nodes"):
            self._grad_nodes = tf.gradients(self.agent.value_loss, [self.var[n] for n in self.var])
        return dict(zip(self.var, self.sess.run(self._grad_nodes, feed_dict=feed)))


class ReferenceApex(_TwoScopeAgent):
    ORDER = APEX_VAR_ORDER

    def __init__(self, params, target_params, float_dtype=None, **cfg):
        import torch
        from oracle import apex_torch as ax
        self.ref = load(("agent.apex", "model.apex_value", "optimizer.dqn", "utils"),
                        float_dtype=float_dtype or torch.float64)
        c = dict(ax.DEFAULT_CFG)
        c.update(cfg)
        self.cfg = c
        self.agent = self.ref["agent.apex"].Agent(
            input_shape=list(c["input_shape"]), num_action=c["num_action"], discount_factor=c["discount_factor"],
            gradient_clip_norm=c["gradient_clip_norm"], reward_clipping=c["reward_clipping"],
            start_learning_rate=c["start_learning_rate"], end_learning_rate=c["end_learning_rate"],
            learning_frame=c["learning_frame"], model_name="learner", learner_name="learner")
        self.sess = self.ref.tf.Session()
        self.agent.set_session(self.sess)
        self._bind(params, target_params)

    def feed(self, state, next_state, previous_action, action, reward, done, is_weight):
        """feed_dict of distributed_train (agent/apex.py:137-149)."""
        import numpy as np
        a = self.agent
        return {a.state_ph: np.stack(state) / 255, a.next_state_ph: np.stack(next_state) / 255,
                a.previous_action_ph: previous_action, a.action_ph: action, a.reward_ph: reward, a.done_ph: done,
                a.weight_ph: is_weight}

    def fetch(self, batch_args, names):
        a = self.agent
        return dict(zip(names, self.sess.run([getattr(a, n) for n in names], feed_dict=self.feed(*batch_args))))


class ReferenceR2D2(_TwoScopeAgent):
    ORDER = R2D2_VAR_ORDER

    def __init__(self, params, target_params, float_dtype=None, **cfg):
        import torch
        from oracle import r2d2_torch as rt
        self.ref = load(("agent.r2d2", "model.r2d2_lstm", "optimizer.burn_in", "utils"),
                        float_dtype=float_dtype or torch.float64)
        c = dict(rt.DEFAULT_CFG)
        c.update(cfg)
        self.cfg = c
        self.agent = self.ref["agent.r2d2"].Agent(
            seq_len=c["seq_len"], burn_in=c["burn_in"], input_shape=list(c["input_shape"]),
            num_action=c["num_action"], lstm_size=c["lstm_size"], discount_factor=c["discount_factor"],
            start_learning_rate=c.get("start_learning_rate", 1e-4), end_learning_rate=c.get("end_learning_rate", 0.0),
            learning_frame=c.get("learning_frame", 1), gradient_clip_norm=c.get("gradient_clip_norm", 40.0),
            model_name="learner", learner_name="learner")
        self.sess = self.ref.tf.Session()
        self.agent.set_session(self.sess)
        self._bind(params, target_params)

    def feed(self, state, previous_action, action, h, c, reward, done, weight):
        """feed_dict of Agent.train (agent/r2d2.py:134-152)."""
        import numpy as np
        a = self.agent
        return {a.main_s_ph: np.stack(state) / 255, a.main_h_ph: np.stack(h)[:, 0], a.main_c_ph: np.stack(c)[:, 0],
                a.main_d_ph: done, a.main_pa_ph: previous_action, a.target_s_ph: np.stack(state) / 255,
                a.target_h_ph: np.stack(h)[:, 0], a.target_c_ph: np.stack(c)[:, 0], a.target_d_ph: done,
                a.target_pa_ph: previous_action, a.reward_ph: reward, a.done_ph: done, a.action_ph: action,
                a.weight_ph: weight}

    def fetch(self, batch_args, names):
        a = self.agent
        return dict(zip(names, self.sess.run([getattr(a, n) for n in names], feed_dict=self.feed(*batch_args))))


# ----------------------------------------------------------------------------------------------------------------
# A3C learner through the reference's own Agent (agent/a3c.py:9-103): one scope <model_name>/a3c, variables shared by
# network(s, a_prev) and network(s', a) (model/actor_critic.py:41-56)
# ----------------------------------------------------------------------------------------------------------------
A3C_VAR_ORDER = (("conv2d", "conv1"), ("conv2d_1", "conv2"), ("conv2d_2", "conv3"), ("dense", "emb1"),
                 ("dense_1", "emb2"), ("dense_2", "actor1"), ("dense_3", "actor2"), ("dense_4", "actor3"),
                 ("dense_5", "critic1"), ("dense_6", "critic2"), ("dense_7", "critic3"))


class ReferenceA3C:
    def __init__(self, params, float_dtype=None, **cfg):
        import torch
        from oracle import a3c_torch as a3
        self.ref = load(("agent.a3c", "model.actor_critic", "optimizer.a2c", "utils"),
                        float_dtype=float_dtype or torch.float64)
        tf = self.ref.tf
        c = dict(a3.DEFAULT_CFG)
        c.update(cfg)
        self.cfg = c
        self.agent = self.ref["agent.a3c"].Agent(
            input_shape=list(c["input_shape"]), num_action=c["num_action"], discount_factor=c["discount_factor"],
            start_learning_rate=c["start_learning_rate"], end_learning_rate=c["end_learning_rate"],
            learning_frame=c["learning_frame"], baseline_loss_coef=c["baseline_loss_coef"],
            entropy_coef=c["entropy_coef"], gradient_clip_norm=c["gradient_clip_norm"],
            reward_clipping=c["reward_clipping"], model_name="learner", learner_name="learner")
        self.sess = tf.Session()
        self.agent.set_session(self.sess)
        self.var, expect = {}, []
        for tf_name, our in A3C_VAR_ORDER:
            for kind, suffix in (("kernel", ".w"), ("bias", ".b")):
                full = "learner/a3c/%s/%s" % (tf_name, kind)
                expect.append(full)
                self.var[our + suffix] = tf.get_default_graph().var_by_name[full]
        names = [v.op_name for v in tf.trainable_variables()]
        assert names == expect, "variable creation order differs from the oracle's parameter order: %r" % (names,)
        for n, v in params.items():
            assert tuple(self.var[n]._shape) == tuple(v.shape), (n, self.var[n]._shape, tuple(v.shape))
            self.var[n].set(v.detach().to(torch.float32).numpy())

    def feed(self, state, next_state, previous_action, action, reward, done):
        """feed_dict of Agent.train (agent/a3c.py:86-101): next_previous_action = action."""
        import numpy as np
        a = self.agent
        return {a.s_ph: np.stack(state) / 255, a.ns_ph: np.stack(next_state) / 255, a.pa_ph: previous_action,
                a.npa_ph: action, a.a_ph: action, a.r_ph: reward, a.d_ph: done}

    def fetch(self, batch_args, names):
        a = self.agent
        return dict(zip(names, self.sess.run([getattr(a, n) for n in names], feed_dict=self.feed(*batch_args))))

    def gradients(self, batch_args):
        tf = self.ref.tf
        if not hasattr(self, "_grad_nodes"):
            self._grad_nodes = tf.gradients(self.agent.total_loss, [self.var[n] for n in self.var])
        return dict(zip(self.var, self.sess.run(self._grad_nodes, feed_dict=self.feed(*batch_args))))

    def params(self):
        return {n: v.numpy() for n, v in self.var.items()}

    def adam_slots(self):
        opt = self.agent.optimizer
        return ({n: opt.get_slot(v, "m").numpy() for n, v in self.var.items()},
                {n: opt.get_slot(v, "v").numpy() for n, v in self.var.items()})
