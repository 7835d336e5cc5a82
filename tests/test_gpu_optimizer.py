"""The update kernels of the learners (csrc/optimizer.cu) against a float64 restatement of the TF 1.14 update tails,
at inputs where each branch acts: global-norm clipping engaged and not, norm 0, heavy-tailed gradients, a single
nonzero at either end of the flat vector, the learning-rate decay past its end, a restored int64 step with a nonzero
high word, and the data-parallel ``grad_scale`` of the Adam learners.

Most tests drive the update in isolation.  The gradient bucket ``[padded grads | loss sums | pad]`` that
``drl_<family>_grad_bucket`` exposes is exactly what the update reads, so a test stages a batch, runs
``forward_backward``, overwrites the bucket with a chosen vector on the learner's stream and calls ``apply``.  The
packed <-> padded map of the bucket is learnt from the device (``probe_layout``).

Tolerances follow from the float32 error of the kernels, not from measurement.  The elementwise reference is built from
the norm the GPU reported, and that norm is checked on its own against the float64 norm of the float32 bucket (1e-5
relative), which separates the reduction error from the elementwise error.  Slots: 4 float32 ulps of the terms they
are summed from.  Parameters: ``4 eps |w0| + 16 eps |dw_ref|`` (RMSProp uses rsqrtf, within 2 ulp), plus, for Adam
with a restored first moment, 4 ulps of ``|m0| * alpha / (sqrt(v) + eps)`` for the cancellation in ``m``.

Run with ``-s`` to see the worst error / tolerance ratio of each check.
"""
import ctypes as C
import functools

import numpy as np
import pytest
import torch

import apex_parity as ap
import parity
from oracle import a3c_torch as at
from oracle import apex_torch as ax
from oracle import impala_torch as it
from oracle import r2d2_torch as rt
from oracle import synthetic

EPS = float(np.finfo(np.float32).eps)
F32 = np.float32
# TF keeps the decay constants as float32 tensors and forms 1 - rho / 1 - beta in float32, as the kernels do
ONE_MINUS_RHO = float(F32(1.0) - F32(0.99))
ONE_MINUS_B1 = float(F32(1.0) - F32(ax.BETA1))
ONE_MINUS_B2 = float(F32(1.0) - F32(ax.BETA2))
TAIL = np.array([1.25, 0.75, -2.5], np.float32)       # loss sums written behind the injected gradients

ADAM = ("apex", "a3c", "r2d2")
FAMILIES = ("impala",) + ADAM
REGIMES = ("below_clip", "above_clip", "zero", "heavy_tailed", "first_only", "last_only")


# ---- float64 reference of the update tails ------------------------------------------------------------------------
polynomial_decay_f32 = it.polynomial_decay_f32


def clip_scale(norm, clip):
    """tf.clip_by_global_norm's factor clip * min(1/norm, 1/clip); 1 for norm 0 and, for Adam, for clip <= 0."""
    if clip <= 0 or norm == 0:
        return 1.0
    return clip * min(1.0 / norm, 1.0 / clip)


def adam_alpha_f32(lr, b1p, b2p):
    """ApplyAdam's lr * sqrt(1 - beta2_power) / (1 - beta1_power), in float32 like TF."""
    return float(F32(lr) * np.sqrt(F32(1.0) - F32(b2p)) / (F32(1.0) - F32(b1p)))


def rmsprop_ref(w0, ms0, g, scale, lr, one_minus_rho=ONE_MINUS_RHO):
    """-> (w, ms): ms += (g^2 - ms)(1 - rho); w -= lr g / sqrt(ms + 0.1), g = scale * g (float64, elementwise)."""
    gc = np.asarray(g, np.float64) * scale
    ms = ms0 + (gc * gc - ms0) * one_minus_rho
    return w0 - lr * gc / np.sqrt(ms + 0.1), ms


def adam_ref(w0, m0, v0, g, scale, alpha, one_minus_b1=ONE_MINUS_B1, one_minus_b2=ONE_MINUS_B2):
    """-> (w, m, v) of ApplyAdam on g = scale * g (float64, elementwise).  For the data-parallel update ``scale``
    includes grad_scale: adam_apply_kernel clips g * grad_scale by its norm ||g|| * grad_scale."""
    gc = np.asarray(g, np.float64) * scale
    m = m0 + (gc - m0) * one_minus_b1
    v = v0 + (gc * gc - v0) * one_minus_b2
    return w0 - m * alpha / (np.sqrt(v) + ax.ADAM_EPS), m, v


def test_reference_reproduces_impala_oracle_update_with_clipping():
    """The reference tail equals one oracle.impala_torch.Learner.train update (RMSProp) with clipping engaged."""
    B, T, A, clip = 2, 5, 6, 0.05
    batch = synthetic.make_batch(B, T=T, A=A, seed=5)
    args = [batch[k] for k in synthetic.TRAIN_FIELDS]
    L = it.Learner(it.init_params(0, torch.float32, num_action=A), torch.float64, trajectory=T, num_action=A,
                   gradient_clip_norm=clip, learning_frame=3, end_learning_rate=1e-5)
    L.step = 1
    w0 = {n: p.detach().numpy().copy() for n, p in L.params.items()}
    ms0 = {n: v.numpy().copy() for n, v in L.ms.items()}
    res, _, g, gn = L.train(*args, return_all=True)
    assert gn > 4 * clip                                                     # clipping engaged
    lr = polynomial_decay_f32(6e-4, 1, 3, 1e-5)
    assert res[3] == float(lr)
    for n in L.params:
        w, ms = rmsprop_ref(w0[n], ms0[n], g[n].numpy(), clip_scale(gn, clip), float(lr), one_minus_rho=1.0 - 0.99)
        np.testing.assert_allclose(L.ms[n].numpy(), ms, rtol=1e-12, atol=0)
        dw = L.params[n].detach().numpy() - w0[n]
        assert np.max(np.abs(dw - (w - w0[n]))) <= 1e-12 * max(np.max(np.abs(dw)), 1e-30), n


def test_reference_reproduces_apex_oracle_update_with_clipping():
    """The reference tail equals one oracle.apex_torch.Learner.distributed_train update (Adam) with clipping engaged."""
    B, A, clip = 3, 4, 0.05
    b = ax.make_transitions(B, A=A, seed=8)
    L = ax.Learner(ax.init_params(0, torch.float32, num_action=A), ax.init_params(1, torch.float32, num_action=A),
                   torch.float64, num_action=A, gradient_clip_norm=clip, learning_frame=3, end_learning_rate=1e-5)
    rng = np.random.default_rng(0)
    with torch.no_grad():                                                   # a restored, nonzero Adam state
        for n in L.params:
            L.m[n].copy_(torch.from_numpy(rng.standard_normal(tuple(L.m[n].shape)) * 1e-3))
            L.v[n].copy_(torch.from_numpy(rng.uniform(1e-8, 1e-6, tuple(L.v[n].shape))))
    L.step, L.beta1_power, L.beta2_power = 2, F32(0.9 ** 3), F32(0.999 ** 3)
    w0 = {n: p.detach().numpy().copy() for n, p in L.params.items()}
    m0 = {n: v.numpy().copy() for n, v in L.m.items()}
    v0 = {n: v.numpy().copy() for n, v in L.v.items()}
    b1p, b2p = float(L.beta1_power), float(L.beta2_power)
    _, _, g, gn, lr = L.distributed_train(*[b[k] for k in ax.TRAIN_FIELDS], return_all=True)
    assert gn > 4 * clip
    assert lr == float(polynomial_decay_f32(1e-4, 2, 3, 1e-5))
    # the oracle forms alpha and 1 - beta in float64; TF and the kernels in float32 (adam_alpha_f32, ONE_MINUS_B*)
    alpha = lr * np.sqrt(1.0 - b2p) / (1.0 - b1p)
    assert abs(adam_alpha_f32(lr, b1p, b2p) - alpha) <= 2 * EPS * alpha
    for n in L.params:
        w, m, v = adam_ref(w0[n], m0[n], v0[n], g[n].numpy(), clip_scale(gn, clip), alpha,
                           one_minus_b1=1.0 - ax.BETA1, one_minus_b2=1.0 - ax.BETA2)
        np.testing.assert_allclose(L.m[n].numpy(), m, rtol=1e-12, atol=1e-20)
        np.testing.assert_allclose(L.v[n].numpy(), v, rtol=1e-12, atol=0)
        dw = L.params[n].detach().numpy() - w0[n]
        assert np.max(np.abs(dw - (w - w0[n]))) <= 1e-12 * max(np.max(np.abs(dw)), 1e-30), n
    assert L.beta1_power == F32(F32(b1p) * F32(ax.BETA1)) and L.beta2_power == F32(F32(b2p) * F32(ax.BETA2))


# ---- the learners behind one interface ----------------------------------------------------------------------------
START_LR = {"impala": 6e-4, "apex": 1e-4, "a3c": 1e-4, "r2d2": 1e-4}


class Engine:
    """One learner handle with a staged batch and the calls the update tests need.  ``clip``, ``learning_frame``
    and ``end_lr`` are the learner's configuration; R2D2 has neither clipping nor decay (clip 0, start == end)."""

    def __init__(self, family, B=2, clip=40.0, learning_frame=1e9, end_lr=0.0, **kw):
        import distributed_reinforcement_learning_b200._native as N
        self.N = N
        self.family = family
        self.start_lr = START_LR[family]
        if family == "r2d2":
            clip, learning_frame, end_lr = 0.0, 1.0, self.start_lr
        self.clip, self.learning_frame, self.end_lr = clip, learning_frame, end_lr
        sched = dict(gradient_clip_norm=clip, learning_frame=learning_frame, start_learning_rate=self.start_lr,
                     end_learning_rate=end_lr)
        if family == "impala":
            from distributed_reinforcement_learning_b200.learner import NativeLearner
            A, T = 18, 5
            kw.setdefault("use_cuda_graph", False)
            self.eng = NativeLearner(batch=B, trajectory=T, num_action=A, **sched, **kw)
            self.eng.set_params(it.flatten_params(it.init_params(0, torch.float32, num_action=A)))
            b = synthetic.make_batch(B, T=T, A=A, seed=11)
            self._args = [b[k] for k in synthetic.TRAIN_FIELDS]
        elif family == "r2d2":
            from distributed_reinforcement_learning_b200.r2d2_learner import NativeR2D2Learner
            kwp = dict(num_action=4, lstm_size=64, input_shape=(84, 84, 1))
            self.eng = NativeR2D2Learner(batch=B, seq_len=4, burn_in=1, learning_rate=self.start_lr, **kwp, **kw)
            self.eng.set_params(rt.flatten_params(rt.init_params(0, torch.float32, **kwp)), 0)
            self.eng.set_params(rt.flatten_params(rt.init_params(1, torch.float32, **kwp)), 1)
            b = rt.make_sequences(B, S=4, seed=12)
            self._args = [b["state"], b["previous_action"], b["action"], b["h"][:, 0], b["c"][:, 0], b["reward"],
                          b["done"], b["weight"]]
        else:
            from distributed_reinforcement_learning_b200.a3c_learner import NativeA3CLearner
            from distributed_reinforcement_learning_b200.apex_learner import NativeApexLearner
            b = ax.make_transitions(B, A=4, seed=13)
            if family == "apex":
                self.eng = NativeApexLearner(batch=B, num_action=4, **sched, **kw)
                self.eng.set_params(ax.flatten_params(ax.init_params(1, torch.float32, num_action=4)), 1)
                self._args = [b[k] for k in ax.TRAIN_FIELDS]
            else:
                self.eng = NativeA3CLearner(batch=B, num_action=4, **sched, **kw)
                self._args = [b[k] for k in ax.TRAIN_FIELDS[:-1]]
            self.eng.set_params(ax.flatten_params(ax.init_params(0, torch.float32, num_action=4)))
        self.packed = self.eng.param_count
        self.eng.stage(0, *self._args)
        self.forward_backward()
        if family == "impala":
            self.bucket = self.eng.bucket_tensor()
            self.stream = self.eng._ext_stream
        else:
            self.bucket = self.eng._dp._tensor()
            self.stream = self.eng._dp._stream
        self.padded = self.bucket.numel() - 4
        self.map = probe_layout(self)
        self.initial = self.state()

    def forward_backward(self):
        if self.family == "impala":
            self.eng.forward_backward(0)
        else:
            self.N.check(self.eng._fn("forward_backward")(self.eng._h, 0))

    def write(self, vec):
        """vec -> the device bucket, in order on the learner's stream"""
        with torch.cuda.stream(self.stream):
            self.bucket.copy_(torch.from_numpy(np.ascontiguousarray(vec, np.float32)).to(self.bucket.device))

    def read(self):
        torch.cuda.synchronize(self.bucket.device)
        return self.bucket.cpu().numpy()

    def apply(self, grad_scale=1.0):
        if self.family == "impala":
            assert grad_scale == 1.0
            self.eng.apply()
        else:
            self.N.check(self.eng._fn("apply")(self.eng._h, C.c_float(grad_scale)))

    def wait(self):
        out = self.eng.wait()
        return dict(out[0] if isinstance(out, tuple) else out)

    def state(self):
        if self.family == "impala":
            ms, step = self.eng.get_opt_state()
            return dict(params=self.eng.get_params(), slots=(ms,), step=step)
        s = self.eng.get_opt_state()
        return dict(params=self.eng.get_params(), slots=(s["m"], s["v"]), step=s["step"], b1p=s["beta1_power"],
                    b2p=s["beta2_power"])

    def restore(self, st):
        self.eng.set_params(st["params"])
        if self.family == "impala":
            self.eng.set_opt_state(st["slots"][0], st["step"])
        else:
            self.eng.set_opt_state(st["slots"][0], st["slots"][1], st["step"], st["b1p"], st["b2p"])

    def lr_at(self, step):
        return float(polynomial_decay_f32(self.start_lr, step, self.learning_frame, self.end_lr))

    def place(self, g_packed, tail=TAIL):
        """packed gradients -> a full bucket: gradients at their padded offsets, pad lanes 0, the loss sums behind"""
        b = np.zeros(self.padded + 4, np.float32)
        b[self.map] = g_packed
        b[self.padded:self.padded + 3] = tail
        return b

    def close(self):
        self.eng.close()


def probe_layout(E):
    """The packed -> padded map of the bucket, read from the device: arange(padded) (exact in float32 below 2^24)
    written into the bucket and read back through get_grads."""
    assert E.padded < 2 ** 24 and E.padded % 4 == 0
    E.write(np.arange(E.padded + 4, dtype=np.float32))
    got = E.eng.get_grads()
    idx = got.astype(np.int64)
    assert np.array_equal(idx.astype(np.float32), got) and np.all(np.diff(idx) > 0) and idx[-1] < E.padded
    assert E.padded - E.packed < 4 * 24                                      # at most 3 pad lanes per bias
    E.write(np.zeros(E.padded + 4, np.float32))      # pad lanes back to 0: the backward pass writes only real lanes
    return idx


WORST = {}


def _note(key, ratio):
    WORST[key] = max(WORST.get(key, 0.0), float(ratio))


@pytest.fixture(scope="module", autouse=True)
def _report():
    yield
    if WORST:
        print("\nworst error / tolerance (or relative error for norm/*):")
        for k in sorted(WORST):
            print("  %-40s %.3g" % (k, WORST[k]))


_ENGINES = {}


@pytest.fixture(scope="module")
def engines(native):
    """Engine(family, **cfg), created once per configuration in this module; each test restores its own state."""
    def get(family, **cfg):
        key = (family,) + tuple(sorted(cfg.items()))
        if key not in _ENGINES:
            _ENGINES[key] = Engine(family, **cfg)
        return _ENGINES[key]
    yield get
    for e in _ENGINES.values():
        e.close()
    _ENGINES.clear()


def make_gradient(E, regime, rng):
    n = E.packed
    ref = E.clip if E.clip > 0 else 40.0       # R2D2: the norms another learner would clip at
    g = np.zeros(n)
    if regime in ("below_clip", "above_clip"):
        g = rng.standard_normal(n)
        g *= (0.05 if regime == "below_clip" else 1e3) * ref / np.linalg.norm(g)
    elif regime == "heavy_tailed":
        g = 10.0 ** rng.uniform(-8, 2, n) * rng.choice([-1.0, 1.0], n)
    elif regime == "first_only":
        g[0] = 2.5 * ref
    elif regime == "last_only":
        g[-1] = -2.5 * ref
    else:
        assert regime == "zero"
    return g.astype(np.float32)


def apply_and_check(E, bucket, grad_scale=1.0, tag=""):
    """bucket -> device, apply, wait; then every reported scalar, the slots and the parameters against the float64
    reference from the state before.  Returns (scalars, state after)."""
    st0 = E.state()
    E.write(bucket)
    E.apply(grad_scale)
    out = E.wait()
    st1 = E.state()
    tag = E.family + (":" + tag if tag else "")
    gs = float(F32(grad_scale))
    NP = E.padded
    g = bucket[E.map].astype(np.float64)
    norm64 = float(np.sqrt(np.sum(bucket[:NP].astype(np.float64) ** 2))) * gs
    if norm64 == 0.0:
        assert out["grad_norm"] == 0.0
    else:
        rel = abs(out["grad_norm"] - norm64) / norm64
        _note("norm/" + E.family, rel)
        assert rel <= 1e-5, (tag, out["grad_norm"], norm64)
    assert out["step"] == st0["step"] + 1 and st1["step"] == st0["step"] + 1, (tag, out["step"], st0["step"])
    lr = E.lr_at(st0["step"])
    if "learning_rate" in out:
        assert abs(out["learning_rate"] - lr) <= 2 * np.spacing(F32(lr)), (tag, out["learning_rate"], lr)
    tail = bucket[NP:NP + 3]
    if E.family == "impala":
        assert (out["pi_loss"], out["baseline_loss"], out["entropy"]) == tuple(float(x) for x in tail)
        total = float(tail[0]) + float(tail[1]) * 1.0 + float(tail[2]) * float(F32(0.05))   # coefs of the config
        assert abs(out["total_loss"] - total) <= 4 * EPS * (abs(tail[0]) + abs(tail[1]) + abs(tail[2])), tag
    elif E.family == "a3c":
        assert (out["pi_loss"], out["baseline_loss"], out["entropy"]) == tuple(float(x * F32(gs)) for x in tail)
    else:
        assert out["loss"] == float(tail[0] * F32(gs)), (tag, out["loss"], tail[0], gs)
    scale = clip_scale(float(out["grad_norm"]), E.clip) * gs
    w0 = st0["params"].astype(np.float64)
    s0 = [s.astype(np.float64) for s in st0["slots"]]
    if E.family == "impala":
        w, ms = rmsprop_ref(w0, s0[0], g, scale, lr)
        slots = (ms,)
        extra = 0.0
        terms = (np.abs(s0[0]) + (g * scale) ** 2 * ONE_MINUS_RHO,)
    else:
        alpha = adam_alpha_f32(lr, st0["b1p"], st0["b2p"])
        w, m, v = adam_ref(w0, s0[0], s0[1], g, scale, alpha)
        slots = (m, v)
        extra = 4 * EPS * np.abs(s0[0]) * alpha / (np.sqrt(v) + ax.ADAM_EPS)
        gc = np.abs(g * scale)
        terms = (np.abs(s0[0]) + gc * ONE_MINUS_B1, np.abs(s0[1]) + gc * gc * ONE_MINUS_B2)
        assert st1["b1p"] == float(F32(st0["b1p"]) * F32(ax.BETA1)), tag
        assert st1["b2p"] == float(F32(st0["b2p"]) * F32(ax.BETA2)), tag
    for i, (got, ref, t) in enumerate(zip(st1["slots"], slots, terms)):
        tol = np.maximum(4 * EPS * (t + np.abs(ref)), np.finfo(np.float32).tiny)
        r = np.abs(got - ref) / tol
        _note("slot%d/%s" % (i, E.family), r.max())
        assert r.max() <= 1.0, (tag, "slot", i, int(np.argmax(r)), got[np.argmax(r)], ref[np.argmax(r)])
    tol = np.maximum(4 * EPS * np.abs(w0) + 16 * EPS * np.abs(w - w0) + extra, np.finfo(np.float32).tiny)
    r = np.abs(st1["params"] - w) / tol
    _note("params/" + E.family, r.max())
    k = int(np.argmax(r))
    assert r.max() <= 1.0, (tag, "params", k, st1["params"][k], w[k], w0[k])
    return out, st1


# ---- the bucket and its layout ------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("family,mode", [("impala", m) for m in (1, 2, 3, 4, 5)] +
                         [(f, m) for f in ADAM for m in (1, 2)])
def test_bucket_pad_lanes_are_zero_after_backward(native, family, mode):
    """Pad lanes of the bucket would enter the clip norm: a real forward_backward leaves every one exactly 0, and
    writes every gradient lane and the loss sum."""
    E = Engine(family, math_mode=mode)
    try:
        E.write(E.place(np.full(E.packed, np.nan, np.float32), np.array([np.nan, 0, 0], np.float32)))
        E.forward_backward()
        b = E.read()
        pad = np.ones(E.padded, bool)
        pad[E.map] = False
        assert pad.sum() == E.padded - E.packed
        assert np.all(b[:E.padded][pad] == 0.0), np.flatnonzero(b[:E.padded][pad] != 0.0)[:8]
        assert np.all(np.isfinite(b[E.map])) and np.isfinite(b[E.padded])
    finally:
        E.close()


# ---- the update in isolation --------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("regime", REGIMES)
@pytest.mark.parametrize("family", FAMILIES)
def test_injected_bucket_regimes(engines, family, regime):
    E = engines(family)
    E.restore(E.initial)
    g = make_gradient(E, regime, np.random.default_rng([FAMILIES.index(family), REGIMES.index(regime)]))
    out, _ = apply_and_check(E, E.place(g), tag=regime)
    if regime == "above_clip":
        assert out["grad_norm"] > 100 * (E.clip if E.clip > 0 else 40.0)   # R2D2 applies it unclipped


@pytest.mark.gpu
@pytest.mark.parametrize("family", FAMILIES)
def test_learning_rate_decays_then_clamps_at_end(engines, family):
    """learning_frame = 3, end 1e-5: five applies see lr(0) > lr(1) > lr(2) > lr(3) = lr(4) = end (R2D2: constant)."""
    E = engines(family, learning_frame=3, end_lr=1e-5)
    E.restore(E.initial)
    rng = np.random.default_rng(3)
    lrs = []
    for s in range(5):
        out, _ = apply_and_check(E, E.place(make_gradient(E, ("above_clip", "below_clip")[s % 2], rng)),
                                 tag="schedule@%d" % s)
        lrs.append(out.get("learning_rate", E.lr_at(s)))
    if family == "r2d2":
        assert len(set(lrs)) == 1
    else:
        assert lrs[0] > lrs[1] > lrs[2] > lrs[3] == lrs[4] == float(F32(1e-5)), lrs


@pytest.mark.gpu
@pytest.mark.parametrize("step", [7, 2 ** 32 + 5])
@pytest.mark.parametrize("family", FAMILIES)
def test_restored_optimizer_state(engines, family, step):
    """set_opt_state with random slots, a step with a nonzero high word and matching beta powers: the update takes lr
    from the restored step and alpha from the restored powers, and reports step + 1."""
    E = engines(family, learning_frame=2.0 ** 33, end_lr=1e-5)     # step 2^32 + 5 sits half-way down the decay
    rng = np.random.default_rng(step % 1000)
    n = E.packed
    st = dict(E.initial, step=step)
    if family == "impala":
        st["slots"] = (rng.uniform(0.5, 2.0, n).astype(np.float32),)
    else:
        st["slots"] = ((rng.standard_normal(n) * 1e-2).astype(np.float32), rng.uniform(1e-6, 1e-2, n).astype(np.float32))
        st["b1p"], st["b2p"] = float(F32(0.9 ** step)), float(F32(0.999 ** step))
    E.restore(st)
    assert E.state()["step"] == step
    out, st1 = apply_and_check(E, E.place(make_gradient(E, "below_clip", rng)), tag="restored@%d" % step)
    assert out["step"] == step + 1 and st1["step"] == step + 1
    if family in ("impala", "apex", "a3c") and step > 2 ** 32:
        assert E.end_lr < out["learning_rate"] < E.start_lr


@pytest.mark.gpu
@pytest.mark.parametrize("grad_scale", [1.0, 0.5, 1.0 / 3.0, 0.125])
@pytest.mark.parametrize("family", ADAM)
def test_grad_scale(engines, family, grad_scale):
    """The data-parallel scale: reported norm = ||bucket|| * gs, losses = bucket tail * gs, update on gs * g clipped
    by that norm -- with clipping engaged and not."""
    E = engines(family)
    rng = np.random.default_rng(int(grad_scale * 1000))
    for regime in ("below_clip", "above_clip"):
        E.restore(E.initial)
        apply_and_check(E, E.place(make_gradient(E, regime, rng)), grad_scale, tag="gs=%g,%s" % (grad_scale, regime))


@pytest.mark.gpu
@pytest.mark.parametrize("family", ADAM)
def test_invalid_grad_scale_is_refused_and_changes_nothing(engines, family):
    E = engines(family)
    E.restore(E.initial)
    E.write(E.place(make_gradient(E, "above_clip", np.random.default_rng(1))))
    before = E.state()
    for gs in (0.0, -1.0, float("nan")):
        with pytest.raises(E.N.DrlError):
            E.apply(gs)
        after = E.state()
        assert after["step"] == before["step"] and after["b1p"] == before["b1p"] and after["b2p"] == before["b2p"]
        assert np.array_equal(after["params"], before["params"])
        for a, b in zip(after["slots"], before["slots"]):
            assert np.array_equal(a, b)


# ---- determinism and graphs ---------------------------------------------------------------------------------------
def _same(s1, s2):
    return (s1["step"] == s2["step"] and np.array_equal(s1["params"], s2["params"]) and
            all(np.array_equal(a, b) for a, b in zip(s1["slots"], s2["slots"])) and
            s1.get("b1p") == s2.get("b1p") and s1.get("b2p") == s2.get("b2p"))


@pytest.mark.gpu
@pytest.mark.parametrize("family", FAMILIES)
def test_same_state_and_bucket_give_identical_bits(engines, family):
    """The norm reduction is in a fixed order: the same state and bucket applied twice give the same bits."""
    E = engines(family)
    bucket = E.place(make_gradient(E, "heavy_tailed", np.random.default_rng(9)))
    runs = []
    for _ in range(2):
        E.restore(E.initial)
        E.write(bucket)
        E.apply()
        runs.append((E.wait(), E.state()))
    assert runs[0][0] == runs[1][0]
    assert _same(runs[0][1], runs[1][1])


@pytest.mark.gpu
def test_impala_graphs_match_eager_bit_for_bit(engines):
    """use_cuda_graph=True captures forward_backward and apply; both graphs give the eager path's bits."""
    eager = engines("impala")
    graph = engines("impala", use_cuda_graph=True)
    rng = np.random.default_rng(21)
    for E in (eager, graph):
        E.restore(eager.initial)
    for rnd in range(2):
        bucket = eager.place(make_gradient(eager, ("above_clip", "heavy_tailed")[rnd], rng))
        res = []
        for E in (eager, graph):
            E.forward_backward()                  # first call on `graph` captures, later calls launch the graph
            grads = E.eng.get_grads()
            E.write(bucket)
            E.apply()
            res.append((grads, E.wait(), E.state()))
        assert np.array_equal(res[0][0], res[1][0]), "forward_backward gradients differ (round %d)" % rnd
        assert res[0][1] == res[1][1], (res[0][1], res[1][1])
        assert _same(res[0][2], res[1][2])


# ---- the data-parallel halves of the Adam learners on one GPU -----------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("family", ADAM)
def test_forward_backward_apply_equals_step(native, family):
    """forward_backward -> apply(1) -> wait is the step, bit for bit; apply(0.5) on the same bucket is the update of
    0.5 * g."""
    one, two = Engine(family), Engine(family)
    try:
        one.eng.stage(0, *one._args)
        two.eng.stage(0, *two._args)
        r1 = one.eng.step(0)
        two.forward_backward()
        two.apply(1.0)
        r2 = two.eng.wait()
        if isinstance(r1, tuple):
            assert np.array_equal(r1[1], r2[1])                             # td_error
            r1, r2 = r1[0], r2[0]
        assert r1 == r2
        assert np.array_equal(one.eng.get_grads(), two.eng.get_grads())
        assert _same(one.state(), two.state())
        bucket = two.read()
        assert np.array_equal(bucket[two.map], two.eng.get_grads())
        apply_and_check(two, bucket, 0.5, tag="dp-half")
    finally:
        one.close()
        two.close()


# ---- whole steps with clipping engaged and the learning rate decayed past its end ---------------------------------
# clip = 1/4 of the oracle's unclipped norm at the first step; learning_frame = 2, so the third step runs at end_lr
END_TO_END = dict(learning_frame=2, end_learning_rate=1e-5)


@functools.lru_cache(maxsize=None)
def _unclipped_norm(family):
    if family == "impala":
        batch, params, cfg = parity.make_case(4, 20)
        return it.Learner(params, torch.float64, "dedup", **cfg).train(
            *[batch[k] for k in synthetic.TRAIN_FIELDS], return_all=True)[3]
    b = ax.make_transitions(4, A=4, seed=4321)
    if family == "apex":
        L = ax.Learner(ax.init_params(0, torch.float32, num_action=4), ax.init_params(1, torch.float32, num_action=4),
                       torch.float64, num_action=4)
        return L.distributed_train(*[b[k] for k in ax.TRAIN_FIELDS], return_all=True)[3]
    L = at.Learner(at.init_params(0, torch.float32, num_action=4), torch.float64, num_action=4)
    return L.train(*[b[k] for k in at.TRAIN_FIELDS], return_all=True)[3]


def _no_failures(bad):
    assert not bad, sorted(bad.items(), key=lambda kv: -kv[1])[:10]


@pytest.mark.gpu
@pytest.mark.parametrize("graph", [False, True])
@pytest.mark.parametrize("mode", [1, 5])
def test_impala_steps_clipped_past_decay_end(native, mode, graph):
    clip = 0.25 * _unclipped_norm("impala")
    errs = parity.compare_step(4, T=20, steps=3, layers=False, gradient_clip_norm=clip, math_mode=mode,
                               use_cuda_graph=graph, **END_TO_END)
    assert all(errs["clip_engaged@%d" % s] == 0.0 for s in range(3))
    _no_failures(parity.failures(errs))


@pytest.mark.gpu
def test_apex_steps_clipped_past_decay_end_with_target_sync(native):
    clip = 0.25 * _unclipped_norm("apex")
    errs = ap.compare_step(4, A=4, steps=3, sync_target_at=1, gradient_clip_norm=clip, **END_TO_END)
    assert all(errs["clip_engaged@%d" % s] == 0.0 for s in range(3))
    _no_failures(ap.apex_failures(errs))


@pytest.mark.gpu
def test_a3c_steps_clipped_past_decay_end_cuda_graph(native):
    import test_gpu_a3c
    clip = 0.25 * _unclipped_norm("a3c")
    errs = test_gpu_a3c.compare_step(4, A=4, steps=3, use_cuda_graph=True, gradient_clip_norm=clip, **END_TO_END)
    assert all(errs["clip_engaged@%d" % s] == 0.0 for s in range(3))
    _no_failures(parity.failures(errs))
