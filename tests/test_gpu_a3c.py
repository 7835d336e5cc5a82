"""GPU parity tests of the A3C learner: every call goes through the C-ABI (``drl_a3c_*``) and is compared with the
float64 oracle to 1e-4 relative; same ReLU-kink handling and Adam check as tests/apex_parity.py."""
import numpy as np
import pytest
import torch

import apex_parity as ap
from oracle import a3c_torch as at
from oracle import impala_torch as it
from parity import TOL, failures, rel_err

pytestmark = pytest.mark.gpu


def _masks(eng, B, A):
    m = ap.gpu_masks(eng, B, A)
    return {k.replace("value", "actor").replace("mean", "critic"): v for k, v in m.items()}


def compare_step(B, A=4, seed=4321, steps=1, reward_clipping="abs_one", gradient_clip_norm=None, learning_frame=None,
                 end_learning_rate=None, **kw):
    """The schedule arguments are optional and reach both learners, as in apex_parity.compare_step."""
    from distributed_reinforcement_learning_b200.a3c_learner import NativeA3CLearner
    params = at.init_params(0, torch.float32, num_action=A)
    schedule = {k: v for k, v in (("gradient_clip_norm", gradient_clip_norm), ("learning_frame", learning_frame),
                                  ("end_learning_rate", end_learning_rate)) if v is not None}
    L = at.Learner(params, torch.float64, num_action=A, reward_clipping=reward_clipping, **schedule)
    eng = NativeA3CLearner(batch=B, num_action=A, reward_clipping=reward_clipping, **schedule, **kw)
    eng.set_params(at.flatten_params(params))
    errs = {}
    flips = elems = 0
    max_abs = 0.0
    try:
        for s in range(steps):
            tag = "" if steps == 1 else "@%d" % s
            b = at.make_transitions(B, A=A, seed=seed + s)
            args = [b[k] for k in at.TRAIN_FIELDS]
            st0, p0 = eng.get_opt_state(), eng.get_params()
            eng.stage(s % eng.num_slots, *args)
            out = eng.step(s % eng.num_slots)
            taps = eng.taps()
            with it.activation_pattern(_masks(eng, B, A)) as stt:
                res, o, grads, gn = L.train(*args, return_all=True)
            flips, elems, max_abs = flips + stt["flips"], elems + stt["elems"], max(max_abs, stt["max_abs_at_flip"])
            for i, k in enumerate(("pi_loss", "baseline_loss", "entropy")):
                errs["loss/" + k + tag] = rel_err(out[k], res[i])
            errs["lr" + tag] = abs(out["learning_rate"] - res[3])
            errs["grad_norm" + tag] = rel_err(out["grad_norm"], gn)
            if gradient_clip_norm is not None:
                errs["clip_engaged" + tag] = 0.0 if gn > gradient_clip_norm else float("inf")
            if out["step"] != s + 1:
                errs["step" + tag] = float("inf")
            for k in ("policy", "value", "next_value", "advantage"):
                errs["tap/" + k + tag] = rel_err(taps[k], o[k].detach().numpy())
            g_gpu = eng.get_grads()
            gd = at.unflatten_params(g_gpu, torch.float64, num_action=A)
            for n in grads:
                errs["grad/" + n + tag] = rel_err(gd[n].numpy(), grads[n].detach().numpy())
            st1, p1 = eng.get_opt_state(), eng.get_params()
            g64 = g_gpu.astype(np.float64)
            exp_p, exp_m, exp_v = ap.adam_expected(p0.astype(np.float64), g64, st0["m"].astype(np.float64),
                                                   st0["v"].astype(np.float64), float(np.sqrt(np.sum(g64 ** 2))),
                                                   L.cfg["gradient_clip_norm"],
                                                   float(out["learning_rate"]), st0["beta1_power"], st0["beta2_power"])
            floor = 4.0 * np.finfo(np.float32).eps * np.max(np.abs(p0)) / TOL
            errs["update/adam" + tag] = float(np.max(np.abs(p1 - exp_p)) / (np.max(np.abs(exp_p - p0)) + floor))
            errs["adam/m" + tag] = rel_err(st1["m"], exp_m)
            errs["adam/v" + tag] = rel_err(st1["v"], exp_v)
            pd = at.unflatten_params(p1, torch.float64, num_action=A)
            md = at.unflatten_params(st1["m"], torch.float64, num_action=A)
            vd = at.unflatten_params(st1["v"], torch.float64, num_action=A)
            with torch.no_grad():
                for n in L.params:
                    L.params[n].copy_(pd[n])
                    L.m[n].copy_(md[n])
                    L.v[n].copy_(vd[n])
            L.beta1_power, L.beta2_power = np.float32(st1["beta1_power"]), np.float32(st1["beta2_power"])
        errs["kink/flip_fraction"] = flips / max(elems, 1)
        errs["kink/max_abs_at_flip"] = max_abs
    finally:
        eng.close()
    return errs


def _check(errs):
    bad = failures(errs)
    assert not bad, sorted(bad.items(), key=lambda kv: -kv[1])[:10]


@pytest.mark.parametrize("mode", [1, 2])
def test_step_small(native, mode):
    _check(compare_step(3, A=4, math_mode=mode))


def test_step_reference_config(native):
    """config.json:2-41: one unroll of trajectory = 32 transitions, 4 actions."""
    _check(compare_step(32, A=4))


@pytest.mark.parametrize("B,A", [(1, 2), (7, 18)])
def test_step_ragged(native, B, A):
    _check(compare_step(B, A=A))


def test_three_steps_soft_asymmetric_cuda_graph(native):
    _check(compare_step(4, A=4, steps=3, reward_clipping="soft_asymmetric", use_cuda_graph=True))


def test_agent_train_and_act(native):
    from distributed_reinforcement_learning_b200.agent import a3c
    kw = dict(input_shape=[84, 84, 4], num_action=4, discount_factor=0.997, start_learning_rate=1e-4,
              end_learning_rate=0.0, learning_frame=1000000000, baseline_loss_coef=1.0, entropy_coef=0.05,
              gradient_clip_norm=40.0, reward_clipping="abs_one", model_name="learner", learner_name="learner")
    ag = a3c.Agent(**kw)
    ag.set_session(None)
    b = at.make_transitions(8, seed=3)
    L = at.Learner(at.unflatten_params(ag._params, torch.float32, num_action=4), torch.float64, num_action=4)
    for _ in range(2):
        got = ag.train(*[b[k] for k in at.TRAIN_FIELDS])
    ref = None
    res = L.train(*[b[k] for k in at.TRAIN_FIELDS])
    assert len(got) == 4 and all(np.isfinite(got))
    assert ag.num_env_frames == 2
    action, policy, max_prob = ag.get_policy_and_action(b["state"][0], 1)
    assert policy.shape == (4,) and abs(policy.sum() - 1) < 1e-5 and max_prob == policy[action]
    pol, val = ag._engine.act(b["state"][:3], b["previous_action"][:3])
    assert pol.shape == (3, 4) and val.shape == (3,)
