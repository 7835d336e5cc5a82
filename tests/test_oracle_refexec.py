"""PIN of the oracle to the reference itself.  ``tests/golden/refexec.npz`` holds what the UNMODIFIED reference files
(``agent/impala.py``, ``optimizer/vtrace.py``, ``model/impala_actor_critic.py``, ``distributed_queue/buffer_queue.py``,
``utils.py``; and the Ape-X / R2D2 / A3C files) computed when executed over ``oracle/tf1_shim`` (a TF 1.14 API stand-in
on torch-CPU that restates only TF's op semantics -- see its docstring); ``tests/golden/make_golden.py refexec``
writes it from a reference checkout.  The restatements under ``oracle/`` (and, where the reference has a host-side
counterpart, the native FIFO ring and prioritized replay memory) must agree with it on every slice, window, loss,
stop_gradient and optimizer decision: V-trace taps, the three losses, all 24 gradients, three RMSProp steps with slots
and global_step, both reward-clipping modes, the reference-shaped 54-copy graph against the deduplicated forward,
variable names/order/sharing, parameter_sync, single-step inference and the FIFO queue's order.

Tensors are stored as a strided sample plus the l2 norm of the whole tensor (``_check_tensors``); everything else whole.
CPU-only."""
import os
import random

import numpy as np
import pytest
import torch

from oracle import impala_torch as it
from oracle import ref_exec, synthetic, vtrace_np

Z = np.load(os.path.join(os.path.dirname(__file__), "golden", "refexec.npz"))


def _rel(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return float(np.max(np.abs(a - b)) / max(np.max(np.abs(b)), 1e-300)) if b.size else 0.0


def _np(v):
    return v.detach().numpy() if hasattr(v, "detach") else np.asarray(v)


def _check_tensors(key, got, tol):
    """``got`` (name -> tensor) against the reference's tensors stored under ``key`` by make_golden.py: the same names,
    the strided sample within ``tol`` relative (``_rel``), the l2 norm of the whole tensor within ``tol`` relative."""
    names, strides, l2, sample = list(Z[key + ":names"]), Z[key + ":stride"], Z[key + ":l2"], Z[key + ":sample"]
    assert sorted(names) == sorted(got), key
    off = 0
    for n, s, norm in zip(names, strides, l2):
        v = np.asarray(_np(got[n]), np.float64).ravel()
        m = -(-v.size // int(s))
        assert _rel(v[::s], sample[off:off + m]) <= tol, (key, n)
        assert abs(np.sqrt(np.sum(v ** 2)) - norm) <= tol * max(norm, 1e-300), (key, n)
        off += m
    assert off == sample.size, key


def _case(B, T, A, seed=4321, **cfg):
    batch = synthetic.make_batch(B, T=T, A=A, seed=seed)
    params = it.init_params(0, torch.float32, num_action=A)
    return batch, params, [batch[k] for k in synthetic.TRAIN_FIELDS], dict(trajectory=T, num_action=A, **cfg)


TAPS = ("vs", "clipped_rho", "vs_plus_1", "pg_advantage", "pi_loss", "baseline_loss", "entropy", "total_loss")


@pytest.mark.parametrize("clipping", ["abs_one", "soft_asymmetric"])
def test_impala_executed_reference_equals_restatement(clipping):
    """agent/impala.py:31-100,132-148 executed == oracle/impala_torch.py (reference-shaped AND deduplicated)."""
    key = "impala_" + clipping
    batch, params, args, cfg = _case(2, 6, 18, reward_clipping=clipping)
    for shaped, tol in (("reference", 1e-13), ("dedup", 1e-11)):
        L = it.Learner(params, torch.float64, shaped, **cfg)
        out, g = L.gradients(*args)
        for k in TAPS:
            assert _rel(out[k].detach().numpy(), Z[key + ":" + k]) <= tol, (shaped, k)
        assert _rel(out["first_policy"].detach().numpy(), Z[key + ":unrolled_first_policy"]) <= tol
        assert _rel(out["middle_value"].detach().numpy(), Z[key + ":unrolled_middle_value"]) <= tol
        assert _rel(out["last_value"].detach().numpy(), Z[key + ":unrolled_last_value"]) <= tol
        assert len(g) == 24
        _check_tensors(key + ":grad", g, tol * 10)
    assert Z[key + ":clipped_r_ph"].min() >= (-1.0 if clipping == "abs_one" else -1.5)


def test_impala_three_train_steps_track_the_executed_reference():
    """Agent.train x3: returned scalars, every parameter, the RMSProp ``rms`` slots (ms0 = 1, eps inside the sqrt),
    global_step and the learning rate -- TF1 optimizer semantics as restated in the shim's docstring."""
    batch, params, args, cfg = _case(2, 6, 18)
    L = it.Learner(params, torch.float64, "dedup", **cfg)
    for step in range(3):
        r, o = Z["train3:%d:result" % step], L.train(*args)
        for a, b in zip(r[:3], o[:3]):
            assert abs(a - b) <= 1e-9 * max(abs(b), 1.0)
        assert abs(r[3] - o[3]) < 1e-10                  # lr: float32 polynomial_decay in the oracle, exact here
        assert int(Z["train3:%d:global_step" % step]) == step + 1 == L.step
        _check_tensors("train3:%d:param" % step, L.params, 1e-9)
        _check_tensors("train3:%d:rms" % step, L.ms, 1e-9)
    # slots started at ones (TF1), not zeros
    assert bool(Z["train3:rms_all_moved"]) and float(Z["train3:rms_min"]) > 0.9
    assert all(np.any(v.numpy() != 1.0) and np.all(v.numpy() > 0.9) for v in L.ms.values())


def test_baseline_config0_b4_t20_54_graph_copies_equal_one_forward():
    """BASELINE configs[0] (T=20, B=4): the reference's 3 x 18 per-timestep network copies (executed) against the
    ONE forward over the 20 distinct rows that the CUDA path runs (shift identity, SURVEY App. C.4)."""
    batch, params, args, cfg = _case(4, 20, 18, seed=1234)
    L = it.Learner(params, torch.float64, "dedup", **cfg)
    out, g = L.gradients(*args)
    for k in TAPS:
        assert _rel(out[k].detach().numpy(), Z["b4t20:" + k]) <= 1e-11, k
    _check_tensors("b4t20:grad", g, 1e-10)


def test_float32_execution_is_within_the_parity_bar_of_float64():
    """The same reference graph evaluated in float32 (TF's arithmetic type) sits inside the 1e-4 bar that the CUDA path
    is held to: the bar is meaningful for a float32 implementation of this graph.  The float64 side is the
    reference-shaped restatement, which equals the executed float64 reference to 1e-13 (first test above)."""
    batch, params, args, cfg = _case(2, 6, 18)
    out, _ = it.Learner(params, torch.float64, "reference", **cfg).gradients(*args)
    assert Z["f32:vs"].dtype == np.float32
    for k in TAPS:
        assert _rel(Z["f32:" + k], out[k].detach().numpy()) < 1e-4, k


def test_variable_names_sharing_and_parameter_sync():
    """model/impala_actor_critic.py:47-109 re-enters variable_scope('impala', reuse=AUTO_REUSE) 55 times: exactly 24
    trainable variables result, named as TF1 names them, in the oracle's parameter order and shapes; a second agent
    (train_impala.py:64-80, 'actor_0') adds its own 24 and utils.copy_src_to_dst (parameter_sync) copies learner ->
    actor in creation order.  The learner held init_params(0) when the actor was synced."""
    names = list(Z["sync:names"])
    assert len(names) == 24
    assert names[:2] == ["learner/impala/conv2d/kernel", "learner/impala/conv2d/bias"]
    assert names[10:12] == ["learner/impala/rnn/lstm_cell/kernel", "learner/impala/rnn/lstm_cell/bias"]
    assert names[-2:] == ["learner/impala/dense_7/kernel", "learner/impala/dense_7/bias"]
    specs = it.param_specs(num_action=6)
    assert names == ["learner/impala/%s/%s" % (tf_name, kind) for tf_name, _ in ref_exec.IMPALA_VAR_ORDER
                     for kind in ("kernel", "bias")]
    assert [n for n, _ in specs] == [our + sfx for _, our in ref_exec.IMPALA_VAR_ORDER for sfx in (".w", ".b")]
    assert list(Z["sync:shapes"]) == [str(tuple(s)) for _, s in specs]
    assert Z["sync:shapes"][10] == "(3648, 1024)"
    assert int(Z["sync:n_vars_two_agents"]) == 48 and int(Z["sync:n_global_to_session"]) == 24
    assert bool(Z["sync:differ_before"]) and bool(Z["sync:equal_after"])
    # single-step inference (agent/impala.py:118-130) on the synced actor == the oracle's ``network``
    rng = np.random.default_rng(3)
    state = rng.integers(0, 256, (84, 84, 4), dtype=np.uint8)
    h, c = rng.standard_normal(256).astype(np.float32) * 0.3, rng.standard_normal(256).astype(np.float32)
    p = {n: v.double() for n, v in it.init_params(0, torch.float32, num_action=6).items()}
    x = torch.from_numpy((state[None].astype(np.float64) / 255).astype(np.float32)).double()
    pol, val, oc, oh = it.network(p, x, torch.tensor([2]), torch.from_numpy(h[None]).double(),
                                  torch.from_numpy(c[None]).double(), 6, 256)
    policy, action = Z["sync:policy"], int(Z["sync:action"])
    assert _rel(policy, pol[0].numpy()) < 1e-12 and float(Z["sync:max"]) == max(policy) and 0 <= action < 6
    # returns (.., h, c) in that order
    assert _rel(Z["sync:h"], oh[0].numpy()) < 1e-12 and _rel(Z["sync:c"], oc[0].numpy()) < 1e-12


def test_static_placeholder_shapes_reject_a_wrong_trajectory_length():
    """Error behaviour at the boundary (SURVEY 8b): feeding T+1 steps to the [None, T, ...] placeholders raises in the
    reference, and the restatement rejects the same batch."""
    assert str(Z["wrong_t:error"]) == "ValueError"
    batch, params, args, cfg = _case(2, 6, 18)
    L = it.Learner(params, torch.float64, "dedup", **cfg)
    bad = synthetic.make_batch(2, T=7, A=18, seed=1)
    with pytest.raises((ValueError, RuntimeError)):
        L.train(*[bad[k] for k in synthetic.TRAIN_FIELDS])


# ---- optimizer/vtrace.py, function by function -------------------------------------------------------------------
def test_vtrace_functions_executed_equal_numpy_and_c_restatements():
    z = np.load(os.path.join(os.path.dirname(__file__), "golden", "vtrace_T18_B8.npz"))
    kw = {k: z[k] for k in ("log_rhos", "discounts", "rewards", "values", "bootstrap_value")}
    ovs, orho = vtrace_np.from_importance_weights(**kw)
    np.testing.assert_allclose(ovs, z["vs"], rtol=1e-13, atol=1e-13)
    np.testing.assert_allclose(orho, z["clipped_rhos"], rtol=1e-13, atol=1e-13)
    from oracle import vtrace_c
    cvs, crho = vtrace_c.from_importance_weights(**kw)               # plain-C restatement (gcc, built on demand)
    np.testing.assert_allclose(cvs, z["vs"], rtol=1e-12, atol=1e-12)
    # clip_rho_threshold honoured, clip_pg_rho_threshold dead, cs hard-coded at 1 (optimizer/vtrace.py:72-80)
    b = vtrace_np.from_importance_weights(clip_rho_threshold=0.5, **kw)
    np.testing.assert_allclose(Z["vtrace:clip05_vs"], b[0], rtol=1e-13, atol=1e-13)
    np.testing.assert_allclose(Z["vtrace:clip05_rho"], b[1], rtol=1e-13, atol=1e-13)
    assert Z["vtrace:clip05_rho"].max() <= 0.5

    rng = np.random.default_rng(11)
    B, T, A = 5, 9, 7
    sm = lambda x: np.exp(x) / np.exp(x).sum(-1, keepdims=True)
    mu, pi = sm(rng.standard_normal((B, T, A))), sm(rng.standard_normal((B, T, A)))
    act = rng.integers(0, A, (B, T)).astype(np.int32)
    disc = (rng.random((B, T)) > 0.1) * 0.99
    rew, val, nval = rng.standard_normal((B, T)), rng.standard_normal((B, T)), rng.standard_normal((B, T))
    exp = vtrace_np.from_softmax(mu, pi, act, disc, rew, val, nval, A)
    np.testing.assert_allclose(Z["vtrace:softmax_vs"], exp[0], rtol=1e-12, atol=1e-12)
    np.testing.assert_allclose(Z["vtrace:softmax_rho"], exp[1], rtol=1e-12, atol=1e-12)
    adv = rng.standard_normal((B, T))
    assert float(Z["vtrace:pg_loss"]) == pytest.approx(vtrace_np.compute_policy_gradient_loss(pi, act, adv, A), rel=1e-12)
    assert float(Z["vtrace:baseline_loss"]) == pytest.approx(vtrace_np.compute_baseline_loss(val, nval), rel=1e-12)
    assert float(Z["vtrace:entropy_loss"]) == pytest.approx(vtrace_np.compute_entropy_loss(pi), rel=1e-12)
    np.testing.assert_allclose(Z["vtrace:log_probs"], vtrace_np.log_probs_from_softmax_and_actions(pi, act, A),
                               rtol=1e-12)
    for k, e in zip(("split_first", "split_middle", "split_last"), vtrace_np.split_data(val)):
        np.testing.assert_array_equal(Z["vtrace:" + k], e)


# ---- distributed_queue/buffer_queue.py:418-512 against the pinned-ring replacement ---------------------------------
def test_reference_fifo_queue_order_equals_the_ring(native):
    from distributed_reinforcement_learning_b200.distributed_queue import buffer_queue
    T, shape, A, L, cap, batch = 5, [6, 6, 2], 4, 8, 8, 3
    ours = buffer_queue.FIFOQueue(T, shape, A, cap, batch, 2, L, pinned=False)
    rng = np.random.default_rng(5)

    def rec():
        return dict(unrolled_state=rng.integers(0, 256, (T, *shape), dtype=np.uint8),
                    unrolled_next_state=rng.integers(0, 256, (T, *shape), dtype=np.uint8),
                    unrolled_reward=rng.standard_normal(T).astype(np.float32), unrolled_done=rng.random(T) < 0.3,
                    unrolled_behavior_policy=rng.random((T, A)).astype(np.float32),
                    unrolled_action=rng.integers(0, A, T).astype(np.int32),
                    unrolled_previous_action=rng.integers(0, A, T).astype(np.int32),
                    unrolled_previous_h=rng.standard_normal((T, L)).astype(np.float32),
                    unrolled_previous_c=rng.standard_normal((T, L)).astype(np.float32))

    recs = [rec() for _ in range(7)]
    for i, r in enumerate(recs):
        ours.append_to_queue(task=i % 2, **r)
    assert ours.get_size() == int(Z["fifo:size_full"]) == 7
    assert tuple(Z["fifo:fields"]) == ("state", "next_state", "reward", "done", "behavior_policy", "action",
                                       "previous_action", "previous_h", "previous_c")
    for j, lo in enumerate((0, 3)):
        idx = [int(i) for i in Z["fifo:sample%d" % j]]
        assert idx == list(range(lo, lo + batch))          # the reference's queue is first in, first out
        ob = ours.sample_batch()
        for name in ("state", "reward", "done", "behavior_policy", "action", "previous_action", "previous_h",
                     "previous_c"):
            np.testing.assert_array_equal(np.stack(getattr(ob, name)),
                                          np.stack([recs[i]["unrolled_" + name] for i in idx]), err_msg=name)
    assert ours.get_size() == int(Z["fifo:size_left"]) == 1


def test_learner_loop_call_pattern_on_the_executed_reference(native):
    """train_impala.py:93-113 with the reference's own FIFOQueue and Agent (over the shim): gate on size > 3*batch,
    sample_batch, np.stack of every field, Agent.train.  Replayed here on the native ring and the oracle: the same
    records in each batch, the same number of steps, scalars equal to the reference's."""
    from distributed_reinforcement_learning_b200.distributed_queue import buffer_queue
    B, T, A, L = 2, 5, 6, 256
    params = it.init_params(0, torch.float32, num_action=A)
    queue = buffer_queue.FIFOQueue(T, [84, 84, 4], A, 128, B, 1, L, pinned=False)
    O = it.Learner(params, torch.float64, "dedup", trajectory=T, num_action=A)
    big = synthetic.make_batch(3 * B + 1 + B, T=T, A=A, seed=77)
    for i in range(big["state"].shape[0]):
        queue.append_to_queue(task=0, unrolled_state=big["state"][i], unrolled_next_state=big["state"][i],
                              unrolled_reward=big["reward"][i], unrolled_done=big["done"][i],
                              unrolled_behavior_policy=big["behavior_policy"][i], unrolled_action=big["action"][i],
                              unrolled_previous_action=big["previous_action"][i],
                              unrolled_previous_h=big["initial_h"][i], unrolled_previous_c=big["initial_c"][i])
    steps = 0
    while queue.get_size() > 3 * B:
        batch = queue.sample_batch()
        kw = dict(state=np.stack(batch.state), reward=np.stack(batch.reward), action=np.stack(batch.action),
                  done=np.stack(batch.done), behavior_policy=np.stack(batch.behavior_policy),
                  previous_action=np.stack(batch.previous_action), initial_h=np.stack(batch.previous_h),
                  initial_c=np.stack(batch.previous_c))
        np.testing.assert_array_equal(kw["state"], big["state"][Z["loop:%d:records" % steps]])
        got = Z["loop:%d:result" % steps]
        exp = O.train(**kw)
        for a, b in zip(got[:3], exp[:3]):
            assert abs(a - b) <= 1e-9 * max(abs(b), 1.0)
        steps += 1
    assert steps == int(Z["loop:steps"]) == 2 and queue.get_size() == int(Z["loop:size_left"]) == 3 * B - 1


# ---- next rows: Ape-X and R2D2 agents executed -------------------------------------------------------------------
def test_apex_executed_reference_equals_restatement():
    from oracle import apex_torch as ax
    A = 4
    b = ax.make_transitions(3, A=A, seed=1357)
    p, tp = ax.init_params(0, torch.float32, num_action=A), ax.init_params(1, torch.float32, num_action=A)
    L = ax.Learner(p, tp, torch.float64, num_action=A)
    args = [b[k] for k in ax.TRAIN_FIELDS]
    out, g = L.gradients(*args[:6], is_weight=args[6])
    for k, ok in (("main_q_value", "main_q"), ("next_main_q_value", "next_main_q"), ("target_q_value", "target_q"),
                  ("target_value", "target_value"), ("state_action_value", "state_action_value"),
                  ("value_loss", "value_loss")):
        assert _rel(out[ok].detach().numpy(), Z["apex:" + k]) < 1e-12, k
    assert np.array_equal(Z["apex:next_action"], out["next_action"].numpy())
    assert len(Z["apex:grad:names"]) == 22                # target variables receive no gradient (None in TF)
    _check_tensors("apex:grad", g, 1e-11)
    assert _rel(Z["apex:td_single"], L.get_td_error(*args[:6])) < 1e-12
    for i in range(3):
        r2 = L.distributed_train(*args)
        assert float(Z["apex:%d:loss" % i]) == pytest.approx(r2[0], rel=1e-6) and _rel(Z["apex:%d:td" % i], r2[1]) < 1e-6
    _check_tensors("apex:param", L.params, 1e-6)
    _check_tensors("apex:adam_m", L.m, 1e-5)
    _check_tensors("apex:adam_v", L.v, 1e-5)
    assert bool(Z["apex:target_differs"]) and any(np.any(L.target[n].numpy() != L.params[n].detach().numpy())
                                                  for n in L.params)
    L.target_to_main()                                    # despite the name: target <- main (utils.py:27-32)
    for n in L.params:
        assert np.array_equal(L.target[n].numpy(), L.params[n].detach().numpy())
    _check_tensors("apex:param", L.target, 1e-6)


def test_r2d2_executed_reference_equals_restatement():
    from oracle import r2d2_torch as rt
    S, bi = 6, 2
    b = rt.make_sequences(2, S=S, seed=2468)
    p, tp = rt.init_params(0, torch.float32), rt.init_params(1, torch.float32)
    L = rt.Learner(p, tp, torch.float64, seq_len=S, burn_in=bi)
    args = [b[k] for k in rt.TRAIN_FIELDS]
    out, g = L.gradients(*args[:7], weight=args[7])
    for k in ("main_q", "target_q", "target_value", "state_action_value", "value_loss"):
        assert _rel(out[k].detach().numpy(), Z["r2d2:" + k]) < 1e-12, k
    assert len(Z["r2d2:grad:names"]) == 18
    _check_tensors("r2d2:grad", g, 1e-11)
    for i in range(3):
        r2 = L.train(*args)
        assert float(Z["r2d2:%d:loss" % i]) == pytest.approx(r2[0], rel=1e-6) and _rel(Z["r2d2:%d:td" % i], r2[1]) < 1e-5
    _check_tensors("r2d2:param", L.params, 1e-6)
    L.main_to_target()
    for n in L.params:
        assert np.array_equal(L.target[n].numpy(), L.params[n].detach().numpy())


# ---- distributed_queue/buffer_queue.py:326-415 SumTree / Memory: plain NumPy in the reference -----------------------
def test_reference_sumtree_and_memory_executed_equal_restatement_and_native(native):
    """The reference's prioritized replay memory has no TF in it: its own ``SumTree`` / ``Memory`` classes were executed
    (CPython ``random`` seeded) and ``oracle.per_np`` and the ``drl_per_*`` mirror must reproduce them over a
    wrap-around fill, interleaved priority updates and 40 ``sample`` calls: tree nodes, sampled tree indices, data and
    the beta schedule bit for bit, importance weights bit for bit (NumPy) / to 1 ulp (libm ``pow`` in csrc/per.cu)."""
    from distributed_reinforcement_learning_b200.distributed_queue import buffer_queue
    from oracle import per_np
    cap, n = 37, 8
    omem, nmem = per_np.MemoryNP(cap), buffer_queue.Memory(cap)
    rng = np.random.default_rng(11)
    for i in range(cap + 9):                            # wraps: the 9 oldest records are overwritten
        e = float(abs(rng.standard_normal()) * 3)
        omem.add(e)
        nmem.add(e, ("rec", i))
    latest = {i % cap: i for i in range(cap + 9)}       # record held by each data slot after the wrap
    np.testing.assert_array_equal(Z["per:tree_filled"], omem.tree.nodes)
    assert int(Z["per:n_entries"]) == omem.tree.n_entries == cap and int(Z["per:write"]) == 9
    for k in range(40):
        ridx, rw, beta = [int(j) for j in Z["per:idx"][k]], Z["per:weight"][k], float(Z["per:beta"][k])
        rrec = [int(r) for r in Z["per:record"][k]]
        random.seed(1000 + k)
        u = [random.random() for _ in range(n)]
        oidx, odata, oprio, ow = omem.sample(n, u)
        assert list(oidx) == ridx and beta == omem.beta == pytest.approx(min(1.0, 0.4 + 0.001 * (k + 1)), abs=1e-15)
        np.testing.assert_array_equal(ow, rw)
        assert [latest[int(j)] for j in odata] == rrec
        nbatch, nidx, nw = nmem.sample(n, u)
        assert list(nidx) == ridx and nbatch == [("rec", r) for r in rrec] and nmem.beta == beta
        np.testing.assert_allclose(nw, rw, rtol=4e-16, atol=0)   # libm pow vs NumPy's SIMD pow: <= 1 ulp
        for j in ridx[::2]:                             # the learner writes new |td| back (train_apex.py:121-124)
            e = float(abs(rng.standard_normal()))
            omem.update(j, e)
            nmem.update(j, e)
        np.testing.assert_allclose(omem.tree.nodes, Z["per:tree"][k], rtol=0, atol=0)
        assert omem.tree.total() == float(Z["per:total"][k]) == nmem.tree.total()


# ---- agent/a3c.py + model/actor_critic.py + optimizer/a2c.py (the fourth learner family) ---------------------------
@pytest.mark.parametrize("clipping", ["abs_one", "soft_asymmetric"])
def test_a3c_executed_reference_equals_restatement(clipping):
    from oracle import a3c_torch as a3
    key = "a3c_" + clipping
    A = 5
    b = a3.make_transitions(4, A=A, seed=97)
    b["reward"] = (b["reward"] * 3).astype(np.float32)            # both branches of either clipping
    p = a3.init_params(0, torch.float32, num_action=A)
    L = a3.Learner(p, torch.float64, num_action=A, reward_clipping=clipping)
    args = [b[k] for k in a3.TRAIN_FIELDS]
    out = L.losses(*args)
    for k in ("policy", "value", "next_value"):
        assert _rel(out[k].detach().numpy(), Z["%s:%s" % (key, k)]) < 1e-12, k
    for k in ("pi_loss", "baseline_loss", "entropy", "total_loss"):
        assert float(out[k].detach()) == pytest.approx(float(Z["%s:%s" % (key, k)]), rel=1e-12), k
    names = list(L.params)
    g = torch.autograd.grad(out["total_loss"], [L.params[n] for n in names], allow_unused=True)
    assert len(Z[key + ":grad:names"]) == 22
    _check_tensors(key + ":grad", dict(zip(names, g)), 1e-11)
    # three Agent.train calls: poly-decay lr, clip_by_global_norm 40, Adam with float32 beta powers
    for i in range(3):
        r2 = L.train(*args)
        for x, y in zip(Z["%s:%d:result" % (key, i)], r2):
            assert float(x) == pytest.approx(float(y), rel=1e-6, abs=1e-12)
    _check_tensors(key + ":param", L.params, 1e-6)
    _check_tensors(key + ":adam_m", L.m, 1e-5)
    _check_tensors(key + ":adam_v", L.v, 1e-5)
