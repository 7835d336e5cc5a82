"""Generates the committed golden vectors of the IMPALA learner step, of optimizer/vtrace.py and of the Ape-X / R2D2
steps by EXECUTING THE UNMODIFIED REFERENCE FILES (``agent/impala.py`` etc. of a reference checkout) over the TF 1.14
API stand-in ``oracle/tf1_shim`` in float64 (``oracle/ref_exec.py``), the A3C family included; ``refexec`` writes what
tests/test_oracle_refexec.py compares the restatements with.

    DRL_REFERENCE_DIR=/path/to/distributed_reinforcement_learning \
        python tests/golden/make_golden.py [impala] [vtrace] [apex] [r2d2] [a3c] [refexec]   # default: all

Needs the reference checkout; the tests do not.  Every file records ``source``.  What these vectors pin: the
restatements under ``oracle/`` (CPU suite, float64, ~1e-12) and the CUDA path (``-m gpu`` suite, 1e-4) against the
reference's own graph-construction code; TensorFlow's op kernels themselves are restated by the shim (see its
docstring) -- ``tests/golden/make_golden_tf1.py`` regenerates the same files under a real tensorflow==1.14.0 where
one exists.  Inputs are regenerated from the stored seed by oracle/synthetic.py::make_batch and
oracle/impala_torch.py::init_params(0).
"""
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))

from oracle import impala_torch as it  # noqa: E402
from oracle import synthetic, vtrace_np  # noqa: E402


STRIDE = 61


SOURCE = "reference files executed over oracle/tf1_shim (float64)"


def learner_case(B, T, A, seed, path):
    """agent/impala.py:132-148 ``Agent.train`` executed once; taps/gradients fetched from the agent's own graph."""
    from oracle import ref_exec
    batch = synthetic.make_batch(B, T=T, A=A, seed=seed)
    params = it.init_params(0, torch.float32, num_action=A)
    args = [batch[k] for k in synthetic.TRAIN_FIELDS]
    R = ref_exec.ReferenceImpala(params, trajectory=T, num_action=A)
    f = R.fetch(args, ["vs", "clipped_rho", "vs_plus_1", "pg_advantage", "unrolled_first_policy",
                       "unrolled_first_value", "total_loss"])
    g = {n: torch.from_numpy(np.asarray(v)) for n, v in R.gradients(args).items()}
    gn = float(np.sqrt(sum(float(torch.sum(v.double() ** 2)) for v in g.values())))
    pi, bl, en, lr = R.train(*args)
    rec = dict(B=B, T=T, A=A, seed=seed, pi_loss=pi, baseline_loss=bl, entropy=en, learning_rate=lr, grad_norm=gn,
               total_loss=float(f["total_loss"]), source=SOURCE)
    for k, src in (("vs", "vs"), ("clipped_rho", "clipped_rho"), ("vs_plus_1", "vs_plus_1"),
                   ("pg_advantage", "pg_advantage"), ("first_policy", "unrolled_first_policy"),
                   ("first_value", "unrolled_first_value")):
        rec[k] = f[src]
    # gradients and the applied update (clip_by_global_norm 40 + TF1 RMSProp, one step): every tensor as a strided
    # sample (stride_<name>) of the gradient, the new parameters and the new slots, plus the gradient's l2 norm
    params, rms = R.params(), R.rms()
    for n, v in g.items():
        v = v.numpy()
        s = rec["stride_" + n] = sample_stride(v.size)
        rec["gradsample_" + n] = v.ravel()[::s].astype(np.float32)
        rec["gradl2_" + n] = np.float64(np.sqrt(np.sum(v.astype(np.float64) ** 2)))
        rec["paramsample_" + n] = params[n].ravel()[::s]
        rec["rmssample_" + n] = rms[n].ravel()[::s]
    np.savez_compressed(path, **rec)
    return rec


def sample_stride(n, most=512):
    """Stride of a sample of at most ``most`` elements; odd, so that it visits every column of a power-of-two row."""
    return -(-n // most) | 1


def vtrace_case(path):
    rng = np.random.default_rng(2024)
    T, B = 18, 8
    kw = dict(log_rhos=rng.standard_normal((T, B)) * 0.7, discounts=(rng.random((T, B)) > 0.1) * 0.99,
              rewards=rng.standard_normal((T, B)), values=rng.standard_normal((T, B)),
              bootstrap_value=rng.standard_normal(B))
    from oracle import ref_exec
    ref = ref_exec.load(("optimizer.vtrace",), float_dtype=torch.float64)
    tf, vt = ref.tf, ref["optimizer.vtrace"]
    vs, rho = tf.Session().run(list(vt.from_importance_weights(**{k: tf.constant(np.asarray(v, np.float64))
                                                                   for k, v in kw.items()})))
    np.savez_compressed(path, vs=vs, clipped_rhos=rho, source=SOURCE, **kw)


def _pack_grads(rec, g):
    for n, v in g.items():
        v = v.detach().numpy() if hasattr(v, "detach") else np.asarray(v)
        if v.size > 70000:
            rec["gradsample_" + n] = v.ravel()[::STRIDE].astype(np.float32)
            rec["gradl2_" + n] = np.float64(np.sqrt(np.sum(v.astype(np.float64) ** 2)))
        else:
            rec["grad_" + n] = v.astype(np.float32)


def apex_case(path, B=3, A=4, seed=1357):
    """agent/apex.py:135-154 ``distributed_train`` executed once (inputs regenerated from make_transitions(B, A, seed),
    parameters from init_params(0) / init_params(1))."""
    from oracle import apex_torch as ax
    from oracle import ref_exec
    b = ax.make_transitions(B, A=A, seed=seed)
    p, tp = ax.init_params(0, torch.float32, num_action=A), ax.init_params(1, torch.float32, num_action=A)
    R = ref_exec.ReferenceApex(p, tp, num_action=A)
    args = [b[k] for k in ax.TRAIN_FIELDS]
    f = R.fetch(args, ["main_q_value", "next_main_q_value", "target_q_value", "target_value", "state_action_value",
                       "learning_rate"])
    g = {n: torch.from_numpy(np.asarray(v)) for n, v in R.gradients(R.feed(*args)).items()}
    gn = float(np.sqrt(sum(float(torch.sum(v.double() ** 2)) for v in g.values())))
    loss, td = R.agent.distributed_train(*args)
    rec = dict(B=B, A=A, seed=seed, loss=loss, td_error=td, grad_norm=gn, learning_rate=float(f["learning_rate"]),
               source=SOURCE)
    for k, src in (("main_q", "main_q_value"), ("next_main_q", "next_main_q_value"), ("target_q", "target_q_value"),
                   ("target_value", "target_value"), ("state_action_value", "state_action_value")):
        rec[k] = f[src]
    _pack_grads(rec, g)
    np.savez_compressed(path, **rec)
    return rec


def r2d2_case(path, B=2, S=6, bi=2, seed=2468):
    """agent/r2d2.py:132-159 ``Agent.train`` executed once."""
    from oracle import r2d2_torch as rt
    from oracle import ref_exec
    b = rt.make_sequences(B, S=S, seed=seed)
    p, tp = rt.init_params(0, torch.float32), rt.init_params(1, torch.float32)
    R = ref_exec.ReferenceR2D2(p, tp, seq_len=S, burn_in=bi)
    args = [b[k] for k in rt.TRAIN_FIELDS]
    f = R.fetch(args, ["main_q", "target_q", "target_value", "state_action_value"])
    g = {n: torch.from_numpy(np.asarray(v)) for n, v in R.gradients(R.feed(*args)).items()}
    gn = float(np.sqrt(sum(float(torch.sum(v.double() ** 2)) for v in g.values())))
    loss, td = R.agent.train(*args)
    rec = dict(B=B, S=S, burn_in=bi, seed=seed, loss=loss, td_error=td, grad_norm=gn, source=SOURCE)
    for k in ("main_q", "target_q", "target_value", "state_action_value"):
        rec[k] = f[k]
    _pack_grads(rec, g)
    np.savez_compressed(path, **rec)
    return rec


def a3c_case(path, B=3, A=4, seed=97531):
    """agent/a3c.py:85-103 ``Agent.train`` executed once (inputs regenerated from make_transitions(B, A, seed), parameters
    from init_params(0)); taps and gradients fetched from the agent's own graph."""
    from oracle import a3c_torch as at
    from oracle import ref_exec
    b = at.make_transitions(B, A=A, seed=seed)
    p = at.init_params(0, torch.float32, num_action=A)
    R = ref_exec.ReferenceA3C(p, num_action=A)
    args = [b[k] for k in at.TRAIN_FIELDS]
    f = R.fetch(args, ["policy", "value", "next_value", "clipped_r_ph", "discounts"])
    g = R.gradients(args)
    gn = float(np.sqrt(sum(np.sum(np.asarray(v, np.float64) ** 2) for v in g.values())))
    pi, bl, en, lr = R.agent.train(*args)
    rec = dict(B=B, A=A, seed=seed, pi_loss=float(pi), baseline_loss=float(bl), entropy=float(en), learning_rate=float(lr),
               grad_norm=gn, source=SOURCE)
    for k in ("policy", "value", "next_value"):
        rec[k] = np.asarray(f[k])
    rec["advantage"] = np.asarray(f["clipped_r_ph"]) + np.asarray(f["discounts"]) * rec["next_value"] - rec["value"]
    _pack_grads(rec, g)
    np.savez_compressed(path, **rec)
    return rec


REFEXEC_TAPS = ("vs", "clipped_rho", "vs_plus_1", "pg_advantage", "pi_loss", "baseline_loss", "entropy", "total_loss")


def _tensors(rec, key, tensors, most=64):
    """A dict of tensors as four arrays: ``key:names``, ``key:stride`` (per tensor), ``key:l2`` (per tensor, float64)
    and ``key:sample``, the strided samples of all tensors concatenated in that order (float64)."""
    vs = [np.asarray(v, np.float64) for v in tensors.values()]
    strides = [sample_stride(v.size, most) for v in vs]
    rec[key + ":names"] = np.array(list(tensors))
    rec[key + ":stride"] = np.array(strides)
    rec[key + ":l2"] = np.array([np.sqrt(np.sum(v ** 2)) for v in vs])
    rec[key + ":sample"] = np.concatenate([v.ravel()[::s] for v, s in zip(vs, strides)])


def refexec_case(path):
    """What tests/test_oracle_refexec.py compares the restatements with: the reference's own agents, V-trace
    functions, FIFO queue and prioritized replay memory executed over the shim, test by test (keys ``<test>:...``)."""
    import random

    from oracle import a3c_torch as a3
    from oracle import apex_torch as ax
    from oracle import ref_exec
    from oracle import r2d2_torch as rt
    rec = dict(source=SOURCE)
    f64 = torch.float64

    def impala(B, T, A, seed=4321, **cfg):
        batch = synthetic.make_batch(B, T=T, A=A, seed=seed)
        params = it.init_params(0, torch.float32, num_action=A)
        return [batch[k] for k in synthetic.TRAIN_FIELDS], params, dict(trajectory=T, num_action=A, **cfg)

    for clipping in ("abs_one", "soft_asymmetric"):
        args, params, cfg = impala(2, 6, 18, reward_clipping=clipping)
        R = ref_exec.ReferenceImpala(params, **cfg)
        for k, v in R.fetch(args, REFEXEC_TAPS + ("unrolled_first_policy", "unrolled_middle_value",
                                                  "unrolled_last_value", "clipped_r_ph")).items():
            rec["impala_%s:%s" % (clipping, k)] = v
        _tensors(rec, "impala_%s:grad" % clipping, R.gradients(args))

    args, params, cfg = impala(2, 6, 18)
    R = ref_exec.ReferenceImpala(params, **cfg)
    for step in range(3):
        rec["train3:%d:result" % step] = np.array(R.train(*args), np.float64)
        rec["train3:%d:global_step" % step] = R.global_step()
        _tensors(rec, "train3:%d:param" % step, R.params())
        _tensors(rec, "train3:%d:rms" % step, R.rms())
    rms = R.rms()
    rec["train3:rms_min"] = min(float(v.min()) for v in rms.values())
    rec["train3:rms_all_moved"] = all(np.any(v != 1.0) for v in rms.values())

    args, params, cfg = impala(4, 20, 18, seed=1234)
    R = ref_exec.ReferenceImpala(params, **cfg)
    for k, v in R.fetch(args, REFEXEC_TAPS).items():
        rec["b4t20:" + k] = v
    _tensors(rec, "b4t20:grad", R.gradients(args))

    args, params, cfg = impala(2, 6, 18)
    R32 = ref_exec.ReferenceImpala(params, float_dtype=torch.float32, **cfg)
    for k, v in R32.fetch(args, REFEXEC_TAPS).items():
        rec["f32:" + k] = v
    R32.ref.tf._shim.FLOAT = f64

    # variable names / sharing / parameter_sync / single-step inference: the learner holds init_params(0) before the sync
    ref = ref_exec.load(float_dtype=f64)
    tf = ref.tf
    kw = dict(trajectory=5, input_shape=[84, 84, 4], num_action=6, lstm_hidden_size=256, discount_factor=0.99,
              start_learning_rate=6e-4, end_learning_rate=0.0, learning_frame=10 ** 9, baseline_loss_coef=1.0,
              entropy_coef=0.05, gradient_clip_norm=40.0, reward_clipping="abs_one")
    learner = ref["agent.impala"].Agent(model_name="learner", learner_name="learner", **kw)
    rec["sync:names"] = np.array([v.op_name for v in tf.trainable_variables()])
    rec["sync:shapes"] = np.array([str(tuple(int(d) for d in v._shape)) for v in tf.trainable_variables()])
    actor = ref["agent.impala"].Agent(model_name="actor_0", learner_name="learner", **kw)
    rec["sync:n_vars_two_agents"] = len(tf.trainable_variables())
    rec["sync:n_global_to_session"] = len(actor.global_to_session)
    sess = tf.Session()
    learner.set_session(sess)
    src, dst = tf.trainable_variables("learner"), tf.trainable_variables("actor_0")
    for s, (n, v) in zip(src, it.init_params(0, torch.float32, num_action=6).items()):
        s.set(v.numpy())
    rec["sync:differ_before"] = any(np.any(s.numpy() != d.numpy()) for s, d in zip(src, dst))
    actor.sess = sess
    actor.parameter_sync()
    rec["sync:equal_after"] = all(np.array_equal(s.numpy(), d.numpy()) for s, d in zip(src, dst))
    rng = np.random.default_rng(3)
    state = rng.integers(0, 256, (84, 84, 4), dtype=np.uint8)
    h, c = rng.standard_normal(256).astype(np.float32) * 0.3, rng.standard_normal(256).astype(np.float32)
    np.random.seed(0)
    for k, v in zip(("action", "policy", "max", "h", "c"), actor.get_policy_and_action(state, 2, h, c)):
        rec["sync:" + k] = v

    args, params, cfg = impala(2, 6, 18)
    bad = synthetic.make_batch(2, T=7, A=18, seed=1)
    try:
        ref_exec.ReferenceImpala(params, **cfg).train(*[bad[k] for k in synthetic.TRAIN_FIELDS])
        rec["wrong_t:error"] = ""
    except Exception as e:
        rec["wrong_t:error"] = type(e).__name__

    ref = ref_exec.load(("optimizer.vtrace",), float_dtype=f64)
    vt, tf = ref["optimizer.vtrace"], ref.tf
    z = np.load(os.path.join(HERE, "vtrace_T18_B8.npz"))
    kw = {k: tf.constant(z[k]) for k in ("log_rhos", "discounts", "rewards", "values", "bootstrap_value")}
    run = lambda t: tf.Session().run(t)
    rec["vtrace:clip05_vs"], rec["vtrace:clip05_rho"] = run(list(vt.from_importance_weights(
        clip_rho_threshold=0.5, clip_pg_rho_threshold=7.0, **kw)))
    rng = np.random.default_rng(11)
    B, T, A = 5, 9, 7
    sm = lambda x: np.exp(x) / np.exp(x).sum(-1, keepdims=True)
    mu, pi = sm(rng.standard_normal((B, T, A))), sm(rng.standard_normal((B, T, A)))
    act = rng.integers(0, A, (B, T)).astype(np.int32)
    disc = (rng.random((B, T)) > 0.1) * 0.99
    rew, val, nval = rng.standard_normal((B, T)), rng.standard_normal((B, T)), rng.standard_normal((B, T))
    c = tf.constant
    rec["vtrace:softmax_vs"], rec["vtrace:softmax_rho"] = run(list(vt.from_softmax(
        c(mu), c(pi), c(act), c(disc), c(rew), c(val), c(nval), A)))
    adv = rng.standard_normal((B, T))
    got = run([vt.compute_policy_gradient_loss(c(pi), c(act), c(adv), A), vt.compute_baseline_loss(c(val), c(nval)),
               vt.compute_entropy_loss(c(pi)), vt.log_probs_from_softmax_and_actions(c(pi), c(act), A)] +
              list(vt.split_data(c(val))))
    for k, v in zip(("pg_loss", "baseline_loss", "entropy_loss", "log_probs", "split_first", "split_middle",
                     "split_last"), got):
        rec["vtrace:" + k] = v

    # the FIFO queue: which appended records each sample_batch returns (records as in the test, rng 5)
    ref = ref_exec.load(("distributed_queue.buffer_queue",), float_dtype=f64)
    T, shape, A, L, cap, batch = 5, [6, 6, 2], 4, 8, 8, 3
    rq = ref["distributed_queue.buffer_queue"].FIFOQueue(T, shape, A, cap, batch, 2, L)
    rq.set_session(ref.tf.Session())
    rng = np.random.default_rng(5)
    states = []
    for i in range(7):
        r = dict(unrolled_state=rng.integers(0, 256, (T, *shape), dtype=np.uint8),
                 unrolled_next_state=rng.integers(0, 256, (T, *shape), dtype=np.uint8),
                 unrolled_reward=rng.standard_normal(T).astype(np.float32), unrolled_done=rng.random(T) < 0.3,
                 unrolled_behavior_policy=rng.random((T, A)).astype(np.float32),
                 unrolled_action=rng.integers(0, A, T).astype(np.int32),
                 unrolled_previous_action=rng.integers(0, A, T).astype(np.int32),
                 unrolled_previous_h=rng.standard_normal((T, L)).astype(np.float32),
                 unrolled_previous_c=rng.standard_normal((T, L)).astype(np.float32))
        states.append(r["unrolled_state"])
        rq.append_to_queue(task=i % 2, **r)
    rec["fifo:size_full"] = rq.get_size()
    for j in range(2):
        rb = rq.sample_batch()
        rec["fifo:fields"] = np.array(rb._fields)
        rec["fifo:sample%d" % j] = [next(i for i, s in enumerate(states) if np.array_equal(s, x)) for x in rb.state]
    rec["fifo:size_left"] = rq.get_size()

    # train_impala.py:93-113 over the reference's own FIFOQueue and Agent
    B, T, A, L = 2, 5, 6, 256
    R = ref_exec.ReferenceImpala(it.init_params(0, torch.float32, num_action=A), trajectory=T, num_action=A)
    queue = R.ref["distributed_queue.buffer_queue"].FIFOQueue(T, [84, 84, 4], A, 128, B, 1, L)
    queue.set_session(R.sess)
    big = synthetic.make_batch(3 * B + 1 + B, T=T, A=A, seed=77)
    for i in range(big["state"].shape[0]):
        queue.append_to_queue(task=0, unrolled_state=big["state"][i], unrolled_next_state=big["state"][i],
                              unrolled_reward=big["reward"][i], unrolled_done=big["done"][i],
                              unrolled_behavior_policy=big["behavior_policy"][i], unrolled_action=big["action"][i],
                              unrolled_previous_action=big["previous_action"][i],
                              unrolled_previous_h=big["initial_h"][i], unrolled_previous_c=big["initial_c"][i])
    steps = 0
    while queue.get_size() > 3 * B:
        bt = queue.sample_batch()
        rec["loop:%d:records" % steps] = [next(i for i in range(big["state"].shape[0])
                                               if np.array_equal(big["state"][i], s)) for s in bt.state]
        rec["loop:%d:result" % steps] = np.array(R.agent.train(
            state=np.stack(bt.state), reward=np.stack(bt.reward), action=np.stack(bt.action), done=np.stack(bt.done),
            behavior_policy=np.stack(bt.behavior_policy), previous_action=np.stack(bt.previous_action),
            initial_h=np.stack(bt.previous_h), initial_c=np.stack(bt.previous_c))[:3], np.float64)
        steps += 1
    rec["loop:steps"], rec["loop:size_left"] = steps, queue.get_size()

    A = 4
    b = ax.make_transitions(3, A=A, seed=1357)
    R = ref_exec.ReferenceApex(ax.init_params(0, torch.float32, num_action=A),
                               ax.init_params(1, torch.float32, num_action=A), num_action=A)
    args = [b[k] for k in ax.TRAIN_FIELDS]
    for k, v in R.fetch(args, ["main_q_value", "next_main_q_value", "target_q_value", "target_value",
                               "state_action_value", "value_loss", "next_action"]).items():
        rec["apex:" + k] = v
    _tensors(rec, "apex:grad", R.gradients(R.feed(*args)))
    rec["apex:td_single"] = R.agent.get_td_error(*args[:6])
    for i in range(3):
        loss, td = R.agent.distributed_train(*args)
        rec["apex:%d:loss" % i], rec["apex:%d:td" % i] = loss, td
    rec["apex:target_differs"] = any(np.any(R.target_params()[n] != R.params()[n]) for n in R.var)
    _tensors(rec, "apex:param", R.params())
    m, v = R.adam_slots()
    _tensors(rec, "apex:adam_m", m)
    _tensors(rec, "apex:adam_v", v)

    S, bi = 6, 2
    b = rt.make_sequences(2, S=S, seed=2468)
    R = ref_exec.ReferenceR2D2(rt.init_params(0, torch.float32), rt.init_params(1, torch.float32), seq_len=S, burn_in=bi)
    args = [b[k] for k in rt.TRAIN_FIELDS]
    for k, v in R.fetch(args, ["main_q", "target_q", "target_value", "state_action_value", "value_loss"]).items():
        rec["r2d2:" + k] = v
    _tensors(rec, "r2d2:grad", R.gradients(R.feed(*args)))
    for i in range(3):
        loss, td = R.agent.train(*args)
        rec["r2d2:%d:loss" % i], rec["r2d2:%d:td" % i] = loss, td
    _tensors(rec, "r2d2:param", R.params())

    # the prioritized replay memory (plain NumPy in the reference), CPython ``random`` seeded per sample call
    RMem = ref_exec.load(("distributed_queue.buffer_queue",), float_dtype=f64)["distributed_queue.buffer_queue"].Memory
    cap, n = 37, 8
    rmem = RMem(cap)
    rng = np.random.default_rng(11)
    for i in range(cap + 9):
        rmem.add(float(abs(rng.standard_normal()) * 3), ("rec", i))
    rec["per:tree_filled"] = rmem.tree.tree.copy()
    rec["per:n_entries"], rec["per:write"] = rmem.tree.n_entries, rmem.tree.write
    calls = []                                         # per sample call: idx, weight, beta, record, tree, total
    for k in range(40):
        random.seed(1000 + k)
        rbatch, ridx, rw = rmem.sample(n)
        beta = rmem.beta
        for j in ridx[::2]:
            rmem.update(j, float(abs(rng.standard_normal())))
        calls.append((ridx, rw, beta, [r[1] for r in rbatch], rmem.tree.tree.copy(), rmem.tree.total()))
    for name, col in zip(("idx", "weight", "beta", "record", "tree", "total"), zip(*calls)):
        rec["per:" + name] = np.array(col)

    A = 5
    for clipping in ("abs_one", "soft_asymmetric"):
        b = a3.make_transitions(4, A=A, seed=97)
        b["reward"] = (b["reward"] * 3).astype(np.float32)
        R = ref_exec.ReferenceA3C(a3.init_params(0, torch.float32, num_action=A), num_action=A, reward_clipping=clipping)
        args = [b[k] for k in a3.TRAIN_FIELDS]
        key = "a3c_" + clipping
        for k, v in R.fetch(args, ["policy", "value", "next_value", "pi_loss", "baseline_loss", "entropy",
                                   "total_loss"]).items():
            rec["%s:%s" % (key, k)] = v
        _tensors(rec, key + ":grad", R.gradients(args))
        for i in range(3):
            rec["%s:%d:result" % (key, i)] = np.array([float(x) for x in R.agent.train(*args)])
        _tensors(rec, key + ":param", R.params())
        m, v = R.adam_slots()
        _tensors(rec, key + ":adam_m", m)
        _tensors(rec, key + ":adam_v", v)
    np.savez_compressed(path, **rec)
    return rec


if __name__ == "__main__":
    which = set(sys.argv[1:]) or {"impala", "vtrace", "apex", "r2d2", "a3c", "refexec"}
    if "impala" in which:
        for B, T, seed in ((2, 6, 4321), (4, 20, 1234)):        # small case; BASELINE configs[0] (T=20, B=4)
            r = learner_case(B, T, 18, seed, os.path.join(HERE, "impala_step_B%d_T%d.npz" % (B, T)))
            print("B%d T%d: pi %.6f bl %.6f ent %.6f gn %.6f" % (B, T, r["pi_loss"], r["baseline_loss"], r["entropy"],
                                                                 r["grad_norm"]))
    if "vtrace" in which:
        vtrace_case(os.path.join(HERE, "vtrace_T18_B8.npz"))
    if "apex" in which:
        r = apex_case(os.path.join(HERE, "apex_step_B3.npz"))
        print("apex loss %.6f gn %.6f" % (r["loss"], r["grad_norm"]))
    if "r2d2" in which:
        r = r2d2_case(os.path.join(HERE, "r2d2_step_B2_S6.npz"))
        print("r2d2 loss %.6f gn %.6f" % (r["loss"], r["grad_norm"]))
    if "a3c" in which:
        r = a3c_case(os.path.join(HERE, "a3c_step_B3.npz"))
        print("a3c pi %.6f bl %.6f ent %.6f gn %.6f" % (r["pi_loss"], r["baseline_loss"], r["entropy"], r["grad_norm"]))
    if "refexec" in which:
        refexec_case(os.path.join(HERE, "refexec.npz"))
