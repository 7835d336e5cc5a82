"""Regenerates tests/golden/impala_step_*.npz and vtrace_T18_B8.npz under a REAL tensorflow==1.14.0 (the version the
reference pins, README.md:14 / Dockerfile:2), for any machine that has one (CPython <= 3.7):

    pip install tensorflow==1.14.0 numpy torch          # torch only for oracle.impala_torch.init_params (seeded weights)
    python tests/golden/make_golden_tf1.py --reference /path/to/distributed_reinforcement_learning [--check]

It imports the reference's own ``agent/impala.py`` and ``optimizer/vtrace.py``, loads the seeded parameters
(oracle/impala_torch.py::init_params(0)) into the TF variables in creation order, feeds the seeded synthetic batch
(oracle/synthetic.py::make_batch) and writes the same keys as make_golden.py with ``source = "tensorflow 1.14.0"``.
With ``--check`` nothing is written: the TF results are compared with the committed files (which were produced by
executing the same reference files over oracle/tf1_shim) at float32 resolution (1e-4 relative, the north_star bar).

NOT runnable in the build container (no TF wheel for CPython 3.12, no network) -- it is committed so that the last
unpinned piece, TF's own op kernels versus the shim's restatement of them, can be closed wherever TF 1.14 exists.
"""
import argparse
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
ORDER = ("conv2d", "conv2d_1", "conv2d_2", "dense", "dense_1", "rnn/lstm_cell", "dense_2", "dense_3", "dense_4",
         "dense_5", "dense_6", "dense_7")
NAMES = ("conv1", "conv2", "conv3", "emb1", "emb2", "lstm", "actor1", "actor2", "actor3", "critic1", "critic2", "critic3")


def impala_case(tf, impala, B, T, A, seed):
    sys.path.insert(0, ROOT)
    import torch
    from oracle import impala_torch as it
    from oracle import synthetic
    tf.reset_default_graph()
    agent = impala.Agent(trajectory=T, input_shape=[84, 84, 4], num_action=A, lstm_hidden_size=256, discount_factor=0.99,
                         start_learning_rate=0.0006, end_learning_rate=0.0, learning_frame=1000000000,
                         baseline_loss_coef=1.0, entropy_coef=0.05, gradient_clip_norm=40.0, reward_clipping="abs_one",
                         model_name="learner", learner_name="learner")
    sess = tf.Session()
    agent.set_session(sess)
    params = it.init_params(0, torch.float32, num_action=A)
    by_name = {v.op.name: v for v in tf.trainable_variables()}
    var = {}
    for tf_name, our in zip(ORDER, NAMES):
        var[our + ".w"] = by_name["learner/impala/%s/kernel" % tf_name]
        var[our + ".b"] = by_name["learner/impala/%s/bias" % tf_name]
    for n, v in params.items():
        var[n].load(v.numpy(), sess)
    batch = synthetic.make_batch(B, T=T, A=A, seed=seed)
    feed = {agent.t_s_ph: np.stack(batch["state"]) / 255, agent.t_pa_ph: batch["previous_action"],
            agent.t_initial_h_ph: batch["initial_h"], agent.t_initial_c_ph: batch["initial_c"], agent.a_ph: batch["action"],
            agent.d_ph: batch["done"], agent.r_ph: batch["reward"], agent.b_ph: batch["behavior_policy"]}
    grads = tf.gradients(agent.total_loss, [var[n] for n in var])
    taps = [agent.vs, agent.clipped_rho, agent.vs_plus_1, agent.pg_advantage, agent.unrolled_first_policy,
            agent.unrolled_first_value, agent.total_loss]
    tv, gv = sess.run([taps, grads], feed_dict=feed)
    pi, bl, en, lr = agent.train(*[batch[k] for k in synthetic.TRAIN_FIELDS])
    rec = dict(B=B, T=T, A=A, seed=seed, pi_loss=pi, baseline_loss=bl, entropy=en, learning_rate=lr,
               grad_norm=float(np.sqrt(sum(np.sum(np.asarray(g, np.float64) ** 2) for g in gv))), total_loss=float(tv[6]),
               source="tensorflow %s" % tf.__version__)
    for k, v in zip(("vs", "clipped_rho", "vs_plus_1", "pg_advantage", "first_policy", "first_value"), tv):
        rec[k] = v
    for n, g in zip(var, gv):
        s = rec["stride_" + n] = sample_stride(g.size)
        rec["gradsample_" + n] = g.ravel()[::s].astype(np.float32)
        rec["gradl2_" + n] = np.float64(np.sqrt(np.sum(g.astype(np.float64) ** 2)))
        rec["paramsample_" + n] = sess.run(var[n]).ravel()[::s]
        rec["rmssample_" + n] = sess.run(agent.optimizer.get_slot(var[n], "rms")).ravel()[::s]
    return rec


def sample_stride(n, most=512):
    """The sampling of make_golden.py: a stride that keeps at most ``most`` elements, odd."""
    return -(-n // most) | 1


def compare(rec, path, tol=1e-4):
    z = np.load(path)
    worst = 0.0
    for k in rec:
        if k in ("source", "B", "T", "A", "seed"):
            continue
        a, b = np.asarray(rec[k], np.float64), np.asarray(z[k], np.float64)
        err = float(np.max(np.abs(a - b)) / max(np.max(np.abs(b)), 1e-30))
        worst = max(worst, err)
        print("%-28s rel err %.3e%s" % (k, err, "" if err < tol or k.startswith("paramsample") else "   <-- above the bar"))
    return worst


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--reference", required=True)
    ap.add_argument("--check", action="store_true")
    a = ap.parse_args()
    sys.path.insert(0, a.reference)
    import tensorflow as tf
    assert tf.__version__.startswith("1."), "this script is for a real TF1; the build container uses make_golden.py"
    from agent import impala
    for B, T, seed in ((2, 6, 4321), (4, 20, 1234)):
        rec = impala_case(tf, impala, B, T, 18, seed)
        path = os.path.join(HERE, "impala_step_B%d_T%d.npz" % (B, T))
        if a.check:
            print("== %s: worst rel err %.3e" % (os.path.basename(path), compare(rec, path)))
        else:
            np.savez_compressed(path, **rec)
