"""CPU: pins the learner oracle (oracle/impala_torch.py) -- TF1 semantics restated from SURVEY.md App. A --
by self-consistency (reference-shaped graph vs deduplicated forward, float32 vs float64), hand-derived
head gradients (App. A.5), hand-computed optimizer steps, and the committed golden fixture."""
import os

import numpy as np
import torch

from oracle import impala_torch as it
from oracle import synthetic


def _args(b):
    return [b[k] for k in synthetic.TRAIN_FIELDS]


def test_parameter_inventory():
    assert it.param_count() == 4153267                              # SURVEY.md App. A.6
    specs = dict(it.param_specs())
    assert specs["lstm.w"] == (3648, 1024) and specs["conv1.w"] == (8, 8, 4, 32) and specs["critic3.w"] == (256, 1)
    p = it.init_params(0)
    flat = it.flatten_params(p)
    back = it.unflatten_params(flat)
    assert all(torch.equal(p[k], back[k]) for k in p)
    assert float(p["lstm.b"].abs().max()) == 0.0
    lim = np.sqrt(6.0 / (3648 + 1024))
    assert float(p["lstm.w"].abs().max()) <= lim + 1e-7


def test_uint8_normalisation_is_a_true_fp32_divide():
    """agent/impala.py:133 divides in float64 then feeds float32: identical to float32(u)/255f for every byte,
    but NOT to u * (1/255f) (SURVEY.md section 7)."""
    u = np.arange(256)
    ref = (u.astype(np.float64) / 255).astype(np.float32)
    assert np.array_equal(ref, u.astype(np.float32) / np.float32(255))
    assert np.sum(ref != u.astype(np.float32) * np.float32(1 / 255)) > 0


def test_reference_shaped_equals_dedup_and_shift_identity():
    b = synthetic.make_batch(2, T=6)
    p = it.init_params(0)
    kw = dict(trajectory=6)
    o_ref, g_ref = it.Learner(p, torch.float64, "reference", **kw).gradients(*_args(b))
    o_ded, g_ded = it.Learner(p, torch.float64, "dedup", **kw).gradients(*_args(b))
    for k in ("vs", "pg_advantage", "pi_loss", "baseline_loss", "entropy"):
        np.testing.assert_allclose(o_ref[k].detach().numpy(), o_ded[k].detach().numpy(), rtol=1e-10, atol=1e-12)
    np.testing.assert_allclose(it.flatten_grads(g_ref), it.flatten_grads(g_ded), rtol=1e-8, atol=1e-12)
    # App. C.4: first[:, i+1] == middle[:, i] == last[:, i-1]
    np.testing.assert_allclose(o_ref["first_policy"][:, 1:].detach().numpy(),
                               o_ref["middle_policy"][:, :-1].detach().numpy(), rtol=1e-12)
    np.testing.assert_allclose(o_ref["middle_value"][:, 1:].detach().numpy(),
                               o_ref["last_value"][:, :-1].detach().numpy(), rtol=1e-12)


def test_float32_tracks_float64():
    b = synthetic.make_batch(2, T=5)
    p = it.init_params(0)
    _, g64 = it.Learner(p, torch.float64, "dedup", trajectory=5).gradients(*_args(b))
    _, g32 = it.Learner(p, torch.float32, "dedup", trajectory=5).gradients(*_args(b))
    for n in g64:
        a, c = g64[n].numpy(), g32[n].double().numpy()
        assert np.abs(a - c).max() <= 2e-5 * max(np.abs(a).max(), 1e-30), n


def test_head_gradients_match_hand_derivation():
    """App. A.5: dL/dV = -(vs - V); dL/dlogit_k = pi_k (g_k - sum_a pi_a g_a),
    g_a = -adv [a = a_t] / (pi_a + 1e-8) + 0.05 (log pi_a + 1)."""
    rng = np.random.default_rng(0)
    B, Tp, A = 3, 4, 5
    logits = torch.tensor(rng.standard_normal((B, Tp, A)), requires_grad=True)
    V = torch.tensor(rng.standard_normal((B, Tp)), requires_grad=True)
    a = torch.tensor(rng.integers(0, A, (B, Tp)))
    adv = torch.tensor(rng.standard_normal((B, Tp)))
    vs = torch.tensor(rng.standard_normal((B, Tp)))
    pi = torch.softmax(logits, -1)
    loss = it.compute_policy_gradient_loss(pi, a, adv, A) + it.compute_baseline_loss(vs, V) * 1.0 + \
        it.compute_entropy_loss(pi) * 0.05
    gl, gv = torch.autograd.grad(loss, [logits, V])
    p = pi.detach().numpy()
    onehot = np.eye(A)[a.numpy()]
    g = -adv.numpy()[..., None] * onehot / (p + 1e-8) + 0.05 * (np.log(p) + 1)
    exp = p * (g - np.sum(p * g, -1, keepdims=True))
    np.testing.assert_allclose(gl.numpy(), exp, rtol=1e-9, atol=1e-12)
    np.testing.assert_allclose(gv.numpy(), -(vs.numpy() - V.detach().numpy()), rtol=1e-12)


def test_only_first_window_rows_receive_gradient():
    """Rows t = T-2, T-1 feed V-trace bootstraps only (stop_gradient): perturbing their frames changes vs but
    the gradient flows through the first T-2 rows (optimizer/vtrace.py:103, agent/impala.py:78,88)."""
    b = synthetic.make_batch(1, T=5)
    p = it.init_params(0)
    L = it.Learner(p, torch.float64, "dedup", trajectory=5)
    t = L._prep(*_args(b))
    x = t["x"].clone().requires_grad_(True)
    t["x"] = x
    (fp, fv, mp, mv, lp, lv), _ = L._unrolled(t)
    fv.sum().backward()
    gx = x.grad.abs().reshape(1, 5, -1).sum(-1)[0]
    assert float(gx[3]) == 0.0 and float(gx[4]) == 0.0 and float(gx[0]) > 0


def test_polynomial_decay_float32():
    assert it.polynomial_decay_f32(6e-4, 0, 1e9, 0.0) == np.float32(6e-4)
    assert it.polynomial_decay_f32(6e-4, 5, 1e9, 0.0) == np.float32(6e-4)      # 1 - 5e-9 == 1 in float32
    assert abs(float(it.polynomial_decay_f32(6e-4, 5e8, 1e9, 0.0)) - 3e-4) < 1e-10
    assert it.polynomial_decay_f32(6e-4, 2e9, 1e9, 0.0) == 0.0


def test_rmsprop_and_clip_by_global_norm_hand_step():
    """One update by hand: ms0 = 1, ms += (g^2 - ms) * 0.01, w -= lr * g / sqrt(ms + 0.1); scale = 40 * min(1/norm, 1/40)."""
    b = synthetic.make_batch(1, T=4)
    p = it.init_params(0)
    L = it.Learner(p, torch.float64, "dedup", trajectory=4)
    _, g = it.Learner(p, torch.float64, "dedup", trajectory=4).gradients(*_args(b))
    res, out, g2, gn = L.train(*_args(b), return_all=True)
    norm = np.sqrt(sum(float((v.double() ** 2).sum()) for v in g.values()))
    assert abs(gn - norm) < 1e-9 * norm
    scale = 40.0 * min(1.0 / norm, 1.0 / 40.0)
    for n in ("conv1.w", "lstm.b", "critic3.b"):
        gc = g[n].numpy() * scale
        ms = 1.0 + (gc * gc - 1.0) * (1 - 0.99)
        w = p[n].double().numpy() - float(np.float32(6e-4)) * gc / np.sqrt(ms + 0.1)
        np.testing.assert_allclose(L.params[n].detach().numpy(), w, rtol=1e-12, atol=1e-15)
        np.testing.assert_allclose(L.ms[n].numpy(), ms, rtol=1e-12)
    assert L.step == 1 and res[3] == float(np.float32(6e-4))
    # large-gradient case: the clip engages
    big = {k: v * 1e3 for k, v in g.items()}
    nb = norm * 1e3
    assert abs(40.0 * min(1.0 / nb, 1.0 / 40.0) * nb - 40.0) < 1e-9


def test_reward_clipping_modes():
    b = synthetic.make_batch(2, T=4)
    b["reward"][0, 0], b["reward"][0, 1] = 3.0, -7.0
    p = it.init_params(0)
    o1 = it.Learner(p, torch.float64, "dedup", trajectory=4, reward_clipping="abs_one").losses(*_args(b))
    o2 = it.Learner(p, torch.float64, "dedup", trajectory=4, reward_clipping="soft_asymmetric").losses(*_args(b))
    assert not np.allclose(o1["vs"].numpy(), o2["vs"].numpy())
    r = torch.tensor([3.0, -7.0])
    sq = torch.tanh(r / 5.0)
    exp = torch.where(r < 0, 0.3 * sq, sq) * 5.0
    np.testing.assert_allclose(exp.numpy(), [5 * np.tanh(0.6), 1.5 * np.tanh(-1.4)], rtol=1e-6)


def test_golden_fixture_matches_oracle():
    z = np.load(os.path.join(os.path.dirname(__file__), "golden", "impala_step_B2_T6.npz"))
    B, T, A = int(z["B"]), int(z["T"]), int(z["A"])
    b = synthetic.make_batch(B, T=T, A=A, seed=int(z["seed"]))
    L = it.Learner(it.init_params(0, num_action=A), torch.float64, "dedup", trajectory=T, num_action=A)
    res, out, g, gn = L.train(*_args(b), return_all=True)
    for k, v in zip(("pi_loss", "baseline_loss", "entropy"), res[:3]):
        assert abs(v - float(z[k])) < 1e-9 * abs(float(z[k]))
    assert abs(gn - float(z["grad_norm"])) < 1e-9 * gn
    np.testing.assert_allclose(out["vs"].numpy(), z["vs"], rtol=1e-9)
    for n in g:
        s = int(z["stride_" + n])
        np.testing.assert_allclose(g[n].numpy().ravel()[::s], z["gradsample_" + n], rtol=1e-4, atol=1e-9, err_msg=n)
        np.testing.assert_allclose(np.sqrt(np.sum(g[n].numpy() ** 2)), float(z["gradl2_" + n]), rtol=1e-9, err_msg=n)
