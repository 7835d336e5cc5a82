"""Parity harness of the Ape-X learner: runs the CUDA step (through ``drl_apex_*``) and the float64 CPU oracle
(``oracle/apex_torch.py``) on the same seeded minibatch and reports per-tensor relative errors
(max|gpu - oracle| / max|oracle|, bar 1e-4 as for the IMPALA path; see tests/parity.py for the ReLU-kink handling, which
is the same here: the oracle is evaluated at the GPU's activation pattern of the differentiated pass).

Two things are specific to this path:
* double-DQN argmax: if the two best next_main_q values of a row are within float32 rounding the GPU may pick the
  other action; the oracle is evaluated at the GPU's choice and the harness asserts that they only differ where the
  oracle's gap is < 1e-5 (``argmax/disagree_with_gap``).
* Adam: the first updates are ~ lr * sign(g), ill-conditioned in g for |g| ~ 1e-8, so the applied update is checked
  against TF1's ApplyAdam formula evaluated in float64 FROM THE GPU'S OWN GRADIENT AND SLOTS (the gradient itself is
  checked against the oracle to 1e-4), and the oracle is then set to the GPU's state so that later steps compare like
  with like.
"""
import numpy as np
import torch

from oracle import apex_torch as ax
from oracle import impala_torch as it
from parity import TOL, rel_err, failures, worst   # noqa: F401  (same bar and failure rules)


def native_apex(B, A, params, target, **kw):
    from distributed_reinforcement_learning_b200.apex_learner import MAIN, TARGET, NativeApexLearner
    eng = NativeApexLearner(batch=B, num_action=A, **kw)
    eng.set_params(ax.flatten_params(params), MAIN)
    eng.set_params(ax.flatten_params(target), TARGET)
    return eng


def gpu_masks(eng, B, A):
    M = 2 * B

    def first(name, per_row, shape):
        return torch.from_numpy(eng.read_buffer(name, M * per_row).reshape((M,) + shape)[:B] > 0)
    masks = {"a1": first("a1", 20 * 20 * 32, (20, 20, 32)), "a2": first("a2", 9 * 9 * 64, (9, 9, 64)),
             "a3": first("a3", 7 * 7 * 64, (7, 7, 64)),
             "e1": torch.from_numpy(eng.read_buffer("e1", A * 256).reshape(A, 256) > 0),
             "emb": torch.from_numpy(eng.read_buffer("emb", A * 256).reshape(A, 256) > 0)}
    for name in ("hid1", "hid2"):
        buf = eng.read_buffer(name, 2 * M * 256).reshape(2, M, 256)[:, :B] > 0
        masks["value" + name[-1]] = torch.from_numpy(buf[0])
        masks["mean" + name[-1]] = torch.from_numpy(buf[1])
    return masks


def adam_expected(p0, g, m0, v0, gn, clip, lr, b1p, b2p):
    scale = clip * min(1.0 / gn, 1.0 / clip) if gn > 0 else 1.0
    gc = g * scale
    m = m0 + (gc - m0) * (1.0 - ax.BETA1)
    v = v0 + (gc * gc - v0) * (1.0 - ax.BETA2)
    alpha = lr * np.sqrt(1.0 - b2p) / (1.0 - b1p)
    return p0 - m * alpha / (np.sqrt(v) + ax.ADAM_EPS), m, v


def compare_step(B, A=4, seed=4321, steps=1, reward_clipping="abs_one", sync_target_at=None, gradient_clip_norm=None,
                 learning_frame=None, end_learning_rate=None, **kw):
    """``gradient_clip_norm`` / ``learning_frame`` / ``end_learning_rate``: optional, for both the oracle and the native
    learner (the configuration defaults otherwise); with a clip norm given, ``clip_engaged`` entries are 0 where the
    step's norm exceeded it and inf where it did not."""
    params = ax.init_params(0, torch.float32, num_action=A)
    target = ax.init_params(1, torch.float32, num_action=A)
    schedule = {k: v for k, v in (("gradient_clip_norm", gradient_clip_norm), ("learning_frame", learning_frame),
                                  ("end_learning_rate", end_learning_rate)) if v is not None}
    cfg = dict(num_action=A, reward_clipping=reward_clipping)
    L = ax.Learner(params, target, torch.float64, **cfg, **schedule)
    eng = native_apex(B, A, params, target, reward_clipping=reward_clipping, **schedule, **kw)
    errs = {}
    flips = elems = 0
    max_abs = 0.0
    disagree = 0
    try:
        for s in range(steps):
            tag = "" if steps == 1 else "@%d" % s
            if sync_target_at is not None and s == sync_target_at:
                eng.target_to_main()
                L.target_to_main()
            b = ax.make_transitions(B, A=A, seed=seed + s)
            args = [b[k] for k in ax.TRAIN_FIELDS]
            st0 = eng.get_opt_state()
            p0 = eng.get_params()
            slot = s % eng.num_slots
            eng.stage(slot, *args)
            out, td = eng.step(slot)
            taps = eng.taps()
            masks = gpu_masks(eng, B, A)
            # double-DQN argmax at the GPU's choice; disagreements are only allowed at float32-level ties
            with torch.no_grad():
                o0 = L.losses(*args[:-1], is_weight=args[-1])
            nq = o0["next_main_q"].numpy()
            gpu_na = np.argmax(taps["next_main_q"], axis=1)
            ora_na = np.argmax(nq, axis=1)
            top2 = np.sort(nq, axis=1)[:, -2:]
            gap = top2[:, 1] - top2[:, 0]
            disagree += int(np.sum((gpu_na != ora_na) & (gap > 1e-5)))
            with it.activation_pattern(masks) as stt:
                res, o, grads, gn, lr = L.distributed_train(*args, return_all=True, next_action=gpu_na)
            flips, elems, max_abs = flips + stt["flips"], elems + stt["elems"], max(max_abs, stt["max_abs_at_flip"])
            errs["loss" + tag] = rel_err(out["loss"], res[0])
            errs["td_error" + tag] = rel_err(td, res[1])
            errs["lr" + tag] = abs(out["learning_rate"] - lr)
            errs["grad_norm" + tag] = rel_err(out["grad_norm"], gn)
            if gradient_clip_norm is not None:
                errs["clip_engaged" + tag] = 0.0 if gn > gradient_clip_norm else float("inf")
            if out["step"] != s + 1:
                errs["step" + tag] = float("inf")
            for k in ("main_q", "next_main_q", "target_q", "target_value", "state_action_value"):
                errs["tap/" + k + tag] = rel_err(taps[k], o[k].detach().numpy())
            g_gpu_flat = eng.get_grads()
            gd = ax.unflatten_params(g_gpu_flat, torch.float64, num_action=A)
            for n in grads:
                errs["grad/" + n + tag] = rel_err(gd[n].numpy(), grads[n].detach().numpy())
            # forward activations and activation gradients of the differentiated pass (rows [0, B))
            if s == 0:
                tp, ag = o["taps"], o.get("act_grads", {})
                M = 2 * B
                for nm, shp in (("a1", (20, 20, 32)), ("a2", (9, 9, 64)), ("a3", (7, 7, 64))):
                    got = eng.read_buffer(nm, M * int(np.prod(shp))).reshape((M,) + shp)[:B]
                    errs["act/" + nm] = rel_err(got, tp[nm].detach().numpy().reshape((B,) + shp))
                    if ag.get(nm) is not None:
                        gr = ag[nm].detach().numpy().reshape((B,) + shp) * masks[nm].numpy().astype(np.float64)
                        gotb = eng.read_buffer("d" + nm, B * int(np.prod(shp))).reshape((B,) + shp)
                        errs["bwd/d" + nm] = rel_err(gotb, gr)
            # Adam from the GPU's own gradient and slots
            st1 = eng.get_opt_state()
            p1 = eng.get_params()
            gn_gpu = float(np.sqrt(np.sum(g_gpu_flat.astype(np.float64) ** 2)))
            exp_p, exp_m, exp_v = adam_expected(p0.astype(np.float64), g_gpu_flat.astype(np.float64),
                                                st0["m"].astype(np.float64), st0["v"].astype(np.float64), gn_gpu,
                                                L.cfg["gradient_clip_norm"], float(out["learning_rate"]),
                                                st0["beta1_power"], st0["beta2_power"])
            floor = 4.0 * np.finfo(np.float32).eps * np.max(np.abs(p0)) / TOL
            errs["update/adam" + tag] = float(np.max(np.abs(p1 - exp_p)) / (np.max(np.abs(exp_p - p0)) + floor))
            errs["adam/m" + tag] = rel_err(st1["m"], exp_m)
            errs["adam/v" + tag] = rel_err(st1["v"], exp_v)
            errs["adam/beta1_power" + tag] = abs(st1["beta1_power"] - float(np.float32(st0["beta1_power"]) * np.float32(0.9)))
            errs["adam/beta2_power" + tag] = abs(st1["beta2_power"] - float(np.float32(st0["beta2_power"]) * np.float32(0.999)))
            # the target network must not move
            # teacher forcing: continue the oracle from the GPU's state
            pd = ax.unflatten_params(p1, torch.float64, num_action=A)
            md = ax.unflatten_params(st1["m"], torch.float64, num_action=A)
            vd = ax.unflatten_params(st1["v"], torch.float64, num_action=A)
            with torch.no_grad():
                for n in L.params:
                    L.params[n].copy_(pd[n])
                    L.m[n].copy_(md[n])
                    L.v[n].copy_(vd[n])
            L.beta1_power, L.beta2_power = np.float32(st1["beta1_power"]), np.float32(st1["beta2_power"])
        from distributed_reinforcement_learning_b200.apex_learner import TARGET
        tgt = ax.unflatten_params(eng.get_params(TARGET), torch.float64, num_action=A)
        errs["target_unchanged"] = max(float((tgt[n] - L.target[n]).abs().max()) for n in L.target)
        errs["argmax/disagree_with_gap"] = float(disagree)
        errs["kink/flip_fraction"] = flips / max(elems, 1)
        errs["kink/max_abs_at_flip"] = max_abs
    finally:
        eng.close()
    return errs


def apex_failures(errs):
    bad = failures({k: v for k, v in errs.items() if not k.startswith(("adam/beta", "target_unchanged", "argmax/"))})
    for k, v in errs.items():
        if k.startswith("adam/beta") and not v <= 1e-7:
            bad[k] = v
        if k in ("target_unchanged", "argmax/disagree_with_gap") and not v == 0.0:
            bad[k] = v
    return bad
