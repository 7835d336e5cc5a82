"""Shared parity harness: runs the CUDA learner (through the C-ABI) and the CPU oracle on the same
seeded synthetic batch and reports per-tensor relative errors.  Used by the -m gpu tests, by
``__graft_entry__.smoke()`` and by ``tools/diagnose.py``.

Error metric (the "1e-4 relative fp32" bar of BASELINE.json's north_star): for each tensor,
    rel = max|gpu - oracle| / max(max|oracle|, 1e-30)
with the oracle evaluated in float64 from the same float32 parameters and inputs.

ReLU kinks.  ReLU' is discontinuous at 0.  With ~2 M ReLU outputs per 8 trajectories, a few
pre-activations land within float32 rounding (|x| ~ 1e-8) of zero, where float32 and float64
legitimately disagree on the mask; ONE such flip changes that image's conv gradients by O(1e-3) (measured:
tools/debug_da3.py).  Any two float32 implementations (TF1's Eigen kernels included) differ the same way.
The harness therefore evaluates the float64 oracle AT THE GPU'S ACTIVATION PATTERN
(``oracle.impala_torch.activation_pattern``): forward activations are still compared unmasked, and the
harness asserts that mask flips are rare (< 1e-5 of the ReLU outputs) and occur only where the oracle's
pre-activation is ~0 (|x| < 1e-5 of the layer scale) -- reported as ``kink/flip_fraction`` and
``kink/max_abs_at_flip``.
"""
import numpy as np
import torch

from oracle import impala_torch as it
from oracle import synthetic

TOL = 1e-4          # north_star: within 1e-4 relative fp32
FLIP_FRACTION_MAX = 1e-5
FLIP_ABS_MAX = 1e-5


def rel_err(a, b):
    a = np.asarray(a, np.float64)
    b = np.asarray(b, np.float64)
    if a.shape != b.shape:
        return float("inf")
    if not np.all(np.isfinite(a)):
        return float("inf")
    return float(np.max(np.abs(a - b)) / max(np.max(np.abs(b)), 1e-30)) if b.size else 0.0


def to_time_major(x_bt):
    """[B, T, ...] -> [T*B, ...] rows m = t*B + b (device activation layout)."""
    x = np.asarray(x_bt)
    return np.swapaxes(x, 0, 1).reshape((x.shape[0] * x.shape[1],) + x.shape[2:])


def to_batch_major(x_m, B, T):
    """device rows [T*B, ...] -> oracle rows [B*T, ...] (row b*T + t)."""
    x = np.asarray(x_m)
    return np.swapaxes(x.reshape((T, B) + x.shape[1:]), 0, 1).reshape((B * T,) + x.shape[1:])


SCHEDULE_KEYS = ("gradient_clip_norm", "learning_frame", "end_learning_rate")


def make_case(B, T=20, A=18, seed=1234, param_seed=0, reward_clipping="abs_one", **schedule):
    """``schedule``: optional gradient_clip_norm / learning_frame / end_learning_rate for both the oracle and the
    native learner (the configuration defaults otherwise)."""
    assert set(schedule) <= set(SCHEDULE_KEYS), schedule
    batch = synthetic.make_batch(B, T=T, A=A, seed=seed)
    params = it.init_params(param_seed, torch.float32, num_action=A)
    cfg = dict(trajectory=T, num_action=A, reward_clipping=reward_clipping,
               **{k: v for k, v in schedule.items() if v is not None})
    return batch, params, cfg


def native_learner(batch, params, cfg, **kw):
    from distributed_reinforcement_learning_b200.learner import NativeLearner
    B = batch["state"].shape[0]
    eng = NativeLearner(batch=B, trajectory=cfg["trajectory"], num_action=cfg["num_action"],
                        reward_clipping=cfg.get("reward_clipping", "abs_one"),
                        **{k: cfg[k] for k in SCHEDULE_KEYS if k in cfg}, **kw)
    eng.set_params(it.flatten_params(params))
    return eng


def gpu_activation_pattern(eng, B, T, A):
    """ReLU masks of the forward pass the engine just ran, in the oracle's row order."""
    M = B * T

    def rows(name, per_row, shape):
        buf = eng.read_buffer(name, M * per_row).reshape((M,) + shape)
        return torch.from_numpy(to_batch_major(buf > 0, B, T))
    masks = {"a1": rows("a1", 20 * 20 * 32, (20, 20, 32)), "a2": rows("a2", 9 * 9 * 64, (9, 9, 64)),
             "a3": rows("a3", 7 * 7 * 64, (7, 7, 64)),
             "e1": torch.from_numpy(eng.read_buffer("e1", A * 256).reshape(A, 256) > 0),
             "emb": torch.from_numpy(eng.read_buffer("emb", A * 256).reshape(A, 256) > 0)}
    for name in ("hid1", "hid2"):
        buf = eng.read_buffer(name, 2 * M * 256).reshape(2, M, 256) > 0
        masks["actor" + name[-1]] = torch.from_numpy(to_batch_major(buf[0], B, T))
        masks["critic" + name[-1]] = torch.from_numpy(to_batch_major(buf[1], B, T))
    return masks


def compare_step(B, T=20, A=18, seed=1234, steps=1, reward_clipping="abs_one", layers=True, gradient_clip_norm=None,
                 learning_frame=None, end_learning_rate=None, **kw):
    """Returns {name: rel_err} for activations, taps, losses, every parameter gradient, and the applied
    update / RMSProp slots after each of `steps` updates (GPU step first, then the float64 oracle step
    evaluated at the GPU's ReLU activation pattern).  With ``gradient_clip_norm`` given, ``clip_engaged`` entries
    are 0 where the step's norm exceeded it and inf where it did not."""
    batch, params, cfg = make_case(B, T, A, seed, reward_clipping=reward_clipping,
                                   gradient_clip_norm=gradient_clip_norm, learning_frame=learning_frame,
                                   end_learning_rate=end_learning_rate)
    L = it.Learner(params, torch.float64, "dedup", **cfg)
    eng = native_learner(batch, params, cfg, **kw)
    args = [batch[k] for k in synthetic.TRAIN_FIELDS]
    M, Mb = B * T, B * (T - 2)
    errs = {}
    flips = elems = 0
    max_abs = 0.0
    try:
        for s in range(steps):
            tag = "" if steps == 1 else "@%d" % s
            p_before = {n: v.detach().clone() for n, v in L.params.items()}
            eng.stage(s % eng.num_slots, *args)
            out = eng.step(s % eng.num_slots)
            masks = gpu_activation_pattern(eng, B, T, A)
            with it.activation_pattern(masks) as st:
                res, o, grads, gn = L.train(*args, return_all=True)
            flips, elems, max_abs = flips + st["flips"], elems + st["elems"], max(max_abs, st["max_abs_at_flip"])
            for k in ("pi_loss", "baseline_loss", "entropy", "total_loss"):
                errs["loss/" + k + tag] = rel_err(out[k], float(o[k].detach()))
            errs["lr" + tag] = abs(out["learning_rate"] - res[3])
            errs["grad_norm" + tag] = rel_err(out["grad_norm"], gn)
            if gradient_clip_norm is not None:
                errs["clip_engaged" + tag] = 0.0 if gn > gradient_clip_norm else float("inf")
            if out["step"] != s + 1:
                errs["step" + tag] = float("inf")
            taps = eng.taps()
            for k in ("vs", "clipped_rho", "vs_plus_1", "pg_advantage"):
                errs["tap/" + k + tag] = rel_err(taps[k], o[k].detach().numpy())
            gd = it.unflatten_params(eng.get_grads(), torch.float64, num_action=A)
            for n in grads:
                errs["grad/" + n + tag] = rel_err(gd[n].numpy(), grads[n].detach().numpy())
            # applied update w_after - w_before, judged against its own size plus the float32 storage
            # granularity of the parameter it is added to (the GPU keeps w in float32)
            pd = it.unflatten_params(eng.get_params(), torch.float64, num_action=A)
            for n in L.params:
                p0 = p_before[n].numpy()
                du_exp = L.params[n].detach().numpy() - p0
                # the GPU's own previous parameters differ from the oracle's by accumulated rounding: compare
                # absolute parameters with a floor of a few float32 ulps
                floor = 4.0 * np.finfo(np.float32).eps * max(np.max(np.abs(p0)), 1e-30) / TOL
                errs["update/" + n + tag] = float(np.max(np.abs(pd[n].numpy() - L.params[n].detach().numpy())) /
                                                  (np.max(np.abs(du_exp)) + floor))
            if layers and s == 0:
                tp = o["taps"]
                errs["act/policy"] = rel_err(eng.read_buffer("policy", M * A).reshape(M, A),
                                             to_time_major(tp["policy"].detach().numpy()))
                errs["act/value"] = rel_err(eng.read_buffer("value", M), to_time_major(tp["value"].detach().numpy()))
                for nm in ("h1", "c1"):
                    errs["act/" + nm] = rel_err(eng.read_buffer(nm, M * 256).reshape(M, 256),
                                                to_time_major(tp[nm].detach().numpy()))
                ag = o.get("act_grads", {})
                for nm, shp in (("a1", (20, 20, 32)), ("a2", (9, 9, 64)), ("a3", (7, 7, 64))):
                    ref = tp[nm].detach().numpy().reshape((B, T) + shp)
                    got = eng.read_buffer(nm, M * int(np.prod(shp))).reshape((M,) + shp)
                    errs["act/" + nm] = rel_err(got, to_time_major(ref))
                    if ag.get(nm) is not None:   # GPU buffers hold dL/d(pre-ReLU) for the first Mb rows
                        gr = ag[nm].detach().numpy().reshape((B, T) + shp) * \
                            to_time_major_inv_mask(masks[nm], B, T, shp)
                        gotb = eng.read_buffer("d" + nm, Mb * int(np.prod(shp))).reshape((Mb,) + shp)
                        errs["bwd/d" + nm] = rel_err(gotb, to_time_major(gr)[:Mb])
        ms, st_ = eng.get_opt_state()
        md = it.unflatten_params(ms, torch.float64, num_action=A)
        for n in L.params:
            errs["ms/" + n] = rel_err(md[n].numpy(), L.ms[n].detach().numpy())
        if st_ != steps:
            errs["opt_step"] = float("inf")
        errs["kink/flip_fraction"] = flips / max(elems, 1)
        errs["kink/max_abs_at_flip"] = max_abs
    finally:
        eng.close()
    return errs


def to_time_major_inv_mask(mask_bm, B, T, shp):
    """oracle-row-order mask [B*T, ...] -> [B, T, ...] float array."""
    return mask_bm.numpy().reshape((B, T) + shp).astype(np.float64)


def failures(errs, tol=TOL, update_tol=1e-3):
    """Entries that break the bar: 1e-4 on everything, 1e-3 on the applied update (float32 storage), 1e-9 on
    the learning rate, and the kink statistics."""
    bad = {}
    for k, v in errs.items():
        if k.startswith("lr"):
            lim = 1e-9
        elif k.startswith("update/"):
            lim = update_tol
        elif k == "kink/flip_fraction":
            lim = FLIP_FRACTION_MAX
        elif k == "kink/max_abs_at_flip":
            lim = FLIP_ABS_MAX
        else:
            lim = tol
        if not (v <= lim):
            bad[k] = v
    return bad


def worst(errs, prefix=""):
    items = [(v, k) for k, v in errs.items() if k.startswith(prefix)]
    return max(items) if items else (0.0, "")
