"""GPU tests of the device-resident prioritized replay (drl_apex_replay_*, csrc/replay.cu): the sum tree bit-exact against
sequential SumTree updates of the device's own leaf values, priorities within 2 ulp of (|td| + 0.001)^0.6, sampling
bit-exact against SumTreeNP.find on the NumPy Philox draws, and a replay step bit-identical to stage + step of the same
minibatch on a twin learner."""
import ctypes as C

import numpy as np
import pytest
import torch

import apex_parity as ap
from oracle import apex_torch as ax
from oracle.per_np import MemoryNP, SumTreeNP
from oracle.replay_np import u01

pytestmark = pytest.mark.gpu

FIELDS = ("state", "next_state", "previous_action", "action", "reward", "done")


def _learners(B, A=4, n=2, **kw):
    params = ax.init_params(0, torch.float32, num_action=A)
    target = ax.init_params(1, torch.float32, num_action=A)
    return [ap.native_apex(B, A, params, target, **kw) for _ in range(n)]


def _record(n, seed, A=4):
    t = ax.make_transitions(n, A=A, seed=seed)
    return {k: t[k] for k in FIELDS}


def _ulps(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return np.abs(a.view(np.int64) - b.view(np.int64))


class Mirror:
    """Host copy of the ring (record ids per data index) and the NumPy tree replayed from the device's leaf values."""

    def __init__(self, cap):
        self.tree = SumTreeNP(cap)
        self.rows = {k: [None] * cap for k in FIELDS}

    def add(self, rep, rec):
        n = len(rec["reward"])
        rep.add(*[rec[k] for k in FIELDS])
        leaves, prios = rep.last_update()
        assert len(leaves) == n
        for i in range(n):
            slot = self.tree.add(prios[i])
            assert leaves[i] == slot + self.tree.capacity - 1
            for k in FIELDS:
                self.rows[k][slot] = rec[k][i]
        return leaves, prios

    def after_step(self, rep):
        leaves, prios = rep.last_update()
        for lf, p in zip(leaves, prios):
            self.tree.set_leaf(int(lf), p)

    def batch(self, data_index):
        return [np.stack([self.rows[k][int(i)] for i in data_index]) for k in FIELDS]


def _assert_tree(rep, mirror):
    got = rep.tree()
    assert np.array_equal(got.view(np.int64), mirror.tree.nodes.view(np.int64)), \
        np.flatnonzero(got != mirror.tree.nodes)[:10]
    info = rep.info()
    assert info["n_entries"] == mirror.tree.n_entries and info["write"] == mirror.tree.cursor
    assert info["total"] == mirror.tree.total()


def _replay(eng, cap, seed=0):
    from distributed_reinforcement_learning_b200.apex_learner import NativeApexReplay
    return NativeApexReplay(eng, cap, seed)


def test_ingest_with_wrap():
    B, cap = 16, 50
    eng, twin = _learners(B)
    rep = _replay(eng, cap)
    try:
        m = Mirror(cap)
        for r in range(4):                                   # 3 B + 5 transitions: wraps the ring of 50
            rec = _record(B if r < 3 else 5, seed=10 + r)
            leaves, prios = m.add(rep, rec)
            td = twin.td_error(*[rec[k] for k in FIELDS])
            t = eng.taps(len(td))                            # the add's own forward: |target - q(s, a)| bit for bit
            assert np.array_equal(np.abs(t["target_value"] - t["state_action_value"]), td)
            want = (td.astype(np.float64) + 0.001) ** 0.6
            assert _ulps(prios, want).max() <= 2
            _assert_tree(rep, m)
        assert len(rep) == cap and rep.info()["write"] == (3 * B + 5) % cap
    finally:
        rep.close()
        eng.close()
        twin.close()


def _fill(rep, mirror, n, B, seed, skew=None):
    for lo in range(0, n, B):
        rec = _record(min(B, n - lo), seed=seed + lo)
        if skew is not None and lo == 0:
            rec["reward"][0] = skew                          # one huge |td|: a leaf drawn many times per batch
        mirror.add(rep, rec)


def _sample_np(mirror, beta, seed, B, call):
    mem = MemoryNP(mirror.tree.capacity)
    mem.tree = SumTreeNP(mirror.tree.capacity)
    mem.tree.nodes = mirror.tree.nodes.copy()
    mem.tree.n_entries = mirror.tree.n_entries
    mem.beta = beta
    return mem.sample(B, u01(seed, B, call)), mem.beta


def _step_pair(rep, mirror, twin, slot, seed, call, beta):
    """A replay step, the NumPy sample it must have drawn, and stage + step of the same minibatch on the twin."""
    (ti, di, pr, w), beta_np = _sample_np(mirror, beta, seed, rep.B, call)
    out, td = rep.step(slot)
    ls = rep.last_sample()
    assert np.array_equal(ls["tree_index"], ti) and np.array_equal(ls["data_index"], di)
    assert np.array_equal(ls["priority"].view(np.int64), pr.view(np.int64))
    assert _ulps(ls["is_weight"], w).max() <= 8
    info = rep.info()
    assert info["beta"] == beta_np and info["draws"] == call + 1
    twin.stage(slot, *mirror.batch(ls["data_index"]), np.float32(ls["is_weight"]))
    out2, td2 = twin.step(slot)
    for k in ("loss", "grad_norm", "learning_rate", "step"):
        assert out[k] == out2[k], (k, out[k], out2[k])
    assert np.array_equal(td, td2)
    mirror.after_step(rep)
    return beta_np, ls


def _same_state(a, b):
    from distributed_reinforcement_learning_b200.apex_learner import MAIN, TARGET
    for which in (MAIN, TARGET):
        assert np.array_equal(a.get_params(which), b.get_params(which))
    oa, ob = a.get_opt_state(), b.get_opt_state()
    for k in ("m", "v"):
        assert np.array_equal(oa[k], ob[k]), k
    assert oa["step"] == ob["step"]


@pytest.mark.parametrize("graph", [False, True])
def test_sampling_and_step_equivalence(graph):
    B, cap, seed = 16, 50, 1234
    eng, twin = _learners(B, use_cuda_graph=graph, reward_clipping="none")
    rep = _replay(eng, cap, seed)
    try:
        m = Mirror(cap)
        _fill(rep, m, 40, B, seed=300, skew=500.0)
        _assert_tree(rep, m)
        beta, dup = 0.4, 0
        for call in range(3):
            beta, ls = _step_pair(rep, m, twin, call % 2, seed, call, beta)
            dup = max(dup, int(np.bincount(ls["tree_index"]).max()))
            _assert_tree(rep, m)                             # the post-step update, duplicates included
            if call == 1:
                eng.target_to_main()
                twin.target_to_main()
        assert dup >= 3
        _same_state(eng, twin)
        with pytest.raises(Exception) as ei:                 # the replay left slot 0 unstaged
            eng.step(0)
        assert getattr(ei.value, "code", None) == -3
    finally:
        rep.close()
        eng.close()
        twin.close()


def test_capture_does_not_advance_state():
    B, cap, seed, K = 8, 40, 99, 4
    g, e = _learners(B, use_cuda_graph=True, n=1)[0], _learners(B, n=1)[0]
    rg, re_ = _replay(g, cap, seed), _replay(e, cap, seed)
    try:
        mg, me = Mirror(cap), Mirror(cap)
        _fill(rg, mg, 30, B, seed=7)
        _fill(re_, me, 30, B, seed=7)
        (ti, _, _, _), _ = _sample_np(mg, 0.4, seed, B, 0)
        outs = []
        for k in range(K):
            og, tg = rg.step(0)
            if k == 0:
                assert rg.info()["draws"] == 1 and np.array_equal(rg.last_sample()["tree_index"], ti)
            oe, te = re_.step(0)
            outs.append((og["loss"], oe["loss"]))
            assert np.array_equal(tg, te)
        assert all(a == b for a, b in outs)
        assert np.array_equal(rg.tree().view(np.int64), re_.tree().view(np.int64))
        _same_state(g, e)
    finally:
        rg.close()
        re_.close()
        g.close()
        e.close()


def test_learner_loop_equivalence():
    """train_apex.py:82-155 twice, 20 iterations: host Memory fed with the same Philox draws vs the device replay."""
    from distributed_reinforcement_learning_b200.distributed_queue import buffer_queue
    B, cap, seed, T = 8, 64, 5, 8
    host, dev = _learners(B)
    rep = _replay(dev, cap, seed)
    mem = buffer_queue.Memory(cap)
    try:
        for it in range(20):
            rec = _record(T, seed=1000 + it)
            args = [rec[k] for k in FIELDS]
            td = host.td_error(*args)
            for i in range(T):
                mem.add(td[i], [rec[k][i] for k in FIELDS])
            rep.add(*args)
            batch, idxs, w = mem.sample(B, u01=u01(seed, B, it))
            mb = np.array(batch, dtype=object)
            host.stage(0, *[np.stack(mb[:, j]) for j in range(6)], w)
            _, td_h = host.step(0)
            _, td_d = rep.step(0)
            assert rep.last_sample()["tree_index"].tolist() == idxs, it
            if it % 5 == 4:
                host.target_to_main()
                dev.target_to_main()
            for i in range(B):
                mem.update(idxs[i], td_h[i])
            t_h, t_d = mem.tree.total(), rep.info()["total"]
            assert abs(t_h - t_d) <= 1e-12 * abs(t_h), (it, t_h, t_d)
        ph, pd = host.get_params(), dev.get_params()
        assert np.max(np.abs(ph - pd)) <= 1e-6 * np.max(np.abs(ph))
    finally:
        rep.close()
        mem.tree.close()
        host.close()
        dev.close()


def test_large_capacity_past_the_wrap():
    """Capacity 1e5 filled past the wrap: gathered rows above data index 76,088 (byte offsets > 2^31) equal the host's."""
    B, cap, seed = 32, 100000, 3
    eng, twin = _learners(B)
    rep = _replay(eng, cap, seed)
    try:
        pool = _record(3 * B, seed=77)
        ids = np.zeros(cap, np.int64)
        total = cap + 2 * B
        for t0 in range(0, total, B):
            k = (t0 // B) % 3
            rep.add(*[pool[f][k * B:(k + 1) * B] for f in FIELDS])
            ids[(t0 + np.arange(B)) % cap] = k * B + np.arange(B)
        info = rep.info()
        assert info["n_entries"] == cap and info["write"] == total % cap
        hi = 0
        for call in range(4):
            out, td = rep.step(call % 2)
            ls = rep.last_sample()
            di = ls["data_index"]
            hi += int((di >= 76088).sum())
            twin.stage(call % 2, *[pool[f][ids[di]] for f in FIELDS], np.float32(ls["is_weight"]))
            out2, td2 = twin.step(call % 2)
            assert out["loss"] == out2["loss"] and np.array_equal(td, td2)
        assert hi > 0
    finally:
        rep.close()
        eng.close()
        twin.close()


def test_errors(native):
    from distributed_reinforcement_learning_b200.a3c_learner import NativeA3CLearner
    eng = _learners(4, n=1)[0]
    try:
        with pytest.raises(native.DrlError) as ei:
            _replay(eng, 1)
        assert ei.value.code == native.DRL_ERR_INVALID
        rep = _replay(eng, 10)
        with pytest.raises(native.DrlError) as ei:
            rep.step(0)                                      # empty
        assert ei.value.code == native.DRL_ERR_STATE
        rec = _record(5, seed=1)
        with pytest.raises(native.DrlError):                 # n > B straight through the C-ABI
            arrs = eng._arrays(5, *[rec[k] for k in FIELDS])
            native.check(native.lib.drl_apex_replay_add(rep._r, 5, *[native.ptr(a) for a in arrs]))
        with pytest.raises(ValueError):
            rep.add(rec["state"][:, :80], rec["next_state"], rec["previous_action"], rec["action"], rec["reward"],
                    rec["done"])
        rep.add(*[rec[k] for k in FIELDS])                   # 5 > B = 4: chunked by the wrapper
        assert len(rep) == 5
        # the learner cannot go away under a live replay
        assert native.lib.drl_apex_destroy(eng._h) == native.DRL_ERR_STATE
        rep.step(1)
        with pytest.raises(native.DrlError) as ei:
            eng.step(1)                                      # the replay wrote slot 1: not staged
        assert ei.value.code == native.DRL_ERR_STATE
        rep.close()
    finally:
        eng.close()
    a3c = NativeA3CLearner(batch=4, num_action=4)
    try:
        out = C.c_void_p()
        assert native.lib.drl_apex_replay_create(a3c._h, 10, C.c_uint64(0), C.byref(out)) == native.DRL_ERR_INVALID
    finally:
        a3c.close()


def test_agent_surface_runs_learner_loop(native):
    """The learner branch of train_apex.py:82-155 on Agent.make_device_replay."""
    from distributed_reinforcement_learning_b200.agent import apex
    learner = apex.Agent(input_shape=[84, 84, 4], num_action=4, discount_factor=0.99, gradient_clip_norm=40.0,
                         reward_clipping='abs_one', start_learning_rate=1e-4, end_learning_rate=0.0,
                         learning_frame=100000000000000, model_name='replay_learner', learner_name='replay_learner')
    learner.set_session(None)
    learner.target_to_main()
    replay = learner.make_device_replay(capacity=64, batch_size=8, seed=1)
    try:
        for it_ in range(4):
            fa = ax.make_transitions(12, seed=100 + it_)
            replay.add(state=fa['state'], next_state=fa['next_state'], previous_action=fa['previous_action'],
                       action=fa['action'], reward=fa['reward'], done=fa['done'])
            loss, td = replay.train()
            assert np.isfinite(loss) and td.shape == (8,) and np.all(td >= 0)
            if it_ % 2 == 0:
                learner.target_to_main()
        assert len(replay) == 48 and replay.total() > 0 and replay.beta == pytest.approx(0.404)
        assert learner.num_env_frames == 4
        b = ax.make_transitions(4, seed=5)
        with pytest.raises(ValueError):                      # another batch size would rebuild the learner
            learner.distributed_train(*[b[k] for k in ax.TRAIN_FIELDS])
    finally:
        replay.close()
